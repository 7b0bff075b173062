// Hardware counters of the kernels launched between cc_start() and cc_stop(), read through the CUPTI range profiler
// API.  Loaded by tools/capture_counters.py through ctypes; built there with the toolkit's nvcc (host code only).
#include <cuda.h>
#include <cupti_profiler_host.h>
#include <cupti_profiler_target.h>
#include <cupti_range_profiler.h>
#include <cupti_result.h>
#include <cupti_target.h>

#include <cstdio>
#include <string>
#include <vector>

namespace {
std::string g_err;
std::vector<std::string> g_names;
std::vector<const char*> g_metrics;
std::vector<uint8_t> g_avail, g_config, g_data;
CUpti_RangeProfiler_Object* g_obj = nullptr;
CUpti_Profiler_Host_Object* g_host = nullptr;
bool g_user = false;
}  // namespace

#define CC_CHECK(call)                                                          \
  do {                                                                          \
    CUptiResult r_ = (call);                                                    \
    if (r_ != CUPTI_SUCCESS) {                                                  \
      const char* s_ = nullptr;                                                 \
      cuptiGetResultString(r_, &s_);                                            \
      g_err = std::string(#call) + ": " + (s_ ? s_ : "?") + " (" + std::to_string((int)r_) + ")"; \
      return (int)r_;                                                           \
    }                                                                           \
  } while (0)

extern "C" {

__attribute__((visibility("default"))) const char* cc_error() { return g_err.c_str(); }

// metrics: comma-separated metric names; max_ranges: ranges the capture can hold.  user_range 0: every kernel launched
// between cc_start() and cc_stop() is a range of its own, replayed by CUPTI; 1: all of them together are one range, and
// the caller repeats the work between cc_start() and cc_stop() until cc_stop() reports every pass submitted.
__attribute__((visibility("default"))) int cc_begin(const char* metrics, int max_ranges, int user_range) {
  g_user = user_range != 0;
  g_names.clear();
  g_metrics.clear();
  for (std::string s = metrics; !s.empty();) {
    const size_t c = s.find(',');
    g_names.push_back(s.substr(0, c));
    s = c == std::string::npos ? "" : s.substr(c + 1);
  }
  for (const std::string& n : g_names) g_metrics.push_back(n.c_str());
  CUcontext ctx = nullptr;
  CUdevice dev = 0;
  if (cuCtxGetCurrent(&ctx) != CUDA_SUCCESS || ctx == nullptr || cuCtxGetDevice(&dev) != CUDA_SUCCESS) {
    g_err = "no current CUDA context";
    return -1;
  }
  CUpti_Profiler_Initialize_Params ip = {CUpti_Profiler_Initialize_Params_STRUCT_SIZE};
  CC_CHECK(cuptiProfilerInitialize(&ip));
  CUpti_Device_GetChipName_Params cn = {CUpti_Device_GetChipName_Params_STRUCT_SIZE};
  cn.deviceIndex = (size_t)dev;
  CC_CHECK(cuptiDeviceGetChipName(&cn));
  CUpti_RangeProfiler_Enable_Params ep = {CUpti_RangeProfiler_Enable_Params_STRUCT_SIZE};
  ep.ctx = ctx;
  CC_CHECK(cuptiRangeProfilerEnable(&ep));
  g_obj = ep.pRangeProfilerObject;
  CUpti_Profiler_GetCounterAvailability_Params ca = {CUpti_Profiler_GetCounterAvailability_Params_STRUCT_SIZE};
  ca.ctx = ctx;
  CC_CHECK(cuptiProfilerGetCounterAvailability(&ca));
  g_avail.assign(ca.counterAvailabilityImageSize, 0);
  ca.pCounterAvailabilityImage = g_avail.data();
  CC_CHECK(cuptiProfilerGetCounterAvailability(&ca));
  CUpti_Profiler_Host_Initialize_Params hi = {CUpti_Profiler_Host_Initialize_Params_STRUCT_SIZE};
  hi.profilerType = CUPTI_PROFILER_TYPE_RANGE_PROFILER;
  hi.pChipName = cn.pChipName;
  hi.pCounterAvailabilityImage = g_avail.data();
  CC_CHECK(cuptiProfilerHostInitialize(&hi));
  g_host = hi.pHostObject;
  CUpti_Profiler_Host_ConfigAddMetrics_Params am = {CUpti_Profiler_Host_ConfigAddMetrics_Params_STRUCT_SIZE};
  am.pHostObject = g_host;
  am.ppMetricNames = g_metrics.data();
  am.numMetrics = g_metrics.size();
  CC_CHECK(cuptiProfilerHostConfigAddMetrics(&am));
  CUpti_Profiler_Host_GetConfigImageSize_Params cs = {CUpti_Profiler_Host_GetConfigImageSize_Params_STRUCT_SIZE};
  cs.pHostObject = g_host;
  CC_CHECK(cuptiProfilerHostGetConfigImageSize(&cs));
  g_config.assign(cs.configImageSize, 0);
  CUpti_Profiler_Host_GetConfigImage_Params ci = {CUpti_Profiler_Host_GetConfigImage_Params_STRUCT_SIZE};
  ci.pHostObject = g_host;
  ci.configImageSize = g_config.size();
  ci.pConfigImage = g_config.data();
  CC_CHECK(cuptiProfilerHostGetConfigImage(&ci));
  CUpti_RangeProfiler_GetCounterDataSize_Params ds = {CUpti_RangeProfiler_GetCounterDataSize_Params_STRUCT_SIZE};
  ds.pRangeProfilerObject = g_obj;
  ds.pMetricNames = g_metrics.data();
  ds.numMetrics = g_metrics.size();
  ds.maxNumOfRanges = (size_t)max_ranges;
  ds.maxNumRangeTreeNodes = (uint32_t)max_ranges;
  CC_CHECK(cuptiRangeProfilerGetCounterDataSize(&ds));
  g_data.assign(ds.counterDataSize, 0);
  CUpti_RangeProfiler_CounterDataImage_Initialize_Params di = {
      CUpti_RangeProfiler_CounterDataImage_Initialize_Params_STRUCT_SIZE};
  di.pRangeProfilerObject = g_obj;
  di.counterDataSize = g_data.size();
  di.pCounterData = g_data.data();
  CC_CHECK(cuptiRangeProfilerCounterDataImageInitialize(&di));
  CUpti_RangeProfiler_SetConfig_Params sc = {CUpti_RangeProfiler_SetConfig_Params_STRUCT_SIZE};
  sc.pRangeProfilerObject = g_obj;
  sc.configSize = g_config.size();
  sc.pConfig = g_config.data();
  sc.counterDataImageSize = g_data.size();
  sc.pCounterDataImage = g_data.data();
  sc.range = g_user ? CUPTI_UserRange : CUPTI_AutoRange;
  sc.replayMode = g_user ? CUPTI_UserReplay : CUPTI_KernelReplay;
  sc.maxRangesPerPass = (size_t)max_ranges;
  sc.numNestingLevels = 1;
  sc.minNestingLevel = 1;
  sc.passIndex = 0;
  sc.targetNestingLevel = 1;
  CC_CHECK(cuptiRangeProfilerSetConfig(&sc));
  return 0;
}

__attribute__((visibility("default"))) int cc_start() {
  CUpti_RangeProfiler_Start_Params st = {CUpti_RangeProfiler_Start_Params_STRUCT_SIZE};
  st.pRangeProfilerObject = g_obj;
  CC_CHECK(cuptiRangeProfilerStart(&st));
  if (g_user) {
    CUpti_RangeProfiler_PushRange_Params pr = {CUpti_RangeProfiler_PushRange_Params_STRUCT_SIZE};
    pr.pRangeProfilerObject = g_obj;
    pr.pRangeName = "captured";
    CC_CHECK(cuptiRangeProfilerPushRange(&pr));
  }
  return 0;
}

// *all_submitted: 1 once every pass the metric set needs has been submitted (user ranges: repeat the work until then)
__attribute__((visibility("default"))) int cc_stop(int* all_submitted) {
  if (g_user) {
    CUpti_RangeProfiler_PopRange_Params pr = {CUpti_RangeProfiler_PopRange_Params_STRUCT_SIZE};
    pr.pRangeProfilerObject = g_obj;
    CC_CHECK(cuptiRangeProfilerPopRange(&pr));
  }
  CUpti_RangeProfiler_Stop_Params sp = {CUpti_RangeProfiler_Stop_Params_STRUCT_SIZE};
  sp.pRangeProfilerObject = g_obj;
  CC_CHECK(cuptiRangeProfilerStop(&sp));
  *all_submitted = sp.isAllPassSubmitted ? 1 : 0;
  return 0;
}

// Ends the capture and writes one line per range: "<range name>\t<value of metric 0>\t...\n" (auto ranges are named
// after the kernel), after a first line "#dropped\t<ranges the counter data could not hold>".
__attribute__((visibility("default"))) int cc_end(char* out, int out_len) {
  CUpti_RangeProfiler_DecodeData_Params dd = {CUpti_RangeProfiler_DecodeData_Params_STRUCT_SIZE};
  dd.pRangeProfilerObject = g_obj;
  CC_CHECK(cuptiRangeProfilerDecodeData(&dd));
  CUpti_RangeProfiler_GetCounterDataInfo_Params gi = {CUpti_RangeProfiler_GetCounterDataInfo_Params_STRUCT_SIZE};
  gi.pCounterDataImage = g_data.data();
  gi.counterDataImageSize = g_data.size();
  CC_CHECK(cuptiRangeProfilerGetCounterDataInfo(&gi));
  std::string text = "#dropped\t" + std::to_string(dd.numOfRangeDropped) + "\n";
  std::vector<double> v(g_metrics.size());
  for (size_t r = 0; r < gi.numTotalRanges; ++r) {
    CUpti_RangeProfiler_CounterData_GetRangeInfo_Params ri = {
        CUpti_RangeProfiler_CounterData_GetRangeInfo_Params_STRUCT_SIZE};
    ri.pCounterDataImage = g_data.data();
    ri.counterDataImageSize = g_data.size();
    ri.rangeIndex = r;
    ri.rangeDelimiter = "/";
    CC_CHECK(cuptiRangeProfilerCounterDataGetRangeInfo(&ri));
    CUpti_Profiler_Host_EvaluateToGpuValues_Params ev = {CUpti_Profiler_Host_EvaluateToGpuValues_Params_STRUCT_SIZE};
    ev.pHostObject = g_host;
    ev.pCounterDataImage = g_data.data();
    ev.counterDataImageSize = g_data.size();
    ev.rangeIndex = r;
    ev.ppMetricNames = g_metrics.data();
    ev.numMetrics = g_metrics.size();
    ev.pMetricValues = v.data();
    CC_CHECK(cuptiProfilerHostEvaluateToGpuValues(&ev));
    text += ri.rangeName ? ri.rangeName : "?";
    char buf[64];
    for (double x : v) {
      snprintf(buf, sizeof buf, "\t%.17g", x);
      text += buf;
    }
    text += "\n";
  }
  CUpti_RangeProfiler_Disable_Params dp = {CUpti_RangeProfiler_Disable_Params_STRUCT_SIZE};
  dp.pRangeProfilerObject = g_obj;
  CC_CHECK(cuptiRangeProfilerDisable(&dp));
  CUpti_Profiler_Host_Deinitialize_Params hd = {CUpti_Profiler_Host_Deinitialize_Params_STRUCT_SIZE};
  hd.pHostObject = g_host;
  CC_CHECK(cuptiProfilerHostDeinitialize(&hd));
  CUpti_Profiler_DeInitialize_Params de = {CUpti_Profiler_DeInitialize_Params_STRUCT_SIZE};
  CC_CHECK(cuptiProfilerDeInitialize(&de));
  if ((int)text.size() + 1 > out_len) {
    g_err = "output buffer too small";
    return -2;
  }
  snprintf(out, (size_t)out_len, "%s", text.c_str());
  return 0;
}

}  // extern "C"
