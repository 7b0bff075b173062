// Counter-based random draws of the train step (Philox4x32-10, Salmon et al. SC'11).
//
// The reference makes every draw of one `update` inside the jitted step from ONE key
// (/root/reference/cnf_ot/mfc/applications.py:81-82,233-239,392,416,435; solvers.py:104-105),
// and relies on "equal key => equal draw": every sampler of a loss call sees the same latent rows.
// Here a draw is a pure function of (key, step, kind and leading size of the drawn array, row, column):
//
//   philox key = key ^ salt(kind, n)        kind: 1 normal (n, D), 2 uniform (n,), 3 categorical (n,)
//   counter    = (row_lo, row_hi, column_block, step)
//
// i.e. like jax.random, arrays of different shapes drawn from one key are unrelated (the B-row latent of the
// fit terms and the b = B//32-row latent of the kinetic terms, applications.py:111-116 vs 233-239), while equal
// (key, shape) gives equal numbers.  The kernels generate their rows on chip (nothing crosses PCIe or HBM), any
// shard of the batch can be generated independently (row = GLOBAL row index: the result does not depend on
// how the rows are split over GPUs), and cnfot_philox_* write the very same numbers into arrays for the
// explicit-input entry points and for the CPU oracle.
// jax.random's threefry streams are NOT reproduced (parity tests compare on exported arrays).
#pragma once

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define CNFOT_PHILOX_HD __host__ __device__ __forceinline__
#else
#define CNFOT_PHILOX_HD inline
#endif

namespace cnfot {

enum PhiloxKind { kDrawNormal = 1, kDrawUniform = 2, kDrawCategorical = 3 };
// how a segment of the fused step obtains its rows
enum RowSource {
  kRowsMemory = 0,    // read from the caller's array
  kRowsNormal = 1,    // N(0, I) rows: latent rows, and the target of kl_loss_fn (applications.py:73-82)
  kRowsOtSource = 3   // z + centre[idx] (dim 2: the 8-mode mixture, applications.py:34-71) or z - 3 (other dims),
                      // z being the kRowsNormal draw of the same shape (the reference reuses the key, :81-82)
};

CNFOT_PHILOX_HD uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
// key modifier of a draw of `n` leading entries of kind `kind`
CNFOT_PHILOX_HD uint64_t philox_salt(int kind, uint64_t n) { return splitmix64(splitmix64((uint64_t)kind) ^ n); }

// The key modifiers of one train step's draws (both engines): normal (B, D) rows of the fit terms, categorical (B,)
// mixture modes of the ot source, normal (b, D) rows of the kinetic terms, uniform (n_t,) times
struct StepSalts { uint64_t B, Bc, b, t; };
CNFOT_PHILOX_HD StepSalts step_salts(int64_t global_B, int64_t global_b, int n_t) {
  StepSalts s;
  s.B = philox_salt(kDrawNormal, (uint64_t)global_B);
  s.Bc = philox_salt(kDrawCategorical, (uint64_t)global_B);
  s.b = philox_salt(kDrawNormal, (uint64_t)global_b);
  s.t = philox_salt(kDrawUniform, (uint64_t)n_t);
  return s;
}

struct PhiloxWords { uint32_t w[4]; };

CNFOT_PHILOX_HD uint32_t philox_mulhi(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

CNFOT_PHILOX_HD PhiloxWords philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = philox_mulhi(M0, c0), lo0 = M0 * c0;
    const uint32_t hi1 = philox_mulhi(M1, c2), lo1 = M1 * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += W0; k1 += W1;
  }
  PhiloxWords o;
  o.w[0] = c0; o.w[1] = c1; o.w[2] = c2; o.w[3] = c3;
  return o;
}

CNFOT_PHILOX_HD PhiloxWords philox_draw(uint64_t key, uint32_t step, uint64_t row, uint32_t block) {
  return philox4x32_10((uint32_t)row, (uint32_t)(row >> 32), block, step, (uint32_t)key, (uint32_t)(key >> 32));
}

// 24-bit uniforms: exactly representable in float32, identical on host and device
CNFOT_PHILOX_HD float philox_uniform_open(uint32_t w) { return ((float)(w >> 8) + 0.5f) * (1.0f / 16777216.0f); }  // (0, 1)
CNFOT_PHILOX_HD float philox_uniform(uint32_t w) { return (float)(w >> 8) * (1.0f / 16777216.0f); }                // [0, 1)

// Box-Muller: two words -> two N(0, 1) draws
CNFOT_PHILOX_HD void philox_normal2(uint32_t wa, uint32_t wb, float& z0, float& z1) {
  const float r = sqrtf(-2.0f * logf(philox_uniform_open(wa)));
  float s, c;
#if defined(__CUDA_ARCH__)
  sincospif(2.0f * philox_uniform(wb), &s, &c);
#else
  const float th = 6.283185307179586f * philox_uniform(wb);
  s = sinf(th); c = cosf(th);
#endif
  z0 = r * c;
  z1 = r * s;
}

// the uniform time t_i of one step, i < t_batch_size (applications.py:392,416,435): horizon * U[0, 1);
// key_t = key ^ philox_salt(kDrawUniform, t_batch_size)
CNFOT_PHILOX_HD float philox_time(uint64_t key_t, uint32_t step, int i, float horizon) {
  return philox_uniform(philox_draw(key_t, step, (uint64_t)i, 0).w[0]) * horizon;
}

// One row of `D` draws (row = GLOBAL row index of an (n, D) array); key_n = key ^ philox_salt(kDrawNormal, n),
// key_c = key ^ philox_salt(kDrawCategorical, n) (read by kRowsOtSource at D == 2 only).
CNFOT_PHILOX_HD void philox_row(uint64_t key_n, uint64_t key_c, uint32_t step, int source, uint64_t row, int D, float* out) {
  for (int cb = 0; cb * 4 < D; ++cb) {
    const PhiloxWords p = philox_draw(key_n, step, row, (uint32_t)cb);
    float z[4];
    philox_normal2(p.w[0], p.w[1], z[0], z[1]);
    if (cb * 4 + 2 < D) philox_normal2(p.w[2], p.w[3], z[2], z[3]);
    for (int j = 0; j < 4 && cb * 4 + j < D; ++j) out[cb * 4 + j] = z[j];
  }
  if (source == kRowsOtSource) {
    if (D == 2) {
      // 8 modes on the circle of radius 5 (applications.py:34-71)
      const uint32_t idx = philox_draw(key_c, step, row, 0).w[0] >> 29;
      const float R = 5.0f;
      float cx = 0.f, cy = 0.f;
      switch (idx) {
        case 0: cy = R; break;
        case 1: cx = R; break;
        case 2: cy = -R; break;
        case 3: cx = -R; break;
        case 4: cx = 3.0f; cy = 4.0f; break;     // (0.6 R, 0.8 R)
        case 5: cx = 3.0f; cy = -4.0f; break;
        case 6: cx = -3.0f; cy = -4.0f; break;
        default: cx = -3.0f; cy = 4.0f; break;
      }
      out[0] += cx;
      out[1] += cy;
    } else {
      for (int j = 0; j < D; ++j) out[j] -= 3.0f;   // Gaussian -> Gaussian variant (applications.py:28-32, ot.py:72-80)
    }
  }
}

// Column c alone of philox_row's row (the same operations on the same words): for kernels that write one element
// per thread
CNFOT_PHILOX_HD float philox_entry(uint64_t key_n, uint64_t key_c, uint32_t step, int source, uint64_t row, int D, int c) {
  const PhiloxWords p = philox_draw(key_n, step, row, (uint32_t)(c >> 2));
  const int pair = (c >> 1) & 1;
  float z0, z1;
  philox_normal2(p.w[2 * pair], p.w[2 * pair + 1], z0, z1);
  float v = (c & 1) ? z1 : z0;
  if (source == kRowsOtSource) {
    if (D == 2) {
      const uint32_t idx = philox_draw(key_c, step, row, 0).w[0] >> 29;
      float cx = 0.f, cy = 0.f;   // the modes of philox_row
      switch (idx) {
        case 0: cy = 5.0f; break;
        case 1: cx = 5.0f; break;
        case 2: cy = -5.0f; break;
        case 3: cx = -5.0f; break;
        case 4: cx = 3.0f; cy = 4.0f; break;
        case 5: cx = 3.0f; cy = -4.0f; break;
        case 6: cx = -3.0f; cy = -4.0f; break;
        default: cx = -3.0f; cy = 4.0f; break;
      }
      v += c == 0 ? cx : cy;
    } else {
#if defined(__CUDA_ARCH__)
      // a separately rounded add, as philox_row computes it: contracted with z = r c into one FMA it would round once
      // and differ from philox_row's number by up to one ulp in the kernels where the compiler fuses the two
      v = __fadd_rn(v, -3.0f);
#else
      v -= 3.0f;
#endif
    }
  }
  return v;
}

}  // namespace cnfot
