"""Host-side mirror of the training part of /root/reference/cnf_ot/mfc/solvers.py
(:26-129): model construction, loss selection by `general.type`, the `update`
step (value_and_grad + Adam) and the training loop, plus the energy part of the evaluation
tail (:138-172, `evaluate`).  The plotting / grid-density part of the reference's `main`
(:173-493) is out of scope (SURVEY.md §2).

    from cnf_ot_b200 import solvers
    params, loss_hist = solvers.main(yaml.safe_load(open("cnf_ot_b200/config/mfc.yaml")))
"""
from __future__ import annotations

from functools import partial
from typing import Dict, Tuple

import torch

from . import applications, ops, random, utils
from .flows import ParamTree, RQSFlow, multi_transform, without_apply_rng


class AdamState:
  """optax.adam state (solvers.py:55-56): step count and the two moment blobs."""

  def __init__(self, params: ParamTree):
    self.count = 0
    self.mu = torch.zeros_like(params.blob)
    self.nu = torch.zeros_like(params.blob)


def build(config: Dict):
  """Model + loss selection, solvers.py:29-88.  Returns (model, loss_fn, T)."""
  g = config["general"]
  _type, dim, dt, dx = g["type"], g["dim"], g["dt"], g["dx"]
  t_batch_size = g["t_batch_size"]
  c = config["cnf"]
  model = RQSFlow(
    event_shape=(dim, ),
    num_layers=c["flow_num_layers"],
    hidden_sizes=[c["hidden_size"]] * c["mlp_num_layers"],
    num_bins=c["num_bins"],
    periodized=False,
  )
  model = without_apply_rng(multi_transform(model))
  if _type == "rwpo":
    r = config["rwpo"]
    T = r["T"]
    loss_fn = partial(applications.rwpo_loss_fn, model, dim, T, r["beta"], dt, dx, t_batch_size,
                      r["pot_type"], r["a"])
  elif _type == "fp":
    f = config["fp"]
    T = f["T"]
    loss_fn = partial(applications.fp_loss_fn, model, dim, T, f["a"], f["sigma"], dt, dx,
                      t_batch_size, f["velocity_field_type"])
  elif _type == "ot":
    T = 1
    loss_fn = partial(applications.ot_loss_fn, model, dim, T, dt, t_batch_size,
                      config["ot"]["subtype"])
  else:
    raise Exception(f"Unknown problem type: {_type}...")
  return model, loss_fn, T


def make_update(loss_fn, lr: float, batch_size: int):
  """solvers.py:90-97.  The parameter blob is updated IN PLACE (the returned params are
  the same object): B200-side the 'new pytree per step' of the functional original would
  only add a copy."""
  vg = applications.value_and_grad(loss_fn)

  def update(params: ParamTree, rng, _lambda, opt_state: AdamState) -> Tuple[torch.Tensor, ParamTree, AdamState]:
    loss, grads = vg(params, rng, _lambda, batch_size)
    opt_state.count += 1
    ops.adam_update(params.blob, grads.blob, opt_state.mu, opt_state.nu, lr, opt_state.count)
    return loss, params, opt_state

  return update


def main(config_dict: Dict, progress: bool = False, graph_steps: int = None):
  """Training loop of solvers.py:26-129; returns (params, loss_hist).

  Flows the fused step kernel covers train DEVICE-RESIDENT: one kernel launch per `update` (on-chip draws,
  value_and_grad, the data-parallel all-reduce, Adam: `cnfot_mfc_update`), `graph_steps` updates per CUDA graph
  (default: eval_frequency, at most 100), the loss history written by the kernel -- the host only replays graphs.
  The draws of update k are those of (train key, step k).  Wide-conditioner flows train the same way on one GPU
  (their update is a fixed sequence of launches, captured the same way), so a single-GPU wide run also draws the
  numbers of (train key, step k) -- before, it drew them from one key per step split from the run's key; with
  several GPUs they take the update() loop of `make_update` (that per-step key, as in solvers.py:104, and an NCCL
  all-reduce of the gradient)."""
  config = config_dict
  rng = random.PRNGKey(config["general"]["seed"])
  tr = config["train"]
  epochs, batch_size, eval_frequency, _lambda = tr["epochs"], tr["batch_size"], tr["eval_frequency"], tr["_lambda"]
  model, loss_fn, T = build(config)
  dim = config["general"]["dim"]
  model_rng, rng = random.split(rng)
  params = model.init(model_rng, torch.zeros(1, dim), torch.zeros(1))
  # optional keys beyond the reference's mfc.yaml (it has no checkpointing at all): train.params_in / train.params_out
  # name .npz files of the haiku-shaped pytree (ParamTree.save / load); the file also carries the optimiser state
  # (Adam moments, update count) and the run's key, so a resumed run continues the same trajectory
  resume = None
  if tr.get("params_in"):
    loaded, resume = ParamTree.load(tr["params_in"], device=params.blob.device, with_extras=True)
    if loaded.shape != params.shape:
      raise ValueError("train.params_in holds a different flow shape than the config")
    params = loaded
  rank, world = applications._dist.rank_world()
  step0 = int(resume["opt/count"]) if resume and "opt/count" in resume else 0

  def show(step, loss, rng):
    # solvers.py:108-127: the key is split at every evaluation point whether or not anything is printed
    eval_rng, rng = random.split(rng)
    if progress:
      desc = f"step {step} loss={float(loss):.4e}"
      if config["general"]["type"] == "ot":
        KL = applications.density_fit_kl_loss_fn(model, dim, T, params, eval_rng, batch_size)
        desc += f" KL={float(KL):.4f}"
      if rank == 0:
        print(desc, flush=True)
    return rng

  if params.blob.is_cuda and (ops.fused_update_supported(model.shape) or world == 1):
    sc = applications._step_config(loss_fn)
    shape, problem, n_t = model.shape, sc["problem"], config["general"]["t_batch_size"]
    B, b = batch_size, batch_size // 32
    rs, ss = applications._dist.shard(B, rank, world), applications._dist.shard(b, rank, world)
    train_key, rng = random.split(rng)
    key = int(resume["rng/train_key"]) if resume and "rng/train_key" in resume else train_key.value
    state = ops.TrainState(shape, params.blob, key, step=step0, peers=applications.peer_exchange(shape, model.device),
                           rows_B=rs.stop - rs.start, rows_b=ss.stop - ss.start)
    if resume and "opt/mu" in resume:
      state.mu.copy_(resume["opt/mu"].to(state.mu.device))
      state.nu.copy_(resume["opt/nu"].to(state.nu.device))
    hist = torch.zeros(step0 + epochs, dtype=torch.float32, device=params.blob.device)

    def one_update():
      ops.mfc_update(shape, problem, state, params.blob, n_t, _lambda, B, b, tr["lr"], rows_B=rs, rows_b=ss, loss_hist=hist)

    K = max(1, min(graph_steps or min(eval_frequency, 100), max(epochs, 1)))
    n_eager = epochs % K or min(K, epochs)   # the first updates run eagerly (they also warm the launch path up)
    done = 0
    next_eval = 0
    graph = None
    while done < epochs:
      if done < n_eager:
        one_update()
        done += 1
      else:
        if graph is None:
          # capture K updates once (nothing runs during capture; the calls' host-side bookkeeping is that of the
          # first replay), then replay: the device-side step counter selects draws, Adam's bias correction and
          # the loss slot, so every replay is K NEW updates
          graph = torch.cuda.CUDAGraph()
          with torch.cuda.graph(graph):
            for _ in range(K):
              one_update()
        else:
          state.steps_issued += K
          if state.peers is not None:
            state.peers.epoch += K
        graph.replay()
        done += K
      while next_eval < done:   # the evaluation points step % eval_frequency == 0 (solvers.py:108) passed so far
        rng = show(next_eval, hist[step0 + next_eval], rng)
        next_eval += eval_frequency
    loss_hist = list(hist[step0:].unbind()) if epochs > 0 else []
    opt_extras = {"opt/mu": state.mu, "opt/nu": state.nu, "opt/count": step0 + epochs, "rng/train_key": key}
    if epochs > 0 and state.status() != 0:
      raise RuntimeError("a peer GPU never arrived in the step's all-reduce (see CNFOT_DP_TIMEOUT_MS): results are NaN")
  else:
    opt_state = AdamState(params)
    opt_state.count = step0
    if resume and "opt/mu" in resume:
      opt_state.mu.copy_(resume["opt/mu"].to(opt_state.mu.device))
      opt_state.nu.copy_(resume["opt/nu"].to(opt_state.nu.device))
    update = make_update(loss_fn, tr["lr"], batch_size)
    loss_hist = []
    for step in range(epochs):
      update_rng, rng = random.split(rng)
      loss, params, opt_state = update(params, update_rng, _lambda, opt_state)
      loss_hist.append(loss.clone())  # a detached device scalar: neither a host sync (solvers.py:106) nor a hold on the step's buffer
      if step % eval_frequency == 0:
        rng = show(step, loss, rng)
    opt_extras = {"opt/mu": opt_state.mu, "opt/nu": opt_state.nu, "opt/count": opt_state.count}
  if tr.get("params_out") and rank == 0:
    params.save(tr["params_out"], extras=opt_extras)
  return params, loss_hist


def evaluate(config: Dict, model, params, rng, batch_size: int = 65536, t_size: int = 10000, T=None,
             verbose: bool = True) -> Dict[str, float]:
  """Energy part of the evaluation tail, solvers.py:138-172.
  ot:   the kinetic energy with more / fewer samples (utils.calc_kinetic_energy)
  rwpo: T * score-corrected kinetic energy + potential energy at t = T; for the quadratic potential
        the closed-form total dim (1 + log(T + 1)) / beta and the relative error in percent; for the 2-D double well
        the density at T on the reference's grid (solvers.py:184-222)
  fp:   the L2 errors of solvers.py:254-306 against the Ornstein-Uhlenbeck solution: Monte-Carlo (10^6 samples of
        the flow) and, in 2-D, on the 500 x 500 grid."""
  import math
  g = config["general"]
  _type, dim = g["type"], g["dim"]
  sample_fn, log_prob_fn = model.apply.sample, model.apply.log_prob
  eval_rng, rng = random.split(random.as_key(rng))
  out: Dict[str, float] = {}
  if _type == "ot":
    out["kinetic_more"] = float(utils.calc_kinetic_energy(sample_fn, params, eval_rng, batch_size=batch_size,
                                                          t_size=t_size, dim=dim))
    out["kinetic_less"] = float(utils.calc_kinetic_energy(sample_fn, params, eval_rng,
                                                          batch_size=max(batch_size // 16, 1),
                                                          t_size=max(t_size // 10, 1), dim=dim))
    if verbose:
      print("kinetic energy with more samples: {:.3e}".format(out["kinetic_more"]))
      print("kinetic energy with less samples: {:.3e}".format(out["kinetic_less"]))
  elif _type == "rwpo":
    r = config["rwpo"]
    T = r["T"] if T is None else T
    beta, a, subtype = r["beta"], r["a"], r["pot_type"]
    out["e_kin"] = T * float(utils.calc_score_kinetic_energy(sample_fn, log_prob_fn, params, T, beta, dim, eval_rng,
                                                             batch_size=batch_size, t_size=t_size))
    out["e_pot"] = float(applications.potential_loss_fn(model, dim, a, subtype, params, T, eval_rng, batch_size))
    if verbose:
      print(f"kinetic energy: {out['e_kin']:.3e}")
      print(f"potential energy: {out['e_pot']:.3e}")
    if subtype == "quadratic":
      # the true value for the quadratic potential and Gaussian initial condition (solvers.py:170-172)
      true_val = dim * (1 + math.log(T + 1)) / beta
      out["true_val"] = true_val
      out["relative_err_percent"] = (out["e_kin"] + out["e_pot"] - true_val) / true_val * 100
      if verbose:
        print("total energy: {:.3e}|relative err: {:.3e}".format(out["e_kin"] + out["e_pot"],
                                                                out["relative_err_percent"]))
    elif subtype == "double_well" and dim == 2:
      # the flow's density at t = T on the 100 x 100 grid of [-2, 2]^2 (solvers.py:184-222; the reference compares it
      # with an interpolated reference solution whose data file is not shipped)
      out["density_T"] = utils.density_on_grid(log_prob_fn, params, [T], [-2, 2, -2, 2], 100)[0]
  elif _type == "fp":
    # solvers.py:238-306: L2 error against the Ornstein-Uhlenbeck solution (valid for the drift -a r), Monte-Carlo and,
    # for dim 2, on a 500 x 500 grid
    f = config["fp"]
    T = f["T"] if T is None else T
    out["rmse_mc"] = float(utils.rmse_mc_loss_fn(model, params, 1, eval_rng, 1000000, a=f["a"], T=T))
    if verbose:
      print("L2 error via Monte-Carlo: {:.3e}".format(out["rmse_mc"]))
    if dim == 2:
      out["rmse_grid"] = float(utils.rmse_grid_loss_fn(log_prob_fn, params, 1, 500, a=f["a"], T=T))
      if verbose:
        print("L2 error on grid: {:.3e}".format(out["rmse_grid"]))
  return out


if __name__ == "__main__":
  import os
  import yaml
  here = os.path.dirname(os.path.abspath(__file__))
  with open(os.path.join(here, "config", "mfc.yaml"), "r") as file:
    config_dict = yaml.safe_load(file)
  params, _ = main(config_dict, progress=True)
  model, _, _ = build(config_dict)
  evaluate(config_dict, model, params, random.PRNGKey(config_dict["general"]["seed"] + 1))
