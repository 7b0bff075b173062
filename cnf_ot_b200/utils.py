"""Evaluation energies of the MFC solvers -- the callers right after the train step.

Mirrors `calc_kinetic_energy` / `calc_score_kinetic_energy` of
/root/reference/cnf_ot/utils.py:311-389 (called from cnf_ot/mfc/solvers.py:141-164): same
names, arguments and return values, but each is ONE forward-only CUDA kernel over a chunk of the
time grid (cnfot_kinetic_energy) instead of 2-(3+2 dim) flow evaluations per time in Python.
As in the reference every time of the grid gets a fresh N(0, I) batch (`rng` is split per time);
equal `rng` => equal result.
"""
from __future__ import annotations

import torch

from . import ops, random
from .flows import _blob_of

_T_CHUNK = 128  # times per launch: bounds the latent buffer at _T_CHUNK * batch_size rows


def _model_of(sample_fn):
  model = getattr(sample_fn, "__self__", None)
  if model is None or not hasattr(model, "shape"):
    raise TypeError("sample_fn must be `model.apply.sample` of a cnf_ot_b200 flow model")
  return model


def _energy(model, params, rng, batch_size, t_array, with_score, kappa):
  W = _blob_of(model.shape, params, model.device)
  total = torch.zeros((), dtype=torch.float64, device=model.device)
  n_t = len(t_array)
  rng = random.as_key(rng)
  for lo in range(0, n_t, _T_CHUNK):
    ts = t_array[lo:lo + _T_CHUNK]
    _rng, rng = random.split(rng)
    latent = random.normal(_rng, (len(ts) * batch_size, model.shape.dim), device=model.device)
    e = ops.kinetic_energy(model.shape, W, latent, ts, dt=0.01, with_score=with_score, kappa=kappa, dx=0.01,
                           latent_blocks=len(ts))
    total += e * (len(ts) / n_t)
  return total


def calc_kinetic_energy(sample_fn, params, rng, batch_size: int = 65536, t_size: int = 10000, dim: int = 1):
  """Monte-Carlo kinetic energy, utils.py:311-340: mean over t in linspace(0, 1, t_size) of
  mean(((r(t+dt/2) - r(t-dt/2)) / dt)^2) / 2 * dim, dt = 0.01."""
  model = _model_of(sample_fn)
  if dim != model.shape.dim:
    raise ValueError(f"dim={dim} does not match the flow's dimension {model.shape.dim}")
  t_array = torch.linspace(0, 1, t_size, dtype=torch.float64).tolist()
  return _energy(model, params, rng, batch_size, t_array, False, 0.0)


def calc_score_kinetic_energy(sample_fn, log_prob_fn, params, T: float = 1, beta: float = 1, dim: int = 1,
                              rng=random.PRNGKey(0), batch_size: int = 65536, t_size: int = 10000):
  """Kinetic energy with the score-corrected velocity, utils.py:343-389 (dx = dt = 0.01,
  velocity += score / beta); t in linspace(0, T, t_size).  `log_prob_fn` is accepted for signature
  parity; the kernel evaluates the same model's log-density."""
  model = _model_of(sample_fn)
  if getattr(log_prob_fn, "__self__", model) is not model:
    raise TypeError("sample_fn and log_prob_fn must belong to the same model")
  if dim != model.shape.dim:
    raise ValueError(f"dim={dim} does not match the flow's dimension {model.shape.dim}")
  t_array = torch.linspace(0, T, t_size, dtype=torch.float64).tolist()
  return _energy(model, params, rng, batch_size, t_array, True, 1.0 / beta)


# ------------------------------------------------------------------ densities on grids / at samples (SURVEY.md §8f row 3)
# The numerical content of the reference's plotting helpers and of the fp evaluation tail, without matplotlib:
# each is ONE kernel launch (cnfot_density_grid / cnfot_density_mc; wide flows: one flow pass per row chunk on the
# wide-conditioner engine), the grid generated on chip.
def _model_of_fn(fn):
  model = getattr(fn, "__self__", None)
  if model is None or not hasattr(model, "shape"):
    raise TypeError("expected `model.apply.<fn>` of a cnf_ot_b200 flow model")
  return model


def density_on_grid(log_prob_fn, params, t_array, domain_range, n: int = 100):
  """exp(log_prob_fn(params, XY, cond = t)).reshape(n, n) for every t of `t_array`, XY = the n x n grid of
  domain_range = [x_min, x_max, y_min, y_max] -- exactly what `plot_density_snapshot` (utils.py:572-595, domain
  [-6, 6]^2, ten times) and `plot_density_and_trajectory` (utils.py:598-642) hand to `imshow`, and the `prob1` of the
  double-well evaluation (solvers.py:184-222, [-2, 2]^2 at t = T).  Returns a (len(t_array), n, n) CUDA tensor."""
  model = _model_of_fn(log_prob_fn)
  W = _blob_of(model.shape, params, model.device)
  dens, _ = ops.density_grid(model.shape, W, [float(t) for t in t_array], domain_range, n, n)
  return dens


def plot_density_snapshot(log_prob_fn, params, t_array=None):
  """utils.py:572-595 without the figure: the ten 100 x 100 density snapshots on [-6, 6]^2."""
  t_array = torch.linspace(0, 1, 10, dtype=torch.float64).tolist() if t_array is None else t_array
  return density_on_grid(log_prob_fn, params, t_array, [-6, 6, -6, 6], 100)


def trajectories(forward_fn, inverse_fn, params, r_, t_array):
  """utils.py:619-627: xi = inverse_fn(params, r_, 0); r(t) = forward_fn(params, xi, t) for every t.
  Returns (len(t_array), rows, dim)."""
  xi = inverse_fn(params, r_, torch.zeros(1))
  return torch.stack([forward_fn(params, xi, torch.ones(1) * float(t)) for t in t_array])


def _fp_reference_variances(a: float, T: float):
  """source N(0, 4 I), target N(0, (exp(-2 a T) (4 - 1/(2a)) + 1/(2a)) I): solvers.py:238-252."""
  import math
  return 4.0, math.exp(-2 * a * T) * (4 - 1 / 2 / a) + 1 / 2 / a


def rmse_grid_loss_fn(log_prob_fn, params, cond: float, grid_size: int, a: float = 1.0, T: float = 1.0):
  """solvers.py:282-301: sqrt(mean((exp(log_prob(XY, cond)) - (source (1 - cond) + target cond))^2)) on the
  grid_size x grid_size grid of [-5, 5]^2 (the reference calls it with cond = 1, grid_size = 500)."""
  model = _model_of_fn(log_prob_fn)
  W = _blob_of(model.shape, params, model.device)
  v0, v1 = _fp_reference_variances(a, T)
  _, sq = ops.density_grid(model.shape, W, [float(cond)], [-5, 5, -5, 5], grid_size, grid_size, ref=(float(cond), v0, v1),
                           want_density=False)
  return torch.sqrt(sq / (grid_size * grid_size))


def rmse_mc_loss_fn(model, params, cond: float, rng, batch_size: int, a: float = 1.0, T: float = 1.0):
  """solvers.py:254-278: the same error at `batch_size` samples of the flow itself (the reference: cond = 1, 10^6
  samples).  The latent is the draw `model.apply.sample(seed=rng, sample_shape=(batch_size,))` makes."""
  W = _blob_of(model.shape, params, model.device)
  v0, v1 = _fp_reference_variances(a, T)
  _, _, sq = ops.density_mc(model.shape, W, float(cond), random.as_key(rng).value, batch_size, ref=(float(cond), v0, v1))
  return torch.sqrt(sq / batch_size)
