"""Mirror of ecnf/cnf/sample_and_log_prob.py.  The reference functions are per-trajectory and meant to be
jax.vmap-ed (setup_training.py:47,197) or lax.scan-ned (setup_training.py:180); here a leading batch axis is
accepted directly and every trajectory runs its own adaptive Dopri5 loop on the GPU.

Differences, all documented in DESIGN.md:
  * `approx=True` runs the Hutchinson estimator with one fixed probe per trajectory (`eps=` injects it);
  * noise can be injected (`x0=`) so parity tests bypass the RNG; a jax-style key (uint32[2], or [B, 2] per-trajectory
    keys) reproduces the reference's threefry draws on the host (utils/jax_random.py); an integer seed uses the library's
    Philox stream keyed by (seed, global sample index) on the device (the fast path);
  * the fixed-step branch of sample_and_log_prob_cnf integrates (x0, 0) -- the reference passes y0=x0 there and
    cannot run (sample_and_log_prob.py:140);
  * diffrax raises when max_steps (4096) is reached; the kernel flags the trajectory in its stats row, and the wrappers
    raise EcnfError from that flag by default (`check_status=False` skips the device->host read on hot paths).

`ts=` is diffeqsolve's `saveat=SaveAt(ts=ts)` (at most 1024 times in [0, 1], in the direction of integration): the
functions then also return the path, `xs` [B, n_save, D] and, in the log-density modes, `delta_ts` [B, n_save], the
divergence integral from the start time to each ts[k].  Along a sample path log q_t(x_t) = log p0(x0) - delta_ts; along
the get_log_prob path from the data x (t = 1) towards t = 0, log q_t(x_t) = log_p - delta_ts.  Interior times come from the
Dopri5 dense output; the step sequence, and so every other output, is the same as without `ts`.
"""
from typing import Optional, Tuple

import torch

from .. import lib as L
from ..utils import jax_random as jr
from .core import FlowMatchingCNF


def _batch(features, n_frames: int, n_samples: Optional[int]):
    if features is not None:
        f = torch.as_tensor(features)
        if f.dim() >= 2:
            return f.reshape(-1, n_frames).shape[0], False
    if n_samples is not None:
        return int(n_samples), False
    return 1, True


def _jax_keys(key, B: int):
    """Per-trajectory jax keys: [B, 2] as given, a single key for one trajectory, or `jax.random.split(key, B)` -- what the
    reference's callers vmap over (setup_training.py:47)."""
    k = jr.as_key(key)
    if k.ndim == 1:
        return k[None] if B == 1 else jr.split(k, B)
    return k.reshape(-1, 2)


def _jax_base_and_eps(eng, key, B: int, want_eps: bool):
    """x0 = cnf.sample_base(key_i, 1)[0] per trajectory and (Hutchinson) eps_i = jax.random.normal(key_i, (D,)), the raw
    noise under the same key (sample_and_log_prob.py:55,130; SURVEY C#6), restated on the host."""
    c = eng.cfg
    keys = _jax_keys(key, B)
    x0 = torch.from_numpy(jr.sample_base_per_key(keys, c.n_frames, c.dim, c.base_scale)).to(eng.device)
    eps = None
    if want_eps:
        eps = torch.from_numpy(jr.normal_per_key(keys, c.D)).to(eng.device)
    return x0, eps


def sample_cnf(cnf: FlowMatchingCNF, params, key, features=None, use_fixed_step_size: bool = False,
               rtol: float = 1e-5, atol: float = 1e-5, step_size: float = 0.05, *, n_samples: Optional[int] = None,
               x0=None, global_offset: int = 0, return_stats: bool = False, check_status: bool = True, ts=None):
    """ecnf/cnf/sample_and_log_prob.py:11-38: returns x1, or (x1, xs) with `ts=`."""
    eng = cnf.engine
    if x0 is not None:
        x0 = torch.as_tensor(x0, dtype=torch.float32, device=eng.device)
        single = x0.dim() == 1
        x0 = x0.reshape(-1, eng.cfg.D)
    else:
        B, single = _batch(features, eng.cfg.n_frames, n_samples)
        if jr.is_key(key):
            if jr.as_key(key).ndim == 2:
                B, single = jr.as_key(key).shape[0], False
            x0, _ = _jax_base_and_eps(eng, key, B, False)
        else:
            x0 = eng.base_sample(key, B, global_offset)
    ctrl = L.make_ctrl(use_fixed_step_size, rtol, atol, step_size)
    res = eng.solve(params, L.MODE_SAMPLE, x0, features, ctrl, ts=ts)
    x1, stats = res[0], res[2]
    if check_status:
        eng.check_status(stats, "sample_cnf")
    if ts is None:
        out = x1[0] if single else x1
        return (out, stats) if return_stats else out
    xs = res[3]
    out = (x1[0], xs[0]) if single else (x1, xs)
    return (*out, stats) if return_stats else out


def get_log_prob(cnf: FlowMatchingCNF, params, x, key=None, features=None, approx: bool = False,
                 use_fixed_step_size: bool = False, rtol: float = 1e-5, atol: float = 1e-5, step_size: float = 0.05,
                 *, eps=None, global_offset: int = 0, return_stats: bool = False,
                 check_status: bool = True, ts=None) -> Tuple[torch.Tensor, ...]:
    """ecnf/cnf/sample_and_log_prob.py:41-94: returns (log_p, log_prob_base, delta), + (xs, delta_ts) with `ts=` (times
    decreasing from 1 towards 0).  approx=True = the Hutchinson branch (:69-78): one probe eps ~ N(0, I) per trajectory,
    drawn once from `key` (:55) -- or injected with `eps=`."""
    eng = cnf.engine
    x = torch.as_tensor(x, dtype=torch.float32, device=eng.device)
    single = x.dim() == 1
    x = x.reshape(-1, eng.cfg.D)
    ctrl = L.make_ctrl(use_fixed_step_size, rtol, atol, step_size)
    if approx and eps is None:
        if key is None:
            raise L.EcnfError("get_log_prob(approx=True) draws its Hutchinson probe from `key` "
                              "(sample_and_log_prob.py:55): pass key= (jax-style uint32[2] or an integer seed) or eps=")
        if jr.is_key(key):
            eps = torch.from_numpy(jr.normal_per_key(_jax_keys(key, x.shape[0]), eng.cfg.D)).to(eng.device)
        else:
            eps = eng.normal_noise(key, x.shape[0], global_offset, substream=1)
    res = eng.solve(params, L.MODE_LOGPROB, x, features, ctrl, eps=eps if approx else None, ts=ts)
    logs, stats = res[1], res[2]
    if check_status:
        eng.check_status(stats, "get_log_prob")
    out = (logs[0, 0], logs[0, 1], logs[0, 2]) if single else (logs[:, 0], logs[:, 1], logs[:, 2])
    if ts is not None:
        out = (*out, res[3][0], res[4][0]) if single else (*out, res[3], res[4])
    return (*out, stats) if return_stats else out


def sample_and_log_prob_cnf(cnf: FlowMatchingCNF, params, key, features=None, approx: bool = False,
                            use_fixed_step_size: bool = False, rtol: float = 1e-5, atol: float = 1e-5,
                            step_size: float = 0.05, *, n_samples: Optional[int] = None, x0=None, eps=None,
                            global_offset: int = 0, return_stats: bool = False, check_status: bool = True, ts=None):
    """ecnf/cnf/sample_and_log_prob.py:97-149: returns (x1, log_q), + (xs, delta_ts) with `ts=`.  approx=True = the Hutchinson branch (:123-133); the
    reference draws its probe from the SAME key as the base sample (:130,137; SURVEY C#6), which here means the raw noise
    underneath `sample_base(key)` (substream 0) -- or inject it with `eps=`."""
    eng = cnf.engine
    if x0 is not None:
        x0 = torch.as_tensor(x0, dtype=torch.float32, device=eng.device)
        single = x0.dim() == 1
        x0 = x0.reshape(-1, eng.cfg.D)
    else:
        B, single = _batch(features, eng.cfg.n_frames, n_samples)
        if jr.is_key(key):
            if jr.as_key(key).ndim == 2:
                B, single = jr.as_key(key).shape[0], False
            x0, eps_j = _jax_base_and_eps(eng, key, B, approx and eps is None)
            eps = eps_j if eps is None else eps
        else:
            x0 = eng.base_sample(key, B, global_offset)
    ctrl = L.make_ctrl(use_fixed_step_size, rtol, atol, step_size)
    if approx and eps is None:
        # x0 was injected: the probe still comes from `key`, as the reference draws it (sample_and_log_prob.py:130)
        if key is None:
            raise L.EcnfError("sample_and_log_prob_cnf(approx=True) with x0= given needs key= or eps= for the probe")
        if jr.is_key(key):
            eps = torch.from_numpy(jr.normal_per_key(_jax_keys(key, x0.shape[0]), eng.cfg.D)).to(eng.device)
        else:
            eps = eng.normal_noise(key, x0.shape[0], global_offset, substream=0)
    res = eng.solve(params, L.MODE_SAMPLE_LOGQ, x0, features, ctrl, eps=eps if approx else None, ts=ts)
    x1, logs, stats = res[:3]
    if check_status:
        eng.check_status(stats, "sample_and_log_prob_cnf")
    out = (x1[0], logs[0, 0]) if single else (x1, logs[:, 0])
    if ts is not None:
        out = (*out, res[3][0], res[4][0]) if single else (*out, res[3], res[4])
    return (*out, stats) if return_stats else out
