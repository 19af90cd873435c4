"""Dopri5 dense output -- diffeqsolve(..., saveat=SaveAt(ts=ts)) -- restated for the save-time tests.

``oracle.ecnf_oracle.dopri5`` is the pinned restatement of diffeqsolve and reports the end of the solve only.
``dopri5_saveat`` below runs the same step sequence (same tableau, controller and per-row bookkeeping;
tests/test_saveat_host.py checks that its end state and step counts are bit for bit the oracle's) and in addition fills
the save times from the accepted steps.

Restated from diffrax / torchdiffeq, neither of which is installed here (like ``DP_BERR`` in the oracle): a save time tau
in the internal interval (tprev, tnext] of an accepted step, s = (tau - tprev) / dt, is read from the 4th-order
interpolant of that step (torchdiffeq ``_interp_fit``), built from y0, y1 = the 5th-order solution, the seven stage
increments k_i = dt * F_i (k_6 = the FSAL stage at (tnext, y1)) and y_mid = y0 + sum_i DP_C_MID[i] k_i.  DP_C_MID is
recalled from memory, not read from diffrax; a time equal to tnext returns y1 itself, a time equal to the start time y0.
"""
from typing import Callable, Optional, Sequence, Tuple

import numpy as np
import torch

from oracle import ecnf_oracle as O

DP_C_MID = tuple(c / 2 for c in (6025192743 / 30085553152, 0.0, 51252292925 / 65400821598, -2691868925 / 45128329728,
                                 187940372067 / 1594534317056, -1776094331 / 19743644256, 11237099 / 235043384))


def dopri5_interp(y0: torch.Tensor, y1: torch.Tensor, k: Sequence[torch.Tensor], s: float) -> torch.Tensor:
    """The dense output of one step at the fraction s in [0, 1] of the step."""
    y_mid = y0 + sum(c * kk for c, kk in zip(DP_C_MID, k) if c != 0.0)
    k0, k6 = k[0], k[6]
    a = 2 * (k6 - k0) - 8 * (y1 + y0) + 16 * y_mid
    b = 5 * k0 - 3 * k6 + 18 * y0 + 14 * y1 - 32 * y_mid
    c = k6 - 4 * k0 - 11 * y0 - 5 * y1 + 16 * y_mid
    return (((a * s + b) * s + c) * s + k0) * s + y0


def dopri5_saveat(func: Callable[[torch.Tensor, torch.Tensor], torch.Tensor], y0: torch.Tensor, t0: float, t1: float,
                  ctrl: "O.SolveControl", ts: Optional[Sequence[float]] = None
                  ) -> Tuple[torch.Tensor, "O.SolveStats", Optional[torch.Tensor]]:
    """``oracle.dopri5`` + the path [B, n_save, S] at the times ``ts`` (monotone in the direction t0 -> t1; NaN in the rows
    a trajectory stopped on max_steps never reached).  Without ``ts`` the third result is None."""
    B, S = y0.shape
    dt_ = y0.dtype
    direction = 1.0 if t0 < t1 else -1.0
    T0, T1 = t0 * direction, t1 * direction
    tol_clip = 1e-10 if dt_ == torch.float64 else 1e-6
    n_evals = np.zeros(B, np.int64)
    tau_s = [direction * float(t) for t in (ts if ts is not None else [])]
    path = torch.full((B, len(tau_s), S), float("nan"), dtype=dt_) if ts is not None else None
    nxt = np.zeros(B, np.int64)

    def f(tau, y, mask=None):
        out = direction * func(direction * tau, y)
        n_evals[(np.ones(B, bool) if mask is None else mask.numpy())] += 1
        return out

    def clip_to_end(tprev, tnext, keep):
        clip = tnext > T1 - tol_clip
        tclip = torch.where(keep, torch.full_like(tnext, T1), tprev + 0.5 * (T1 - tprev))
        return torch.where(clip, tclip, tnext)

    tprev = torch.full((B,), T0, dtype=dt_)
    y = y0.clone()
    for r in range(B):
        while nxt[r] < len(tau_s) and tau_s[nxt[r]] <= T0:
            path[r, nxt[r]] = y[r]
            nxt[r] += 1
    f0 = f(tprev, y)
    if ctrl.fixed:
        dt0 = torch.full((B,), abs(ctrl.step_size), dtype=dt_)
    else:
        scale = ctrl.atol + y.abs() * ctrl.rtol
        d0, d1 = O._rms(y / scale), O._rms(f0 / scale)
        cond = (d0 < 1e-5) | (d1 < 1e-5)
        h0 = torch.where(cond, torch.full_like(d0, 1e-6), 0.01 * d0 / torch.where(cond, torch.ones_like(d1), d1))
        f1 = f(tprev + h0, y + h0[:, None] * f0)
        d2 = O._rms((f1 - f0) / scale) / h0
        md = torch.maximum(d1, d2)
        h1 = torch.where(md <= 1e-15, torch.maximum(torch.full_like(h0, 1e-6), h0 * 1e-3),
                         (0.01 / md) ** (1.0 / ctrl.error_order))
        dt0 = torch.minimum(100 * h0, h1)
        dt0 = torch.clamp(dt0, min=ctrl.dtmin)
    tnext = clip_to_end(tprev, tprev + dt0, torch.ones(B, dtype=torch.bool))
    at_dtmin = torch.zeros(B, dtype=torch.bool)
    n_steps = np.zeros(B, np.int32)
    n_acc = np.zeros(B, np.int32)
    status = np.zeros(B, np.int32)
    active = tprev < T1
    while bool(active.any()):
        dt = tnext - tprev
        k = [f0 * dt[:, None]]
        for s in range(1, 7):
            ys = y.clone()
            for j, a in enumerate(O.DP_A[s]):
                if a != 0.0:
                    ys = ys + a * k[j]
            fs = f(tprev + O.DP_C[s] * dt, ys, active)
            k.append(fs * dt[:, None])
        y1 = ys
        yerr = sum(c * kk for c, kk in zip(O.DP_BERR, k) if c != 0.0)
        if ctrl.fixed:
            keep = torch.ones(B, dtype=torch.bool)
            new_prev, new_next = tnext, tnext + dt
        else:
            sc = ctrl.atol + torch.maximum(y.abs(), y1.abs()) * ctrl.rtol
            err = O._rms(ctrl.err_scale * yerr / sc)
            keep = (err < 1) | at_dtmin
            inv = torch.where(err == 0, torch.full_like(err, float("inf")), 1.0 / err)
            factor = ctrl.safety * inv ** (1.0 / ctrl.error_order)
            fmin = torch.where(keep, torch.ones_like(err), torch.full_like(err, ctrl.factormin))
            factor = torch.minimum(torch.maximum(factor, fmin), torch.full_like(err, ctrl.factormax))
            ndt = dt * factor
            new_at = ndt <= ctrl.dtmin
            ndt = torch.clamp(ndt, min=ctrl.dtmin)
            new_prev = torch.where(keep, tnext, tprev)
            new_next = new_prev + ndt
            at_dtmin = torch.where(active, new_at, at_dtmin)
        new_prev = torch.minimum(new_prev, torch.full_like(new_prev, T1))
        new_next = clip_to_end(new_prev, new_next, keep)
        upd = active & keep
        for r in np.flatnonzero(upd.numpy()):                  # save times in (tprev, tnext] of an accepted step
            while nxt[r] < len(tau_s) and tau_s[nxt[r]] <= float(tnext[r]):
                tau = tau_s[nxt[r]]
                if tau < float(tnext[r]):
                    s = (tau - float(tprev[r])) / float(dt[r])
                    path[r, nxt[r]] = dopri5_interp(y[r], y1[r], [kk[r] for kk in k], s)
                else:
                    path[r, nxt[r]] = y1[r]
                nxt[r] += 1
        y = torch.where(upd[:, None], y1, y)
        f0 = torch.where(upd[:, None], fs, f0)
        tprev = torch.where(active, new_prev, tprev)
        tnext = torch.where(active, new_next, tnext)
        n_steps += active.numpy().astype(np.int32)
        n_acc += upd.numpy().astype(np.int32)
        hit = active.numpy() & (n_steps >= ctrl.max_steps) & (tprev < T1).numpy()
        status[hit] = 1
        active = active & (tprev < T1) & torch.as_tensor(n_steps < ctrl.max_steps)
    return y, O.SolveStats(n_steps, n_acc, n_evals.astype(np.int32), status), path


# --- the three drivers of oracle.ecnf_oracle with a path: (oracle results..., path [B, n_save, S])
def sample_cnf(p, cfg, x0, feat, ctrl, ts):
    def func(t, y):
        with torch.no_grad():
            return O.egnn_apply(p, cfg, y, t, feat)
    y1, st, path = dopri5_saveat(func, x0, 0.0, 1.0, ctrl, ts)
    return y1, st, path


def sample_and_log_prob_cnf(p, cfg, x0, feat, ctrl, ts, eps=None):
    y0 = torch.cat([x0, torch.zeros(x0.shape[0], 1, dtype=x0.dtype)], dim=1)
    y1, st, path = dopri5_saveat(O._joint(p, cfg, feat, eps), y0, 0.0, 1.0, ctrl, ts)
    return y1[:, :-1], O.base_log_prob(cfg, x0) - y1[:, -1], st, path


def get_log_prob(p, cfg, x, feat, ctrl, ts, eps=None):
    y0 = torch.cat([x, torch.zeros(x.shape[0], 1, dtype=x.dtype)], dim=1)
    y1, st, path = dopri5_saveat(O._joint(p, cfg, feat, eps), y0, 1.0, 0.0, ctrl, ts)
    lpb = O.base_log_prob(cfg, y1[:, :-1])
    return lpb + y1[:, -1], lpb, y1[:, -1], st, path
