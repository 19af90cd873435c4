"""Host-side engine: owns the library model handle, the packed parameter buffer and workspaces, and exposes the
batched primitives the reference-shaped façade (ecnf_b200.cnf.*, ecnf_b200.nets.*) is built from.

torch supplies device memory, streams and (in ecnf_b200.distributed) NCCL; all arithmetic of the hot path happens
in libecnf_b200.so.  Nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import lib as L


@dataclass(frozen=True)
class CnfConfig:
    """Arguments of the reference's build_cnf (ecnf/cnf/build_cnf.py:34-44)."""
    n_frames: int
    dim: int
    sigma_min: float
    base_scale: float
    n_blocks_egnn: int
    mlp_units: Tuple[int, ...]
    n_invariant_feat_hidden: int
    time_embedding_dim: int
    n_features: int
    normalization_constant: float = 1.0

    @property
    def D(self) -> int:
        return self.n_frames * self.dim


def timestep_frequencies(T: int) -> np.ndarray:
    """fp32 table of build_cnf.py:25-27 evaluated the way jnp does with x64 off."""
    half = T // 2
    emb = np.float32(np.log(np.float32(10_000.0)) / np.float32(half - 1))
    return np.exp(np.arange(half, dtype=np.float32) * -emb).astype(np.float32)


def key_to_seed(key) -> int:
    """Accept an int, or a jax-style uint32[2] key, and fold it into the 64-bit Philox seed."""
    if isinstance(key, (int, np.integer)):
        return int(key) & 0xFFFFFFFFFFFFFFFF
    arr = np.asarray(key.detach().cpu() if isinstance(key, torch.Tensor) else key).astype(np.uint64).ravel()
    if arr.size == 1:
        return int(arr[0])
    return int((arr[0] << np.uint64(32)) | (arr[1] & np.uint64(0xFFFFFFFF)))


def split_key(key, num: int = 2) -> List[int]:
    """Deterministic stand-in for jax.random.split (threefry is not reproducible without jax): SplitMix64."""
    s = key_to_seed(key)
    out = []
    for _ in range(num):
        s = (s + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        z = s
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        out.append(z ^ (z >> 31))
    return out


class PackedParams:
    """Flat fp32 device buffer in the library's aligned layout (+ the pytree view for the caller)."""

    def __init__(self, flat: torch.Tensor):
        self.flat = flat


def _stream_ptr() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


class Engine:
    def __init__(self, cfg: CnfConfig, device: Optional[torch.device] = None):
        units = tuple(int(u) for u in cfg.mlp_units)
        if len(set(units)) != 1:
            raise L.EcnfError(f"mlp_units must be uniform (every shipped reference config is), got {units}")
        self.cfg = cfg
        self.lib = L.load()
        ccfg = L.Config()
        ccfg.n_frames, ccfg.dim, ccfg.n_blocks, ccfg.n_layers = cfg.n_frames, cfg.dim, cfg.n_blocks_egnn, len(units)
        ccfg.mlp_units, ccfg.n_hidden, ccfg.time_dim = units[0], cfg.n_invariant_feat_hidden, cfg.time_embedding_dim
        ccfg.n_features = int(cfg.n_features)
        ccfg.sigma_min, ccfg.base_scale = float(cfg.sigma_min), float(cfg.base_scale)
        ccfg.normalization_constant = float(cfg.normalization_constant)
        fr = timestep_frequencies(cfg.time_embedding_dim)
        for k in range(8):
            ccfg.freqs[k] = float(fr[k]) if k < len(fr) else 0.0
        handle = C.c_void_p()
        L.check(self.lib.ecnf_model_create(C.byref(ccfg), None, C.byref(handle)), "ecnf_model_create")
        self.handle = handle
        self.param_count = int(self.lib.ecnf_model_param_count(handle))
        self.layout: List[Tuple[str, int, Tuple[int, ...]]] = []
        name = C.create_string_buffer(256)
        off, rows, cols = C.c_int64(), C.c_int64(), C.c_int64()
        for i in range(self.lib.ecnf_model_num_tensors(handle)):
            L.check(self.lib.ecnf_model_param_layout(handle, i, name, 256, C.byref(off), C.byref(rows), C.byref(cols)),
                    "ecnf_model_param_layout")
            path = name.value.decode()
            if path.endswith("final_scaling"):
                shape: Tuple[int, ...] = ()
            elif cols.value == 0:
                shape = (rows.value,)
            else:
                shape = (rows.value, cols.value)
            self.layout.append((path, off.value, shape))
        self._device = device
        self._ws: Dict[Tuple[str, int], torch.Tensor] = {}
        self._pack_cache: Dict[int, Tuple[object, PackedParams]] = {}
        self._bound: Optional[torch.Tensor] = None

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.ecnf_model_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # ---------------------------------------------------------------- device / params
    @property
    def device(self) -> torch.device:
        if self._device is None:
            if not torch.cuda.is_available():
                raise L.EcnfError("ecnf_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
            self._device = torch.device("cuda", torch.cuda.current_device())
        return self._device

    def pack(self, params) -> PackedParams:
        """flax-style pytree ({'params': {...}} of numpy / torch arrays) -> PackedParams. Cached per object."""
        if isinstance(params, PackedParams):
            return params
        hit = self._pack_cache.get(id(params))
        if hit is not None and hit[0] is params:
            return hit[1]
        flat_host = np.zeros(self.param_count, np.float32)
        tree = params.get("params", params)
        for path, off, shape in self.layout:
            node = tree
            for part in path.split("/"):
                if part not in node:
                    raise L.EcnfError(f"parameter pytree is missing '{path}'")
                node = node[part]
            arr = node.detach().cpu().numpy() if isinstance(node, torch.Tensor) else np.asarray(node)
            if tuple(arr.shape) != tuple(shape):
                raise L.EcnfError(f"parameter '{path}' has shape {tuple(arr.shape)}, expected {tuple(shape)}")
            flat_host[off:off + arr.size] = arr.astype(np.float32).ravel()
        packed = PackedParams(torch.from_numpy(flat_host).to(self.device))
        if len(self._pack_cache) >= 8:
            self._pack_cache.pop(next(iter(self._pack_cache)))
        self._pack_cache[id(params)] = (params, packed)
        return packed

    def unpack(self, packed: Union[PackedParams, torch.Tensor], to_numpy: bool = False) -> dict:
        """PackedParams -> flax-style pytree of views (torch, on device) or numpy copies."""
        flat = packed.flat if isinstance(packed, PackedParams) else packed
        host = flat.detach().cpu().numpy() if to_numpy else None
        root: dict = {}
        for path, off, shape in self.layout:
            cnt = int(np.prod(shape)) if shape else 1
            v = (host[off:off + cnt].reshape(shape).copy() if to_numpy else flat[off:off + cnt].view(shape))
            d = root
            parts = path.split("/")
            for p in parts[:-1]:
                d = d.setdefault(p, {})
            d[parts[-1]] = v
        return {"params": root}

    def _bind(self, packed: PackedParams) -> None:
        if packed.flat.numel() != self.param_count or packed.flat.dtype != torch.float32 or not packed.flat.is_cuda:
            raise L.EcnfError("packed parameter buffer has the wrong size / dtype / device")
        if self._bound is None or self._bound.data_ptr() != packed.flat.data_ptr():
            L.check(self.lib.ecnf_model_set_params(self.handle, _ptr(packed.flat)), "ecnf_model_set_params")
            self._bound = packed.flat

    def _workspace(self, tag: str, nbytes: int) -> torch.Tensor:
        """Scratch for one library call, keyed by (kind, current stream): calls issued on different streams never
        share a buffer (calls on one stream are ordered, so they may)."""
        key = (tag, torch.cuda.current_stream().cuda_stream)
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=self.device)
            self._ws[key] = ws
        return ws

    def set_engine(self, engine: int) -> None:
        """0 = tensor cores where the shape is eligible (default), 1 = fp32 SIMT everywhere.  Per model handle."""
        L.check(self.lib.ecnf_model_set_engine(self.handle, int(engine)), "ecnf_model_set_engine")

    def set_fm_chunk(self, graphs: int) -> None:
        """Graphs per chunk of a training minibatch (gradients accumulate over the chunks); 0 = the whole minibatch."""
        L.check(self.lib.ecnf_model_set_fm_chunk(self.handle, int(graphs)), "ecnf_model_set_fm_chunk")

    @staticmethod
    def check_status(stats: torch.Tensor, what: str) -> None:
        """diffrax raises when max_steps is reached (throw=True); the kernel flags the trajectory instead.  This is the
        raise: one device->host read of the status column."""
        bad = torch.nonzero(stats[:, 3] != 0).flatten()
        if bad.numel():
            head = ", ".join(str(int(i)) for i in bad[:8].tolist())
            raise L.EcnfError(f"{what}: {bad.numel()} of {stats.shape[0]} trajectories reached max_steps before the end "
                              f"time (first: {head}); their outputs are partial.  Pass check_status=False to get the "
                              "raw results and inspect return_stats=True yourself.")

    def _prep(self, x, feat, B_hint=None):
        dev = self.device
        x = torch.as_tensor(x, dtype=torch.float32, device=dev).contiguous()
        if x.dim() != 2 or x.shape[1] != self.cfg.D:
            raise L.EcnfError(f"positions must be [B, {self.cfg.D}], got {tuple(x.shape)}")
        B = x.shape[0]
        feat = self.features(feat, B)
        return x, feat, B

    def features(self, feat, B: int) -> torch.Tensor:
        n = self.cfg.n_frames
        if feat is None:
            return torch.zeros(B, n, dtype=torch.int32, device=self.device)
        f = torch.as_tensor(feat, device=self.device)
        f = f.reshape(-1, n) if f.dim() != 1 else f.reshape(1, n)
        if f.shape[0] == 1 and B > 1:
            f = f.expand(B, n)
        if f.shape[0] != B:
            raise L.EcnfError(f"features must be [B={B}, {n}], got {tuple(f.shape)}")
        return f.to(torch.int32).contiguous()

    # ---------------------------------------------------------------- vector field
    def apply(self, params, x, t, feat=None) -> torch.Tensor:
        packed = self.pack(params)
        self._bind(packed)
        x, feat, B = self._prep(x, feat)
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device).reshape(-1).contiguous()
        if t.numel() != B:
            raise L.EcnfError(f"t must have {B} entries, got {t.numel()}")
        out = torch.empty_like(x)
        nb = int(self.lib.ecnf_solve_workspace_bytes(self.handle, L.MODE_VF, B))
        ws = self._workspace("solve", nb)
        L.check(self.lib.ecnf_vf_forward(self.handle, _ptr(x), _ptr(t), _ptr(feat), B, _ptr(out), _ptr(ws), ws.numel(),
                                         _stream_ptr()), "ecnf_vf_forward")
        return out

    def apply_div(self, params, x, t, feat=None) -> Tuple[torch.Tensor, torch.Tensor]:
        packed = self.pack(params)
        self._bind(packed)
        x, feat, B = self._prep(x, feat)
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device).reshape(-1).contiguous()
        if t.numel() != B:
            raise L.EcnfError(f"t must have {B} entries, got {t.numel()}")
        out = torch.empty_like(x)
        div = torch.empty(B, dtype=torch.float32, device=self.device)
        nb = int(self.lib.ecnf_solve_workspace_bytes(self.handle, L.MODE_VF_DIV, B))
        ws = self._workspace("solve", nb)
        L.check(self.lib.ecnf_vf_forward_div(self.handle, _ptr(x), _ptr(t), _ptr(feat), B, _ptr(out), _ptr(div),
                                             _ptr(ws), ws.numel(), _stream_ptr()), "ecnf_vf_forward_div")
        return out, div

    def apply_hutchinson(self, params, x, t, eps, feat=None) -> Tuple[torch.Tensor, torch.Tensor]:
        """(f, eps^T J eps): the reference's approx=True divergence (sample_and_log_prob.py:69-78) with the probe eps [B, D]."""
        packed = self.pack(params)
        self._bind(packed)
        x, feat, B = self._prep(x, feat)
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device).reshape(-1).contiguous()
        eps = torch.as_tensor(eps, dtype=torch.float32, device=self.device).reshape(-1, self.cfg.D).contiguous()
        if t.numel() != B or eps.shape[0] != B:
            raise L.EcnfError(f"t and eps must have {B} rows, got {t.numel()} and {eps.shape[0]}")
        out = torch.empty_like(x)
        div = torch.empty(B, dtype=torch.float32, device=self.device)
        nb = int(self.lib.ecnf_solve_workspace_bytes(self.handle, L.MODE_VF_DIV, B))
        ws = self._workspace("solve", nb)
        L.check(self.lib.ecnf_vf_forward_hutchinson(self.handle, _ptr(x), _ptr(t), _ptr(feat), _ptr(eps), B, _ptr(out),
                                                    _ptr(div), _ptr(ws), ws.numel(), _stream_ptr()),
                "ecnf_vf_forward_hutchinson")
        return out, div

    def normal_noise(self, key, n: int, global_offset: int = 0, substream: int = 1) -> torch.Tensor:
        """N(0,1) [n, D] keyed by (key, global sample index, substream); substream 0 = the noise under base_sample(key)."""
        out = torch.empty(n, self.cfg.D, dtype=torch.float32, device=self.device)
        L.check(self.lib.ecnf_normal_noise(self.handle, C.c_uint64(key_to_seed(key)), global_offset, n, substream, _ptr(out),
                                           _stream_ptr()), "ecnf_normal_noise")
        return out

    # ---------------------------------------------------------------- ODE solves
    def solve(self, params, mode: int, x_init, feat=None, ctrl: Optional[L.SolveCtrl] = None, eps=None, ts=None):
        """Returns (x_out [B, D], logs [B, 3] or None, stats int32 [B, 4]).  eps [B, D]: Hutchinson probes (approx=True).

        ts: save times (diffrax SaveAt(ts)), a 1-D sequence of floats in [0, 1], strictly increasing for the sample modes
        and strictly decreasing for MODE_LOGPROB.  Then the result is (x_out, logs, stats, traj [B, n_save, D],
        traj_delta [B, n_save] or None): the state and (log modes) the divergence integral at each time."""
        packed = self.pack(params)
        self._bind(packed)
        x_init, feat, B = self._prep(x_init, feat)
        ctrl = ctrl or L.make_ctrl()
        out_x = torch.empty_like(x_init)
        logs = None if mode == L.MODE_SAMPLE else torch.empty(B, 3, dtype=torch.float32, device=self.device)
        stats = torch.empty(B, 4, dtype=torch.int32, device=self.device)
        if eps is not None:
            eps = torch.as_tensor(eps, dtype=torch.float32, device=self.device).reshape(-1, self.cfg.D).contiguous()
            if eps.shape[0] != B or mode == L.MODE_SAMPLE:
                raise L.EcnfError("Hutchinson probes need one row per trajectory and a log-density mode")
        if ts is None:
            nb = int(self.lib.ecnf_solve_workspace_bytes(self.handle, mode, B))
            ws = self._workspace("solve", nb)
            L.check(self.lib.ecnf_solve_hutchinson(self.handle, mode, _ptr(x_init), _ptr(feat), _ptr(eps), B,
                                                   C.byref(ctrl), _ptr(out_x), _ptr(logs), _ptr(stats), _ptr(ws),
                                                   ws.numel(), _stream_ptr()), "ecnf_solve_hutchinson")
            return out_x, logs, stats
        ts_host = np.ascontiguousarray(
            (ts.detach().cpu().numpy() if isinstance(ts, torch.Tensor) else np.asarray(ts)).astype(np.float32).reshape(-1))
        n_save = int(ts_host.size)
        traj = torch.empty(B, n_save, self.cfg.D, dtype=torch.float32, device=self.device)
        traj_delta = None if mode == L.MODE_SAMPLE else torch.empty(B, n_save, dtype=torch.float32, device=self.device)
        nb = int(self.lib.ecnf_solve_saveat_workspace_bytes(self.handle, mode, B, n_save))
        ws = self._workspace("solve", nb)
        L.check(self.lib.ecnf_solve_saveat(self.handle, mode, _ptr(x_init), _ptr(feat), _ptr(eps), B, C.byref(ctrl),
                                           n_save, ts_host.ctypes.data_as(C.POINTER(C.c_float)), _ptr(out_x), _ptr(logs),
                                           _ptr(stats), _ptr(traj), _ptr(traj_delta), _ptr(ws), ws.numel(),
                                           _stream_ptr()), "ecnf_solve_saveat")
        return out_x, logs, stats, traj, traj_delta

    # ---------------------------------------------------------------- base distribution
    def base_sample(self, key, n: int, global_offset: int = 0) -> torch.Tensor:
        out = torch.empty(n, self.cfg.D, dtype=torch.float32, device=self.device)
        L.check(self.lib.ecnf_base_sample(self.handle, C.c_uint64(key_to_seed(key)), global_offset, n, _ptr(out),
                                          _stream_ptr()), "ecnf_base_sample")
        return out

    def base_sample_from_noise(self, eps) -> torch.Tensor:
        eps = torch.as_tensor(eps, dtype=torch.float32, device=self.device).reshape(-1, self.cfg.D).contiguous()
        out = torch.empty_like(eps)
        L.check(self.lib.ecnf_base_sample_from_noise(self.handle, _ptr(eps), eps.shape[0], _ptr(out), _stream_ptr()),
                "ecnf_base_sample_from_noise")
        return out

    def base_log_prob(self, x) -> torch.Tensor:
        x = torch.as_tensor(x, dtype=torch.float32, device=self.device)
        lead = x.shape[:-1]
        x2 = x.reshape(-1, self.cfg.D).contiguous()
        out = torch.empty(x2.shape[0], dtype=torch.float32, device=self.device)
        L.check(self.lib.ecnf_base_log_prob(self.handle, _ptr(x2), x2.shape[0], _ptr(out), _stream_ptr()),
                "ecnf_base_log_prob")
        return out.reshape(lead)

    # ---------------------------------------------------------------- flow matching
    def fm_draw_noise(self, key, B: int, global_offset: int = 0):
        x0 = torch.empty(B, self.cfg.D, dtype=torch.float32, device=self.device)
        t = torch.empty(B, dtype=torch.float32, device=self.device)
        L.check(self.lib.ecnf_fm_draw_noise(self.handle, C.c_uint64(key_to_seed(key)), global_offset, B, _ptr(x0),
                                            _ptr(t), _stream_ptr()), "ecnf_fm_draw_noise")
        return x0, t

    def fm_loss_grad(self, params, x_data, x0, t, feat=None, loss_denominator: Optional[float] = None,
                     out_grad: Optional[torch.Tensor] = None):
        """(loss [1], grad [param_count]) for the rows given; denominator defaults to B*D (a full batch)."""
        packed = self.pack(params)
        self._bind(packed)
        x_data, feat, B = self._prep(x_data, feat)
        x0 = torch.as_tensor(x0, dtype=torch.float32, device=self.device).reshape(B, self.cfg.D).contiguous()
        t = torch.as_tensor(t, dtype=torch.float32, device=self.device).reshape(B).contiguous()
        loss = torch.zeros(1, dtype=torch.float32, device=self.device)
        grad = out_grad if out_grad is not None else torch.empty(self.param_count, dtype=torch.float32,
                                                                  device=self.device)
        nb = int(self.lib.ecnf_fm_workspace_bytes(self.handle, B))
        ws = self._workspace("fm", nb)
        denom = float(loss_denominator) if loss_denominator is not None else float(B * self.cfg.D)
        L.check(self.lib.ecnf_fm_loss_grad(self.handle, _ptr(x_data), _ptr(x0), _ptr(t), _ptr(feat), B, denom,
                                           _ptr(loss), _ptr(grad), _ptr(ws), ws.numel(), _stream_ptr()),
                "ecnf_fm_loss_grad")
        return loss, grad

    def adam_step(self, flat: torch.Tensor, grad: torch.Tensor, mu: torch.Tensor, nu: torch.Tensor, step: int,
                  lr: float, ema: Optional[torch.Tensor] = None, b1=0.9, b2=0.999, eps=1e-8, ema_beta=0.999):
        norms = torch.empty(2, dtype=torch.float32, device=self.device)
        L.check(self.lib.ecnf_adam_step(_ptr(flat), _ptr(grad), _ptr(mu), _ptr(nu), _ptr(ema), flat.numel(), step,
                                        lr, b1, b2, eps, ema_beta, _ptr(norms), _stream_ptr()), "ecnf_adam_step")
        return norms

    # ---------------------------------------------------------------- weights / targets
    def ess_stats(self, log_w: torch.Tensor) -> torch.Tensor:
        log_w = torch.as_tensor(log_w, dtype=torch.float32, device=self.device).reshape(-1).contiguous()
        out = torch.empty(5, dtype=torch.float32, device=self.device)
        L.check(self.lib.ecnf_ess_stats(_ptr(log_w), log_w.numel(), _ptr(out), _stream_ptr()), "ecnf_ess_stats")
        return out

    def target_log_prob(self, kind: int, x) -> torch.Tensor:
        x = torch.as_tensor(x, dtype=torch.float32, device=self.device).reshape(-1, self.cfg.D).contiguous()
        out = torch.empty(x.shape[0], dtype=torch.float32, device=self.device)
        L.check(self.lib.ecnf_target_log_prob(kind, _ptr(x), x.shape[0], self.cfg.n_frames, self.cfg.dim, _ptr(out),
                                              _stream_ptr()), "ecnf_target_log_prob")
        return out


def ess_from_stats(stats: Sequence[float], n: int) -> Tuple[float, float]:
    """(reverse ESS, forward ESS) from the 5 sufficient statistics (setup_training.py:182,
    utils/evaluation.py:10-22)."""
    mx, s1, s2, nmx, s3 = [float(v) for v in stats]
    rv = (s1 * s1) / s2 / n
    log_z = mx + math.log(s1) - math.log(n)
    log_z_inv = nmx + math.log(s3) - math.log(n)
    return rv, math.exp(-log_z_inv - log_z)
