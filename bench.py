#!/usr/bin/env python
"""Benchmark of the ecnf hot path on B200 (contract in the task statement; metric from BASELINE.json).

Headline workload (BASELINE.json configs[1], `--workload lj13`, the default): LJ13 (13 particles, 3-D) EGNN CNF,
`sample_and_log_prob_cnf` with the exact divergence, Dopri5, batch 10 000 per GPU, followed by the LJ target log-density,
log-weights and the ESS sufficient statistics (setup_training.py:166-185).  One "step" = one such batch.  The solver runs
the reference's fixed-step branch (use_fixed_step_size=True, dt=0.05 -> exactly 121 vector-field evaluations per
trajectory) so the work per sample is deterministic and the roofline numerator is exact; parameters are synthetic
('stiffened' init, SURVEY 8(d)) because no trained checkpoint exists offline.

Other workloads (each prints one contract line; the default run reports small versions of them under "extra"):
  --workload aldp    BASELINE configs[3]: ALDP (22 atoms; aldp.yaml net), sample + exact log q + log-weights + ESS,
                     100 000 trajectories over the N GPUs with --scaling strong (12 500 per GPU with weak).  The reference
                     has no ALDP energy (examples/aldp.py:42-49 passes no target_log_prob_fn): log p is the LJ-style
                     energy of leonard_jones.py:10-27 on the 22 atoms -- a stand-in, stated here and in DESIGN.md.
  --workload dw4     BASELINE configs[0]: DW4, batch 1024, sample + exact log q.
  --workload sweep   BASELINE configs[4]: LJ13 `sample_cnf` (no divergence; load_checkpoint_measure_sampling_time.py:
                     101-119), global batch 1k / 10k / 100k / 1M split over the N GPUs.
  --workload fm      BASELINE configs[2]: QM9-positional flow-matching training step, batch 512 per GPU.
--scaling strong splits a fixed global batch over the ranks (default: weak, per-GPU batch fixed).
--steps sets the number of timed steps of the reported workload (every batch of the sweep).  --dump-outputs DIR writes what
the last timed step returned as DIR/<name>.npy (float32/float64, at most 64 MB, rows sampled with a fixed seed above that):
the solve workloads write `samples`, `logs` (log q, log p0(x0), delta), `solver_stats` and `ess_stats`; fm writes the
updated parameters, EMA, Adam moments, loss and norms.  Inputs and parameters are seeded, so two builds run with the same
arguments can be compared output for output.

`--impl reference` times the CPU restatement of the reference (oracle/, torch fp32, reverse-mode Jacobian exactly like
sample_and_log_prob.py:64-66) on the host cores: JAX is not installable in this image, so the reference itself cannot
run (DESIGN.md, "reference arm").  That arm never touches the CUDA library.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LJ13 = dict(n_frames=13, dim=3, sigma_min=0.01, base_scale=1.0, n_blocks_egnn=3, mlp_units=(128, 128, 128),
            n_invariant_feat_hidden=64, time_embedding_dim=8, n_features=1)
DW4 = dict(n_frames=4, dim=2, sigma_min=0.01, base_scale=1.0, n_blocks_egnn=3, mlp_units=(128, 128, 128),
           n_invariant_feat_hidden=64, time_embedding_dim=8, n_features=1)
QM9 = dict(n_frames=19, dim=3, sigma_min=1e-6, base_scale=2.0, n_blocks_egnn=5, mlp_units=(256, 256, 256, 256),
           n_invariant_feat_hidden=32, time_embedding_dim=8, n_features=1)
ALDP = dict(n_frames=22, dim=3, sigma_min=1e-6, base_scale=0.2, n_blocks_egnn=3, mlp_units=(64, 64),
            n_invariant_feat_hidden=32, time_embedding_dim=8, n_features=22)
CFGS = {"lj13": LJ13, "dw4": DW4, "qm9": QM9, "aldp": ALDP}
N_EVALS_FIXED = 121          # 1 FSAL init + 6 stages x 20 steps (dt = 0.05)
METRIC = "LJ13 samples/s with exact log-q (Dopri5)"
UNIT = "samples/s"


def fwd_flops(c) -> float:
    """SURVEY Appendix E: 2 * blocks * (E * M_e + n * M_n), dense matmuls exactly as the reference's op graph."""
    n, H, T, U, L = c["n_frames"], c["n_invariant_feat_hidden"], c["time_embedding_dim"], c["mlp_units"][0], len(c["mlp_units"])
    E = n * (n - 1)
    m_e = (2 * H + 1) * U + (L - 1) * U * U + L * U * U + 2 * U
    m_n = (H + T) * H + (U + H) * U + (L - 1) * U * U + U * H
    return 2.0 * c["n_blocks_egnn"] * (E * m_e + n * m_n)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def ncu_traffic(kernel_key: str):
    """dram bytes per trajectory of the dominant kernel from the committed ncu capture (profiles/r2_traffic.json): a
    SEPARATE capture of the same kernel, not measured in this run -- the line says so."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(p):
        d = json.load(open(p)).get(kernel_key)
        if d:
            return d["dram_bytes_per_trajectory"], d["source"]
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm_sorted = sorted(sm)       # the busiest half of the samples = "under load"
        return {"sm_mhz": statistics.median(sm_sorted[len(sm_sorted) // 2:]) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py touches oracle/; they never load libecnf_b200.so)
# ----------------------------------------------------------------------------------------------------------
def host_params(name: str, seed: int = 0, head_variance: float = 1.0) -> dict:
    """The GPU arm's synthetic parameters as {flax path: array}, built from the oracle's layout: no Engine, no .so."""
    from oracle import ecnf_oracle as O
    from ecnf_b200.nets.egnn import init_param_tensors
    return init_param_tensors(O.param_layout(O.CnfConfig(**CFGS[name])), seed, head_variance)


def cpu_sample_logq(name: str, params: dict, n_traj: int, threads: int, seed: int = 2, div: bool = True):
    """Time `n_traj` trajectories of sample_and_log_prob (exact, fixed dt=0.05) -- or sample_cnf -- on the host cores."""
    from oracle import ecnf_oracle as O
    torch.set_num_threads(threads)
    torch.set_flush_denormal(True)
    ocfg = O.CnfConfig(**CFGS[name])
    p = O.to_torch(params, torch.float32)
    rng = np.random.default_rng(seed)
    x0 = O.base_sample_from_noise(ocfg, torch.tensor(rng.standard_normal((n_traj, ocfg.D)), dtype=torch.float32))
    feat = torch.arange(ocfg.n_frames).remainder(ocfg.n_features).repeat(n_traj, 1)
    t0 = time.perf_counter()
    if div:
        x1, logq, st = O.sample_and_log_prob_cnf(p, ocfg, x0, feat, O.SolveControl(fixed=True, step_size=0.05))
        if name != "dw4":
            lw = -O.lj_energy(x1.numpy().reshape(n_traj, ocfg.n_frames, ocfg.dim).astype(np.float64)) - logq.numpy()
        else:
            lw = -O.dw_energy(x1.numpy().reshape(n_traj, ocfg.n_frames, ocfg.dim).astype(np.float64)) - logq.numpy()
        O.reverse_ess(lw)
    else:
        x1, st = O.sample_cnf(p, ocfg, x0, feat, O.SolveControl(fixed=True, step_size=0.05))
    dt = time.perf_counter() - t0
    assert int(st.n_evals[0]) == N_EVALS_FIXED
    return n_traj / dt, dt


def cpu_fm_steps(B: int, steps: int, threads: int):
    """QM9-positional FM step on the host cores: oracle loss + autograd gradient + restated Adam/EMA
    (gradient_step.py:20-53), `steps` steps at batch B."""
    from oracle import ecnf_oracle as O
    torch.set_num_threads(threads)
    ocfg = O.CnfConfig(**QM9)
    flat = host_params("qm9", 0, 0.001)
    rng = np.random.default_rng(3)
    x = rng.standard_normal((B, 19, 3)).astype(np.float32) * 1.5
    x = torch.tensor((x - x.mean(axis=1, keepdims=True)).reshape(B, 57))
    feat = torch.zeros(B, 19, dtype=torch.long)
    m = {k: np.zeros_like(v) for k, v in flat.items()}
    v2 = {k: np.zeros_like(v) for k, v in flat.items()}
    ema = {k: v.copy() for k, v in flat.items()}
    t0 = time.perf_counter()
    for s in range(steps):
        x0 = O.base_sample_from_noise(ocfg, torch.tensor(rng.standard_normal((B, 57)), dtype=torch.float32))
        t = torch.tensor(rng.uniform(0, 1, B), dtype=torch.float32)
        loss, g = O.fm_loss_and_grad(flat, ocfg, x, x0, t, feat, dtype=torch.float32)
        for k in flat:
            p_, m_, v_, _ = O.adam_step(flat[k], g[k].numpy(), m[k], v2[k], s, 1e-4)
            flat[k], m[k], v2[k] = p_.astype(np.float32), m_.astype(np.float32), v_.astype(np.float32)
            ema[k] = 0.999 * ema[k] + 0.001 * flat[k]
    dt = time.perf_counter() - t0
    return steps / dt, dt, float(loss)


CPU_TRAJ = 4     # trajectories per CPU step: the SAME bounded sample in the reference arm and in cpu_baseline


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    params = host_params("lj13")
    times = []
    for _ in range(max(0, min(args.warmup, 1))):          # torch-CPU has no compile step: one warm-up pass is enough
        cpu_sample_logq("lj13", params, CPU_TRAJ, threads)
    for _ in range(args.steps):
        _, dt = cpu_sample_logq("lj13", params, CPU_TRAJ, threads)
        times.append(dt)
    value = CPU_TRAJ * len(times) / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "lj13_sample_and_log_prob_exact_dopri5_fixed_dt0.05+lj_log_weights+ess", "batch_per_step": CPU_TRAJ,
                   "n_evals_per_sample": N_EVALS_FIXED, "params": "synthetic stiffened init (seed 0), same as the GPU arm"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{CPU_TRAJ} LJ13 trajectories per step (121 evals each), torch-CPU fp32 restatement "
                                   "of the reference with reverse-mode Jacobian; the JAX reference cannot be installed "
                                   "in this image"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
def count_kernels(fn):
    """(our kernels, other kernels) launched by fn(), counted from CUPTI activity records (torch.profiler sees every kernel
    of the process, including those of libecnf_b200.so).  None when the profiler is unavailable."""
    try:
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        ours = others = 0
        names = {}
        for ev in prof.events():
            if getattr(ev, "device_type", None) != torch.autograd.DeviceType.CUDA:
                continue
            nm = ev.name
            if nm.startswith("Memcpy") or nm.startswith("Memset"):
                continue
            if "at::" in nm or "cub::" in nm or "nccl" in nm.lower() or "cutlass" in nm or "cublas" in nm.lower():
                others += 1
            else:
                ours += 1
                key = nm.split("(")[0][-60:]
                names[key] = names.get(key, 0) + 1
        return ours, others, names
    except Exception as e:  # noqa: BLE001
        return None, None, {"error": repr(e)}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path: str, arrays: dict) -> None:
    """Writes `arrays` (what the timed path returned in its last step) as <path>/<name>.npy in float32 or float64, so that
    two builds can be compared output for output.  Integer outputs become float64 (exact).  When the whole exceeds 64 MB,
    every array keeps the same fixed, seeded sample of its rows."""
    host = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        host[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    total = sum(a.nbytes for a in host.values())
    os.makedirs(path, exist_ok=True)
    for name, a in host.items():
        if total > DUMP_MAX_BYTES and a.ndim > 0 and a.shape[0] > 1:
            keep = max(1, a.shape[0] * DUMP_MAX_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


class Ctx:
    pass


def setup(args):
    c = Ctx()
    c.rank = int(os.environ.get("RANK", "0"))
    c.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(c.local_rank)
    c.dev = torch.device("cuda", c.local_rank)
    import torch.distributed as dist
    c.dist = dist
    if c.world > 1:
        dist.init_process_group("nccl", device_id=c.dev)
    c.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=c.dev)   # > 126 MB L2
    return c


def barrier(c):
    if c.world > 1:
        c.dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(c, ms: float) -> float:
    t = torch.tensor([ms], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    return t.item()


def sum_over_ranks(c, v: float) -> float:
    t = torch.tensor([v], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.SUM)
    return t.item()


def make_model(c, name: str, head_variance: float = 1.0):
    from ecnf_b200.cnf import build_cnf
    from ecnf_b200.engine import PackedParams
    from ecnf_b200.nets.egnn import init_flat_params
    cnf = build_cnf(**CFGS[name])
    eng = cnf.engine
    params = PackedParams(torch.from_numpy(init_flat_params(eng, 0, head_variance=head_variance)).to(c.dev))
    return cnf, eng, params


def shard(c, global_batch: int):
    from ecnf_b200.distributed import shard_range
    return shard_range(global_batch, c.rank, c.world)


def bench_solve(c, name: str, b_begin: int, b_end: int, *, div: bool, adaptive: bool, steps: int, warmup: int,
                target: int | None, e2e_steps: int = 0, sample_clocks: bool = False, count: bool = True, e2e_warm: bool = True):
    """Times `steps` passes of sample(+exact log q)(+target log-density, log-weights, ESS statistics) over the global
    sample indices [b_begin, b_end) of this rank.  Returns a dict with device-timed throughput (max over ranks), the
    solve kernel's own time, evaluation counts, the end-to-end (host buffers) figure and the launch count."""
    from ecnf_b200 import lib as L
    from ecnf_b200.cnf import sample_and_log_prob_cnf, sample_cnf
    from ecnf_b200.distributed import merge_ess_stats
    from ecnf_b200.engine import ess_from_stats
    cfg = CFGS[name]
    cnf, eng, params = make_model(c, name)
    n, D = cfg["n_frames"], cfg["n_frames"] * cfg["dim"]
    B = b_end - b_begin
    feat = (torch.arange(n, dtype=torch.int32, device=c.dev) % cfg["n_features"]).repeat(B, 1).contiguous()
    ctrl = L.make_ctrl(use_fixed_step_size=not adaptive)
    mode = L.MODE_SAMPLE_LOGQ if div else L.MODE_SAMPLE
    kernel_events = []

    def step_resident(x0, timed=False):
        if timed:
            ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ka.record()
        x1, logs, stats = eng.solve(params, mode, x0, feat, ctrl)
        if timed:
            kb.record()
            kernel_events.append((ka, kb))
        st = None
        if div and target is not None:
            log_w = eng.target_log_prob(target, x1) - logs[:, 0]
            st = eng.ess_stats(log_w)
            if c.world > 1:
                st = merge_ess_stats(st)
        return x1, logs, stats, st

    x0_res = eng.base_sample(2, B, b_begin)               # noise keyed by GLOBAL sample index
    for _ in range(warmup):
        step_resident(x0_res)
    barrier(c)
    sampler = None
    if sample_clocks:
        sampler = ClockSampler(c.local_rank)
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    evals_last = 0
    bad = 0
    for i in range(steps):
        c.flush.zero_()
        barrier(c)
        ev[i][0].record()
        x1, logs, stats, st = step_resident(x0_res, timed=True)
        ev[i][1].record()
        barrier(c)
        evals_last = int(stats[:, 2].sum().item())
        bad += int((stats[:, 3] != 0).sum().item())
    t_steps = [a.elapsed_time(b) for a, b in ev]
    total_ms = max_over_ranks(c, sum(t_steps))
    clocks = sampler.stop() if sampler else None
    global_B = int(sum_over_ranks(c, B))
    k_ms = sum(a.elapsed_time(b) for a, b in kernel_events) / len(kernel_events)
    out = {"value": global_B * steps / (total_ms * 1e-3), "ms_per_step": total_ms / steps, "kernel_ms": k_ms,
           "evals_per_launch": evals_last, "batch_this_rank": B, "global_batch": global_B, "step_ms": t_steps,
           "clocks": clocks, "status_failures": bad, "eng": eng, "D": D,
           "outputs": {k: v for k, v in (("samples", x1), ("logs", logs), ("solver_stats", stats), ("ess_stats", st))
                       if v is not None}}
    if st is not None:
        rv, fw = ess_from_stats(st.tolist(), global_B)
        out["reverse_ess"], out["forward_ess"] = rv, fw

    launches_per_step = None
    if count:
        ours, others, names = count_kernels(lambda: step_resident(x0_res))
        out["kernels_per_step"] = {"ours": ours, "torch_or_library": others, "by_name": names}
        launches_per_step = ours
    out["launches_per_step"] = launches_per_step if launches_per_step is not None else 1

    if e2e_steps > 0:
        # end to end through the public API with HOST buffers: H2D of noise + features, D2H of samples, log q, ESS stats
        rng = np.random.default_rng(1000 + c.rank)
        eps_host = torch.from_numpy(rng.standard_normal((B, D)).astype(np.float32)).pin_memory()
        feat_host = feat.cpu().pin_memory()
        out_x = torch.empty(B, D, dtype=torch.float32).pin_memory()
        out_lq = torch.empty(B, dtype=torch.float32).pin_memory()
        out_ess = torch.empty(5, dtype=torch.float32).pin_memory()

        def step_e2e():
            eps = eps_host.to(c.dev, non_blocking=True)
            f = feat_host.to(c.dev, non_blocking=True)
            x0 = eng.base_sample_from_noise(eps)
            if div:
                x1, log_q = sample_and_log_prob_cnf(cnf, params, None, f, use_fixed_step_size=not adaptive, x0=x0,
                                                    check_status=False)
                out_lq.copy_(log_q, non_blocking=True)
                if target is not None:
                    st_ = eng.ess_stats(eng.target_log_prob(target, x1) - log_q)
                    if c.world > 1:
                        st_ = merge_ess_stats(st_)
                    out_ess.copy_(st_, non_blocking=True)
            else:
                x1 = sample_cnf(cnf, params, None, f, use_fixed_step_size=not adaptive, x0=x0, check_status=False)
            out_x.copy_(x1, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        if warmup == 0 and e2e_warm:
            step_e2e()                # one untimed pass through the host-buffer path (skipped for the long sharded ALDP pass: the
                                      # kernels are warm after the resident steps and the pinned buffers are touched above)
        barrier(c)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(e2e_steps):
            step_e2e()
        b.record()
        barrier(c)
        e2e_ms = max_over_ranks(c, a.elapsed_time(b))
        out["e2e"] = {"value": global_B * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "steps": e2e_steps,
                      "h2d_bytes_per_step": B * D * 4 + B * n * 4,
                      "d2h_bytes_per_step": B * D * 4 + (B * 4 if div else 0) + (20 if div and target is not None else 0)}
    return out


def roofline_of(c, name: str, r: dict, div: bool):
    cfg = CFGS[name]
    D = cfg["n_frames"] * cfg["dim"]
    f_eval = ((1 + D) if div else 1) * fwd_flops(cfg)                # SURVEY 8(d): (1 + D) * F_fwd per exact-div evaluation
    alg = r["evals_per_launch"] * f_eval
    pk, pk_kind = peaks()
    peak_tf = pk.get("bf16_tflops_sustained", pk["bf16_tflops"]) if r["kernel_ms"] > 1000 else pk["bf16_tflops"]
    tf = alg / (r["kernel_ms"] * 1e-3) / 1e12
    eng = r["eng"]
    tc_flops = int(eng.lib.ecnf_solve_tensor_flops_per_eval(eng.handle)) if div else 0
    per_traj, src = ncu_traffic(("solve_tc_" if tc_flops else "solve_simt_") + name)
    return {"bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf,
            "traffic": per_traj * r["batch_this_rank"] if per_traj else None,
            "kernel": ("ecnf_solve_tc_kernel (tcgen05 + TMEM, 3-pass bf16 split, fp32 accumulate)" if tc_flops or not div
                       else "ecnf_solve_kernel (fp32 SIMT)"),
            "kernel_ms": r["kernel_ms"], "algorithmic_flops_per_launch": alg,
            "executed_tensor_flops_per_launch": r["evals_per_launch"] * tc_flops if tc_flops else None,
            "peak_source": f"{pk_kind} bf16 dense {'sustained' if r['kernel_ms'] > 1000 else 'burst'} (MEASURED_PEAKS.json); "
                           "numerator = algorithmic (1+D)*F_fwd per evaluation (SURVEY 8(d)); the kernel executes 3 bf16 "
                           "passes over a structurally reduced tangent set, see executed_tensor_flops_per_launch",
            "traffic_source": (src + " -- a separate ncu capture of this kernel, NOT measured in this run") if src else None}


def bench_train(c, *, steps: int = 10, cpu: bool = False, chunk: int = 0, count: bool = True):
    """QM9-positional FM training step (loss + grad + all-reduce + Adam/EMA), batch 512 per GPU; every step copies its
    batch from pinned host memory and reads the loss back (the e2e figure IS the figure)."""
    from ecnf_b200.cnf import flow_matching_update_fn, TrainingState
    from ecnf_b200.distributed import make_grad_allreduce
    from ecnf_b200.utils.optim import Adam, warmup_cosine_decay_schedule
    cnf, eng, params = make_model(c, "qm9", head_variance=0.001)
    eng.set_fm_chunk(chunk)                               # graphs per chunk of the minibatch (0 = the library's choice)
    B = 512
    opt = Adam(warmup_cosine_decay_schedule(1e-4, 1e-4, 10, 100_000, 0.0))
    state = TrainingState(params=params, opt_state=opt.init(params), key=c.rank, ema_params=params)
    rng = np.random.default_rng(3 + c.rank)
    x = rng.standard_normal((B, 19, 3)).astype(np.float32) * 1.5
    x = (x - x.mean(axis=1, keepdims=True)).reshape(B, 57)
    x_host = torch.from_numpy(x).pin_memory()
    feat_host = torch.zeros(B, 19, dtype=torch.int32).pin_memory()
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()
    hook = make_grad_allreduce(c.world) if c.world > 1 else None
    denom = float(c.world * B * 57)

    def step(st, read_loss):
        xd = x_host.to(c.dev, non_blocking=True)
        fd = feat_host.to(c.dev, non_blocking=True)
        st, info = flow_matching_update_fn(cnf, opt.update, st, xd, fd, grad_allreduce=hook,
                                           global_offset=c.rank * B, loss_denominator=denom, donate=True)
        if read_loss:
            loss_host.copy_(info["loss"].reshape(1), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return st, info

    for _ in range(3):
        state, info = step(state, True)
    barrier(c)
    res = {}
    for label, read_loss in (("resident", False), ("e2e", True)):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            state, info = step(state, read_loss)
        b.record()
        barrier(c)
        res[label] = max_over_ranks(c, a.elapsed_time(b)) / steps
    loss = float(info["loss"])
    # copies: the launch-count step below updates the donated buffers in place
    outputs = {"params": state.params.flat, "ema_params": state.ema_params.flat, "adam_mu": state.opt_state.mu,
               "adam_nu": state.opt_state.nu, **info}
    outputs = {k: v.clone() for k, v in outputs.items()}
    holder = {"s": state}

    def one():
        holder["s"], _ = step(holder["s"], True)
    ours, others, names = count_kernels(one) if count else (None, None, {})
    flops = 3.0 * fwd_flops(QM9) * B                     # per GPU (weak scaling: every rank steps its own 512 graphs)
    pk, pk_kind = peaks()
    peak = pk["bf16_tflops"]                              # a 10-20 ms step: burst figure
    tf = flops / (res["resident"] * 1e-3) / 1e12
    out = {"metric": "QM9-positional FM train steps/s (batch 512 per GPU, loss+grad+Adam+EMA, H2D of the batch inside)",
           "value": 1e3 / res["resident"], "unit": "steps/s", "ms_per_step": res["resident"], "loss": loss,
           "global_batch": B * c.world, "graphs_per_s": B * c.world * 1e3 / res["resident"],
           "e2e": {"value": 1e3 / res["e2e"], "unit": "steps/s", "h2d_bytes_per_step": B * 57 * 4 + B * 19 * 4,
                   "d2h_bytes_per_step": 4, "note": "+ a device->host read of the loss every step"},
           "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                        "algorithmic_flops_per_step": flops, "per": "GPU", "peak_source": f"{pk_kind} bf16 dense burst"},
           "kernels_per_step": {"ours": ours, "torch_or_library": others}, "launches_per_step": ours or 1,
           "outputs": outputs}
    if cpu and c.rank == 0 and c.world == 1:
        threads = os.cpu_count() or 1
        v, dt, l_cpu = cpu_fm_steps(B, 3, threads)
        out["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": threads, "kind": "port",
                               "sample": f"3 steps at batch {B} in {dt:.1f} s: oracle loss + torch autograd gradient + restated "
                                         "Adam/EMA (gradient_step.py:20-53), torch-CPU fp32"}
    return out


def contract_line(c, args, *, metric, unit, r, workload, cfg_extra, roofline, cpu, extra, scaling, launches):
    return {
        "metric": metric, "value": r["value"], "unit": unit, "n_gpus": c.world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "params": "synthetic stiffened init (seed 0)",
                   "l2": "256 MiB flush buffer written between timed steps", **cfg_extra},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": r.get("e2e"), "gpu_launches": launches, "clocks": r.get("clocks"),
        "extra": extra,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 2; 10 for --workload fm)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="lj13", choices=["lj13", "aldp", "dw4", "sweep", "fm"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=None, help="trajectories per GPU (weak) or in total (strong) per step")
    ap.add_argument("--no-extra", "--no-train", dest="no_extra", action="store_true", help="skip the secondary measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the bounded CPU baselines")
    ap.add_argument("--adaptive", action="store_true", help="PID-controlled steps (rtol=atol=1e-5) instead of dt=0.05")
    ap.add_argument("--sweep-max", type=int, default=1_000_000)
    ap.add_argument("--fm-chunk", type=int, default=0, help="fm workload: graphs per chunk of the minibatch (0 = automatic)")
    ap.add_argument("--no-count", action="store_true", help="skip the profiler pass that counts kernel launches (one extra step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step as DIR/<name>.npy (rank 0's shard under torchrun)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 10 if args.workload == "fm" else 2
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        return run_reference(args)
    c = setup(args)
    from ecnf_b200 import lib as L
    strong = args.scaling == "strong"

    def rng_for(default_per_gpu, default_total):
        if strong:
            return shard(c, args.batch or default_total)
        b = args.batch or default_per_gpu
        return c.rank * b, (c.rank + 1) * b

    par = (f"dp{c.world} (independent trajectories, " + ("fixed global batch split over ranks" if strong else "fixed per-GPU batch")
           + "; ESS statistics all-gathered)")
    fixed_tag = "adaptive_rtol1e-5" if args.adaptive else "fixed_dt0.05"
    line = None

    if args.workload == "lj13":
        b0, b1 = rng_for(10_000, 10_000)
        r = bench_solve(c, "lj13", b0, b1, div=True, adaptive=args.adaptive, steps=args.steps, warmup=args.warmup,
                        target=L.TARGET_LJ, e2e_steps=max(1, min(args.steps, 5)), sample_clocks=True, count=not args.no_count)
        extra = {"reverse_ess": r.get("reverse_ess"), "forward_ess": r.get("forward_ess"), "step_ms": r["step_ms"],
                 "kernels_per_step": r.get("kernels_per_step"), "status_failures": r["status_failures"]}
        launches = r["launches_per_step"] * args.steps
        if not args.no_extra:
            ra = bench_solve(c, "lj13", c.rank * 2368, (c.rank + 1) * 2368, div=True, adaptive=True, steps=1, warmup=1,
                             target=L.TARGET_LJ, count=False)
            extra["lj13_adaptive"] = {"metric": "LJ13 samples/s with exact log-q (Dopri5 adaptive rtol=atol=1e-5, the reference's shipped setting)",
                                      "value": ra["value"], "unit": UNIT, "batch_per_gpu": 2368,
                                      "evals_per_sample": ra["evals_per_launch"] / 2368, "roofline": roofline_of(c, "lj13", ra, True),
                                      "status_failures": ra["status_failures"]}
            rd = bench_solve(c, "dw4", c.rank * 1024, (c.rank + 1) * 1024, div=True, adaptive=False, steps=2, warmup=1,
                             target=L.TARGET_DW, e2e_steps=2, count=False)
            extra["dw4"] = {"metric": "DW4 samples/s with exact log-q (batch 1024, dt=0.05) + DW log-weights + ESS",
                            "value": rd["value"], "unit": UNIT, "e2e": rd["e2e"], "roofline": roofline_of(c, "dw4", rd, True)}
            rl = bench_solve(c, "aldp", c.rank * 1184, (c.rank + 1) * 1184, div=True, adaptive=False, steps=1, warmup=1,
                             target=L.TARGET_LJ, e2e_steps=1, count=False)
            extra["aldp"] = {"metric": "ALDP samples/s with exact log-q (batch 1184 per GPU, dt=0.05) + stand-in LJ log-weights + ESS",
                             "value": rl["value"], "unit": UNIT, "e2e": rl["e2e"], "roofline": roofline_of(c, "aldp", rl, True)}
            rs = bench_solve(c, "lj13", c.rank * 4736, (c.rank + 1) * 4736, div=False, adaptive=args.adaptive, steps=1, warmup=1,
                             target=None, e2e_steps=1, count=False)
            extra["sample_only"] = {"metric": f"LJ13 sample_cnf samples/s (no divergence, Dopri5 {fixed_tag})", "value": rs["value"],
                                    "unit": UNIT, "batch_per_gpu": 4736, "e2e": rs["e2e"], "roofline": roofline_of(c, "lj13", rs, False)}
            extra["fm_train"] = bench_train(c, cpu=not args.no_cpu)
            if c.world > 1:
                # strong scaling: BASELINE configs[1]'s global batch of 10 000 split over the ranks
                b0, b1 = shard(c, 10_000)
                rt = bench_solve(c, "lj13", b0, b1, div=True, adaptive=False, steps=2, warmup=1, target=L.TARGET_LJ, count=False)
                extra["lj13_strong_10k"] = {"metric": METRIC + ", global batch 10 000 split over the ranks", "value": rt["value"],
                                            "unit": UNIT, "ms_per_step": rt["ms_per_step"], "scaling": "strong",
                                            "batch_this_rank": rt["batch_this_rank"], "roofline": roofline_of(c, "lj13", rt, True)}
                # BASELINE configs[3]: ALDP, 12 500 trajectories per GPU = 100 000 sharded over 8 GPUs, log-weights + merged ESS
                b0, b1 = shard(c, 12_500 * c.world)
                rA = bench_solve(c, "aldp", b0, b1, div=True, adaptive=False, steps=1, warmup=0, target=L.TARGET_LJ,
                                 e2e_steps=1, count=False, e2e_warm=False)     # (warm after the small ALDP run above)
                extra["aldp_sharded"] = {"metric": "ALDP samples/s with exact log-q, 12 500 trajectories per GPU (100 000 over 8 GPUs = BASELINE "
                                                   "configs[3]) + stand-in LJ log-weights + merged ESS",
                                         "value": rA["value"], "unit": UNIT, "ms_per_step": rA["ms_per_step"],
                                         "global_batch": rA["global_batch"], "batch_this_rank": rA["batch_this_rank"],
                                         "is_baseline_config_3_size": rA["global_batch"] == 100_000,
                                         "e2e": rA["e2e"], "reverse_ess": rA.get("reverse_ess"), "forward_ess": rA.get("forward_ess"),
                                         "status_failures": rA["status_failures"], "roofline": roofline_of(c, "aldp", rA, True)}
        cpu = None
        if c.rank == 0 and c.world == 1 and not args.no_cpu:
            threads = os.cpu_count() or 1
            v, dt = cpu_sample_logq("lj13", host_params("lj13"), CPU_TRAJ, threads)
            cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"{CPU_TRAJ} LJ13 trajectories x 121 evals (fixed dt=0.05) in {dt:.1f} s, torch-CPU fp32 restatement of "
                             "the reference (reverse-mode Jacobian); JAX reference not installable here"}
            if not args.no_extra:
                v2, dt2 = cpu_sample_logq("aldp", host_params("aldp"), 2, threads)
                extra["aldp"]["cpu_baseline"] = {"value": v2, "unit": UNIT, "cores": threads, "kind": "port",
                                                 "sample": f"2 ALDP trajectories x 121 evals in {dt2:.1f} s"}
                v3, dt3 = cpu_sample_logq("dw4", host_params("dw4"), 16, threads)
                extra["dw4"]["cpu_baseline"] = {"value": v3, "unit": UNIT, "cores": threads, "kind": "port",
                                                "sample": f"16 DW4 trajectories x 121 evals in {dt3:.1f} s"}
                v4, dt4 = cpu_sample_logq("lj13", host_params("lj13"), 64, threads, div=False)
                extra["sample_only"]["cpu_baseline"] = {"value": v4, "unit": UNIT, "cores": threads, "kind": "port",
                                                        "sample": f"64 LJ13 sample_cnf trajectories x 121 evals in {dt4:.1f} s"}
        line = contract_line(c, args, metric=METRIC, unit=UNIT, r=r,
                             workload=f"lj13_sample_and_log_prob_exact_dopri5_{fixed_tag}+lj_log_weights+ess",
                             cfg_extra={"batch_per_gpu": r["batch_this_rank"], "global_batch": r["global_batch"],
                                        "n_evals_per_sample": r["evals_per_launch"] / r["batch_this_rank"], "parallelism": par},
                             roofline=roofline_of(c, "lj13", r, True), cpu=cpu, extra=extra,
                             scaling=args.scaling, launches=launches)

    elif args.workload in ("aldp", "dw4"):
        name = args.workload
        b0, b1 = rng_for(12_500 if name == "aldp" else 1024, 100_000 if name == "aldp" else 1024)
        target = L.TARGET_LJ if name == "aldp" else L.TARGET_DW
        r = bench_solve(c, name, b0, b1, div=True, adaptive=args.adaptive, steps=args.steps, warmup=args.warmup, target=target,
                        e2e_steps=1, sample_clocks=True, count=not args.no_count, e2e_warm=(name != "aldp"))
        cpu = None
        if c.rank == 0 and not args.no_cpu:
            threads = os.cpu_count() or 1
            nt = 4 if name == "aldp" else 16
            v, dt = cpu_sample_logq(name, host_params(name), nt, threads)
            cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"{nt} {name.upper()} trajectories x 121 evals (fixed dt=0.05) in {dt:.1f} s, torch-CPU fp32 restatement"}
        metric = (f"{name.upper()} samples/s with exact log-q (Dopri5) + log-weights + ESS"
                  + (" [log p = LJ-style stand-in on 22 atoms: the reference has no ALDP energy]" if name == "aldp" else ""))
        line = contract_line(c, args, metric=metric, unit=UNIT, r=r,
                             workload=f"{name}_sample_and_log_prob_exact_dopri5_{fixed_tag}+log_weights+ess",
                             cfg_extra={"batch_this_rank": r["batch_this_rank"], "global_batch": r["global_batch"],
                                        "n_evals_per_sample": r["evals_per_launch"] / r["batch_this_rank"], "parallelism": par},
                             roofline=roofline_of(c, name, r, True), cpu=cpu,
                             extra={"reverse_ess": r.get("reverse_ess"), "forward_ess": r.get("forward_ess"), "step_ms": r["step_ms"],
                                    "kernels_per_step": r.get("kernels_per_step"), "status_failures": r["status_failures"]},
                             scaling=args.scaling, launches=r["launches_per_step"] * args.steps)

    elif args.workload == "sweep":
        table, per_step, total_launches, last_e2e = [], 1, 0, None
        for gb in (1_000, 10_000, 100_000, 1_000_000):
            if gb > args.sweep_max:
                continue
            b0, b1 = shard(c, gb)
            # (the kernel and its workspace are warm after the smaller batches: the long ones are timed without a warm-up pass)
            r = bench_solve(c, "lj13", b0, b1, div=False, adaptive=args.adaptive, steps=args.steps,
                            warmup=1 if gb <= 10_000 else 0, target=None, e2e_steps=1 if gb <= 10_000 else 0,
                            count=(gb == 1_000 and not args.no_count))
            if gb == 1_000:
                per_step = r["launches_per_step"]
            total_launches += per_step * args.steps
            table.append({"global_batch": gb, "samples_per_s": r["value"], "ms": r["ms_per_step"],
                          "e2e_samples_per_s": r["e2e"]["value"] if "e2e" in r else None,
                          "roofline_frac": roofline_of(c, "lj13", r, False)["frac"]})
            if "e2e" in r:
                last_e2e = r["e2e"]
            last = r
        last["e2e"] = dict(last_e2e, note="end-to-end (host buffers) is measured at the batches <= 10k of the sweep; this is the largest of them")
        cpu = None
        if c.rank == 0 and not args.no_cpu:
            threads = os.cpu_count() or 1
            v, dt = cpu_sample_logq("lj13", host_params("lj13"), 128, threads, div=False)
            cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"128 LJ13 sample_cnf trajectories x 121 evals in {dt:.1f} s (the B = 1k point extrapolates linearly)"}
        line = contract_line(c, args, metric=f"LJ13 sample_cnf samples/s (no divergence, Dopri5 {fixed_tag}), largest batch of the sweep",
                             unit=UNIT, r=last, workload="lj13_sample_cnf_sweep (load_checkpoint_measure_sampling_time.py:101-119)",
                             cfg_extra={"global_batch": last["global_batch"],
                                        "parallelism": f"dp{c.world} (independent trajectories, every global batch of the sweep split over the ranks)"},
                             roofline=roofline_of(c, "lj13", last, False), cpu=cpu, extra={"sweep": table}, scaling="strong",
                             launches=total_launches)

    elif args.workload == "fm":
        ft = bench_train(c, steps=args.steps, cpu=not args.no_cpu, chunk=args.fm_chunk, count=not args.no_count)
        line = {"metric": ft["metric"], "value": ft["value"], "unit": "steps/s", "n_gpus": c.world,
                "steps": args.steps, "warmup": 3, "ms_per_step": ft["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "qm9pos_flow_matching_update_fn_batch512_per_gpu", "global_batch": ft["global_batch"],
                           "parallelism": f"dp{c.world} (minibatch shards, one NCCL all-reduce of the flat gradient)"},
                "roofline": ft["roofline"], "cpu_baseline": ft.get("cpu_baseline"), "e2e": ft["e2e"],
                "gpu_launches": ft["launches_per_step"] * args.steps, "extra": {"loss": ft["loss"], "kernels_per_step": ft["kernels_per_step"], "fm_chunk": args.fm_chunk}}

    if args.dump_outputs and c.rank == 0:
        headline = ft if args.workload == "fm" else last if args.workload == "sweep" else r
        dump_outputs(args.dump_outputs, headline["outputs"])
    if c.rank == 0:
        def clean(o):
            if isinstance(o, dict):
                return {k: clean(v) for k, v in o.items() if k not in ("eng", "outputs")}
            if isinstance(o, list):
                return [clean(v) for v in o]
            return o
        print(json.dumps(clean(line)))
    if c.world > 1:
        c.dist.destroy_process_group()


if __name__ == "__main__":
    main()
