"""Cost of saving the path (SaveAt(ts)): LJ13 sample_and_log_prob_cnf (BASELINE.json configs[1], exact log q, fixed
dt = 0.05 as in bench.py's headline workload) with ts=None and with ts = linspace(0, 1, 101), on the automatic engine
(tcgen05) and on forced fp32 SIMT.  The two variants alternate, so drifts of a shared machine hit both alike.
Usage (GPU box): python tools/saveat_overhead.py [--batch 10000] [--simt-batch 2072] [--reps 2]"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from ecnf_b200.cnf import build_cnf, sample_and_log_prob_cnf
from ecnf_b200.engine import PackedParams
from ecnf_b200.nets.egnn import init_flat_params

LJ13 = dict(n_frames=13, dim=3, sigma_min=0.01, base_scale=1.0, n_blocks_egnn=3, mlp_units=(128,) * 3,
            n_invariant_feat_hidden=64, time_embedding_dim=8, n_features=1)


def card() -> str:
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit not read"
    return f"{name} ({q})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=10_000, help="trajectories per timed call on the automatic engine")
    ap.add_argument("--simt-batch", type=int, default=148 * 14,
                    help="trajectories per timed call on fp32 SIMT (about 6x slower per trajectory than tcgen05)")
    ap.add_argument("--reps", type=int, default=2, help="timed calls per variant (alternating)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    cnf = build_cnf(**LJ13)
    eng = cnf.engine
    params = PackedParams(torch.from_numpy(init_flat_params(eng, 0, 1.0)).cuda())
    ts = np.linspace(0.0, 1.0, 101)
    print(f"# {card()}; LJ13 sample_and_log_prob_cnf, exact log q, fixed dt 0.05, {len(ts)} save times", flush=True)
    for engine, label, B in ((0, "auto (tcgen05)", args.batch), (1, "fp32 SIMT", args.simt_batch)):
        eng.set_engine(engine)

        def call(n, with_ts):
            return sample_and_log_prob_cnf(cnf, params, 7, use_fixed_step_size=True, n_samples=n, check_status=False,
                                           ts=ts if with_ts else None)
        for with_ts in (False, True):      # warm-up: module load, workspace allocation
            call(296, with_ts)
        torch.cuda.synchronize()
        ms = {False: [], True: []}
        for _ in range(args.reps):
            for with_ts in (False, True):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                call(B, with_ts)
                b.record()
                torch.cuda.synchronize()
                ms[with_ts].append(a.elapsed_time(b))
        rate = {k: B / (min(v) / 1e3) for k, v in ms.items()}
        print(f"{label:15s} B={B:6d}  ts=None {rate[False]:9.1f} samples/s  ts=101 times {rate[True]:9.1f} samples/s  "
              f"ratio {rate[True] / rate[False]:.4f}  (ms per call: none {['%.1f' % v for v in ms[False]]}, "
              f"ts {['%.1f' % v for v in ms[True]]})", flush=True)
    eng.set_engine(0)


if __name__ == "__main__":
    main()
