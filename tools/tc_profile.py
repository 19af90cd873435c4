"""Coarse per-phase cycle breakdown of the tensor-core solve kernel (CTA 0), read back from the workspace header.
Usage (on a GPU box; build the counter library first, here or there:  ECNF_TC_PROFILE=1 python ecnf_b200/build.py):
    ECNF_B200_LIB=ecnf_b200/libecnf_b200_prof.so python tools/tc_profile.py [lj13|aldp|dw4] [batch] [sample]
("sample": the primal-only sample_cnf path instead of sample + exact log q)"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from ecnf_b200 import lib as L
from ecnf_b200.cnf import build_cnf
from ecnf_b200.engine import PackedParams
from ecnf_b200.nets.egnn import init_flat_params

# epilogue thread 0: phases + its own time inside the edge phase; side thread 0: its own loop
NAMES = ["node_pre", "edge", "node_post", "  epi: wait_mma", "  epi: chain (ld+act+split+st)", "  epi: messages", "  epi: head dot", "  epi: weight_load",
         "  side: wait_heads", "  side: gather issue", "  side: coords", "  side: meta", "  side: copy wait + arrive", "  epi: node build",
         "  epi: shape basis + maps"]
NFALLBACK = len(NAMES)    # the next counter: evaluations of CTA 0 on the canonical path (degenerate rotations), not cycles
NTOP = 3
name = sys.argv[1] if len(sys.argv) > 1 else "lj13"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 148
MODE = L.MODE_SAMPLE if len(sys.argv) > 3 and sys.argv[3] == "sample" else L.MODE_SAMPLE_LOGQ
cfg = bench.CFGS[name]
cnf = build_cnf(**cfg)
eng = cnf.engine
params = PackedParams(torch.from_numpy(init_flat_params(eng, 0, 1.0)).cuda())
x0 = eng.base_sample(2, B)
feat = (torch.arange(cfg["n_frames"], dtype=torch.int32, device="cuda") % cfg["n_features"]).repeat(B, 1).contiguous()
for it in range(2):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    x1, logs, stats = eng.solve(params, MODE, x0, feat, L.make_ctrl(use_fixed_step_size=True))
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
ws = next(v for k, v in eng._ws.items() if k[0] == "solve")
prof = ws[64:64 + 8 * (len(NAMES) + 1)].view(torch.int64).cpu().numpy()
evals = int(stats[:, 2].sum()) / min(B, 148)
tot = prof[:NTOP].sum()
print(f"{name} B={B} kernel {ms:.1f} ms ({B / ms * 1e3:.1f} samples/s); CTA0 ran ~{evals:.0f} evals; instrumented cycles {tot/1e6:.1f} M ({tot/evals/1e3:.0f} k/eval)")
for nm, v in zip(NAMES, prof):
    print(f"  {nm:34s} {v/1e6:10.2f} Mcyc  {100*v/tot:5.1f}%   {v/evals/1e3:8.1f} kcyc/eval")
print(f"  evaluations on the canonical path (CTA 0): {int(prof[NFALLBACK])}")
