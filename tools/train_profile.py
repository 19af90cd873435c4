"""A few QM9-positional flow-matching steps (batch 512) for per-kernel timing under ncu (GPU box).
Usage: python tools/train_profile.py [graphs per chunk, 0 = the whole minibatch]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import argparse
import bench
c = bench.setup(argparse.Namespace())
r = bench.bench_train(c, steps=2, cpu=False, chunk=int(sys.argv[1]) if len(sys.argv) > 1 else 0, count=False)
print(r["value"], "steps/s", r["ms_per_step"], "ms")
