import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from tools import bench_parts
dev = torch.device("cuda", 0)
which = sys.argv[1]
if "t" in which:
    r = bench_parts.crn_stream("teacher", 1024, "tf32", steps=5, dev=dev); print("tf32", r["ms_per_step"], flush=True)
if "p" in which:
    r = bench_parts.crn_stream("teacher", 1024, "fp32", steps=3, dev=dev); print("fp32", r["ms_per_step"], flush=True)
if "l" in which:
    for nb in (1, 16):
        r = bench_parts.crn_stream("teacher", nb, "fp16", steps=20, latency_steps=300, dev=dev); print("lat", nb, r["ms_per_step"], flush=True)
if "s" in which:
    r = bench_parts.crn_stream("student", 2048, "fp16", steps=5, dev=dev); print("student", r["ms_per_step"], flush=True)
if "c" in which:
    r = bench_parts.crn_stream("teacher", 1024, "fp16", steps=5, dev=dev); print("teacher", r["ms_per_step"], flush=True)
if "f" in which:
    r = bench_parts.fsn_utterances(256, seconds=3.0, reps=1, precision="fp16", dev=dev); print("fsn", r["ms_per_utterance_batch"], flush=True)
r = bench_parts.train_step(batch=1, seconds=2.0, steps=5, warmup=2, precision="tf32", graph=True, dev=dev)
print(which, "train", r["ms_per_step"], r["ms_allreduce_clip_adam_rebind"], flush=True)
