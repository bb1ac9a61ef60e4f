#!/usr/bin/env python
"""Cost of d loss / d mixture in the CRN training backward (se_crn_train_backward_input).

    python tools/bench_input_grad.py [--precision tf32] [--reps 30] [--seconds 2] [--batches 1,8]

Teacher model, synthetic [batch, 3, seconds*16000] pieces (the tools/bench_train.py piece is batch 1, 2 s).  Three forms
of the backward, alternated within one run (forward, then the timed backward of one form, round robin), each timed with
CUDA events around the backward call alone:
  params       today's backward: parameter gradients only (se_crn_train_backward)
  params+dmix  parameter gradients and d mixture
  dmix         d mixture alone (grad_flat = NULL: no weight-gradient GEMMs, frozen model)
Prints one JSON line per (batch, form) with the median and quartiles over the repetitions, and the card and its power
limit."""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from speech_enhancement_mi_b200 import CRN_ELU, synth, workload  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--precision", default="tf32")
ap.add_argument("--reps", type=int, default=30)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--seconds", type=float, default=2.0)
ap.add_argument("--batches", default="1,8")
args = ap.parse_args()


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


model = CRN_ELU.TemporalCRN(segment_length=3200, dropout=0.0, precision=args.precision, device=0, **workload.TEACHER)
w = synth.make_crn_weights(seed=0, **workload.TEACHER)
model.load_state_dict({k: torch.from_numpy(v) for k, v in synth.with_alias_keys(w).items()})
model = model.cuda().train()
FORMS = {"params": dict(mixture=False, params=True), "params+dmix": dict(mixture=True, params=True),
         "dmix": dict(mixture=True, params=False)}
gpu = card()
for B in [int(b) for b in args.batches.split(",")]:
    L = int(args.seconds * 16000)
    mix, _ = synth.make_mixture(B, L)
    x = torch.from_numpy(mix).cuda()
    dpred = torch.randn(B, L, generator=torch.Generator().manual_seed(1)).cuda()
    model.realtime_process(x, False)  # creates the training context for this piece
    times = {f: [] for f in FORMS}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(args.warmup + args.reps):
        for form, kw in FORMS.items():
            with torch.no_grad():
                model._train_forward(x, False)
            e0.record()
            model._train_backward(dpred, mixture=x if kw["mixture"] else None, params=kw["params"])
            e1.record()
            torch.cuda.synchronize()
            if it >= args.warmup:
                times[form].append(e0.elapsed_time(e1))
    base = float(np.median(times["params"]))
    for form, t in times.items():
        med = float(np.median(t))
        print(json.dumps({"metric": "CRN training backward", "form": form, "batch": B, "piece_seconds": args.seconds,
                          "precision": args.precision, "ms_median": round(med, 4),
                          "ms_q25": round(float(np.percentile(t, 25)), 4), "ms_q75": round(float(np.percentile(t, 75)), 4),
                          "vs_params": round(med / base, 4), "reps": args.reps, "gpu": gpu}), flush=True)
