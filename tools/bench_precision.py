"""The arithmetic modes side by side on one GPU: CRN chunk step in fp32 / 3xtf32 / tf32, alternated in rounds, FullSubNet
utterances in tf32 / 3xtf32, and how far the 3xtf32 teacher output is from the fp32 one at full size.

    python tools/bench_precision.py [--rounds 3] [--steps 20] [--out FILE]

Prints one JSON line per measurement and a summary line; --out also writes them to FILE.  Every timing is device time
(CUDA events, tools/bench_parts.py); the card's name and power limit are read in the same call.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))


def card():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q[0].split(",")]
    except (OSError, IndexError, ValueError, subprocess.TimeoutExpired):
        info["power_limit"] = "unknown"
    return info


def output_difference(streams, steps):
    """Teacher, `streams` streams, `steps` chunk steps from a reset state in fp32 and in 3xtf32 on the same input:
    max |y_3xtf32 - y_fp32| / max(1, peak |y_fp32|)."""
    import numpy as np
    import torch
    from bench_parts import build_crn, synthetic_signal
    sig = torch.from_numpy(synthetic_signal(streams, (steps + 1) * 1600)).cuda()
    outs = {}
    for precision in ("fp32", "3xtf32"):
        model, _ = build_crn("teacher", precision, streams)
        model.reset()
        outs[precision] = np.concatenate(
            [model.process_chunk(sig[:, :, 1600 * k:1600 * k + 3200]).cpu().numpy() for k in range(steps)], axis=-1)
        model._destroy_ctx()
        del model
    peak = max(1.0, float(np.abs(outs["fp32"]).max()))
    return {"what": "3xtf32 vs fp32 output", "model": "teacher", "streams": streams, "chunk_steps": steps,
            "max_abs_rel_to_peak": float(np.abs(outs["3xtf32"] - outs["fp32"]).max()) / peak, "peak": peak,
            "fp32_tolerance": 2e-5}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--fsn-streams", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_precision.py measures on the GPU; no CUDA device found")
    from bench_parts import crn_stream, fsn_utterances
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    emit(dict(card(), what="card"))
    modes = ("fp32", "3xtf32", "tf32")
    times = {(m, p): [] for m in ("teacher", "student") for p in modes}
    for r in range(a.rounds):
        for model, streams in (("teacher", 1024), ("student", 2048)):
            for p in modes:  # alternated: the modes share every round's conditions
                res = crn_stream(model, streams, p, a.steps)
                times[(model, p)].append(res["ms_per_step"])
                emit(dict(res, round=r))
    fsn = {}
    for r in range(2):
        for p in ("tf32", "3xtf32"):
            res = fsn_utterances(a.fsn_streams, 3.0, 2, p)
            fsn.setdefault(p, []).append(res["value"])
            emit(dict(res, round=r))
    diff = output_difference(1024, 4)
    emit(diff)
    summary = {"what": "summary"}
    for (model, p), v in times.items():
        summary[f"{model}_{p}_ms_min"] = min(v)
    for model in ("teacher", "student"):
        summary[f"{model}_3xtf32_over_fp32"] = min(times[(model, "3xtf32")]) / min(times[(model, "fp32")])
    for p, v in fsn.items():
        summary[f"fsn_{p}_audio_s_per_s_max"] = max(v)
    summary["out_diff_rel_to_peak"] = diff["max_abs_rel_to_peak"]
    emit(summary)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(d) + "\n" for d in lines))


if __name__ == "__main__":
    main()
