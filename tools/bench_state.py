#!/usr/bin/env python
"""Per-stream state export / import (se_crn_state_export / _import, se_fsn_state_export / _import) against one
streaming step at the same stream count, on one GPU.

    python tools/bench_state.py [--iters 30] [--warmup 5] [--out FILE]

Cases: CRN teacher, 1024 streams, fp16 and tf32; FullSubNet full configuration, 256 streams, fp16 and tf32; and the
compaction of a 1024-stream CRN teacher context (fp16) after a random 25 % of its streams ended: the live rows behind
the new end are exported and imported into the holes.  Every working set is larger than the 126 MB L2 (1024 x 0.25 MB,
256 x 0.9-1.2 MB records plus the same again in the arena), except the compaction's (256 records), which is what a
server moves.  Per iteration the step, the export and the import are timed with CUDA events, one after the other, so
that the three alternate in the same run; a JSON line per case gives the median ms of each, the bytes moved (read +
write: 2 x rows x record bytes), GB/s and their share of the 7.7 TB/s HBM3e bandwidth of the data sheet, and the
export / import time as a fraction of the step.  The card's name and power limit are read in the same call; --out also
writes the lines to FILE.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from speech_enhancement_mi_b200 import CRN_ELU, fullsubnet, synth  # noqa: E402
from speech_enhancement_mi_b200._native import check, lib  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
TEACHER = dict(num_channels=[16, 32, 64, 128], num_freqs=201, hidden=512, num_layers=2, num_inputs=3, kernel_size=3)
FSN_FULL = dict(num_freqs=201, num_mics=3, fb_hidden=512, sb_hidden=384, sb_num_neighbors=15, fb_num_neighbors=0,
                num_layers=2)


def card():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["gpu"], info["power_limit"] = [s.strip() for s in q[0].split(",")]
    except (OSError, IndexError, ValueError, subprocess.TimeoutExpired):
        info["power_limit"] = "unknown"
    return info


def crn_teacher(precision, capacity):
    m = CRN_ELU.TemporalCRN(segment_length=3200, precision=precision, max_streams=capacity, **TEACHER)
    w = synth.with_alias_keys(synth.make_crn_weights(seed=0, **TEACHER))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    return m.eval()


def fsn_full(precision, capacity):
    m = fullsubnet.FullSubNet(num_freqs=201, look_ahead=0, sequence_model="LSTM", fb_num_neighbors=0,
                              sb_num_neighbors=15, fb_output_activate_function="ReLU",
                              sb_output_activate_function=False, fb_model_hidden_size=512, sb_model_hidden_size=384,
                              num_mics=3, num_layers=2, weight_init=False, sample_rate=16000, segment_length=3200,
                              win_length=25, hop_length=10, n_fft=400, max_streams=capacity, precision=precision)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in synth.make_fsn_weights(seed=5, **FSN_FULL).items()})
    return m.eval()


def measure(model, kind, B, src_rows, dst_rows, iters, warmup):
    """median ms of (step at B, export of src_rows, import of those records into dst_rows), alternated"""
    L = lib()
    bytes_fn, export_fn, import_fn, layout_fn = (
        (L.se_crn_state_bytes_per_stream, L.se_crn_state_export, L.se_crn_state_import, L.se_crn_state_layout)
        if kind == "crn" else
        (L.se_fsn_state_bytes_per_stream, L.se_fsn_state_export, L.se_fsn_state_import, L.se_fsn_state_layout))
    mix, _ = synth.make_mixture(min(B, 16), 3200)
    chunk = torch.from_numpy(np.tile(mix, (B // mix.shape[0] + 1, 1, 1))[:B].copy()).cuda()
    out = torch.empty((B, 1600), device="cuda")
    for _ in range(3):  # the streams carry state; the step graph for B is captured
        model.process_chunk(chunk, out)
    ctx = model._ctx
    rec = int(bytes_fn(ctx))
    n = len(src_rows)
    buf = torch.empty((n, rec), dtype=torch.uint8, device="cuda")
    src = (C.c_int32 * n)(*src_rows)
    dst = (C.c_int32 * n)(*dst_rows)
    layout = C.c_uint64(int(layout_fn(ctx)))
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    times = []
    for it in range(warmup + iters):
        ev[0].record(stream)
        model.process_chunk(chunk, out)
        ev[1].record(stream)
        check(export_fn(ctx, src, n, C.c_void_p(buf.data_ptr()), sp), "export")
        ev[2].record(stream)
        check(import_fn(ctx, dst, n, C.c_void_p(buf.data_ptr()), layout, sp), "import")
        ev[3].record(stream)
        torch.cuda.synchronize()
        if it >= warmup:
            times.append([ev[i].elapsed_time(ev[i + 1]) for i in range(3)])
    step, exp, imp = np.median(np.array(times), axis=0).tolist()
    moved = 2.0 * n * rec
    return dict(record_bytes=rec, rows=n, bytes_moved=moved, step_ms=step, export_ms=exp, import_ms=imp,
                export_GBps=moved / exp / 1e6, import_GBps=moved / imp / 1e6,
                export_hbm_share=moved / exp / 1e-3 / HBM_BYTES_PER_S, import_hbm_share=moved / imp / 1e-3 / HBM_BYTES_PER_S,
                export_vs_step=exp / step, import_vs_step=imp / step)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_state.py measures on a CUDA device; none is present")
    hw = card()
    lines = []
    cases = [("crn", "fp16", 1024), ("crn", "tf32", 1024), ("fsn", "fp16", 256), ("fsn", "tf32", 256)]
    with torch.no_grad():
        for kind, precision, B in cases:
            model = crn_teacher(precision, B) if kind == "crn" else fsn_full(precision, B)
            rows = list(range(B))
            r = measure(model, kind, B, rows, rows, args.iters, args.warmup)
            lines.append(dict(case=f"{kind}_{'teacher' if kind == 'crn' else 'full'}_{precision}", streams=B, **r, **hw))
            del model
            torch.cuda.empty_cache()
        # compaction: 25 % of 1024 streams ended at random; the live rows at or behind the new end fill the holes
        B = 1024
        ended = np.sort(np.random.default_rng(0).choice(B, B // 4, replace=False))
        n_live = B - len(ended)
        holes = [int(r) for r in ended if r < n_live]
        tail = [int(r) for r in np.setdiff1d(np.arange(B), ended) if r >= n_live]
        model = crn_teacher("fp16", B)
        r = measure(model, "crn", B, tail, holes, args.iters, args.warmup)
        lines.append(dict(case="crn_teacher_fp16_compaction_25pct", streams=B, **r, **hw))
    for line in lines:
        print(json.dumps(line))
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
