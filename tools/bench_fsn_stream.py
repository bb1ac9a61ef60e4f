#!/usr/bin/env python
"""FullSubNet streaming step (FullSubNet.process_chunk / se_fsn_process_chunk) against the chunk loop of
realtime_process(train=False), full configuration (config.yaml:153-172), on one GPU.

    python tools/bench_fsn_stream.py [--streams 1,256,1024] [--precisions fp16,tf32] [--steps 200] [--rounds 2]
                                     [--out FILE]

Per (precision, streams) one JSON line:
  step   device-resident steps (chunk in device memory, result into device memory), each timed with CUDA events
         after a warm-up: mean ms per step over the whole timed window, p50 / p99 of the per-step times, enhanced
         audio-s/s = streams x 0.1 s / step, achieved TFLOP/s against the algorithmic 15,547.6 MFLOP per stream-chunk
  loop   realtime_process(train=False) of `--seconds` utterances at the same stream count, per chunk
         (tools/bench_fsn.py's ms_per_chunk_step); step windows and utterance batches alternate over `--rounds` rounds
  e2e    process_chunk_host with pinned host buffers, the copies inside the timed window
The card's name and power limit are read in the same call; --out also writes the lines to FILE.
"""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from speech_enhancement_mi_b200 import _native, fullsubnet, synth  # noqa: E402

MFLOP_PER_STREAM_CHUNK = 15547.6  # SURVEY.md section 8(d), the full configuration
CFG = dict(num_freqs=201, num_mics=3, fb_hidden=512, sb_hidden=384, sb_num_neighbors=15, fb_num_neighbors=0,
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


def build(precision, capacity):
    m = fullsubnet.FullSubNet(num_freqs=201, look_ahead=0, sequence_model="LSTM", fb_num_neighbors=0,
                              sb_num_neighbors=15, fb_output_activate_function="ReLU",
                              sb_output_activate_function=False, fb_model_hidden_size=512, sb_model_hidden_size=384,
                              num_mics=3, num_layers=2, weight_init=False, sample_rate=16000, segment_length=3200,
                              win_length=25, hop_length=10, n_fft=400, max_streams=capacity, precision=precision)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in synth.make_fsn_weights(seed=5, **CFG).items()})
    return m.eval()


def signal(B, L):
    base, _ = synth.make_mixture(min(B, 16), L)
    return np.ascontiguousarray(np.tile(base, ((B + base.shape[0] - 1) // base.shape[0], 1, 1))[:B])


def measure(model, B, args, info):
    sig = signal(B, int(args.seconds * 16000))
    mix = torch.from_numpy(sig).cuda()
    chunks = [mix[:, :, 1600 * i:1600 * i + 3200].contiguous() for i in range(4)]
    out = torch.empty((B, 1600), dtype=torch.float32, device="cuda")
    L = mix.shape[-1]
    n_chunks = _native.chunk_grid(L + 1600, 3200)[1]

    model.realtime_process(mix, None, flag=False, train=False)  # warm-up: graphs, scratch
    model.reset_state(B)
    for i in range(args.warmup):
        model.process_chunk(chunks[i % 4], out)
    torch.cuda.synchronize()
    step_total, step_times, loop_total = 0.0, [], 0.0
    for _ in range(args.rounds):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        ev[0].record()
        for i in range(args.steps):
            model.process_chunk(chunks[i % 4], out)
            ev[i + 1].record()
        torch.cuda.synchronize()
        step_total += ev[0].elapsed_time(ev[-1])
        step_times += [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            model.realtime_process(mix, None, flag=False, train=False)
        e1.record()
        torch.cuda.synchronize()
        loop_total += e0.elapsed_time(e1)
    step_ms = step_total / (args.rounds * args.steps)
    loop_ms = loop_total / (args.rounds * args.reps * n_chunks)

    host_in = [chunks[i].cpu().pin_memory() for i in range(4)]
    host_out = [torch.empty((B, 1600), dtype=torch.float32).pin_memory() for _ in range(2)]
    model.reset_state(B)
    for i in range(args.warmup):
        model.process_chunk_host(host_in[i % 4], host_out[i % 2])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    done = None
    for i in range(args.steps):
        done = model.process_chunk_host(host_in[i % 4], host_out[i % 2])
    torch.cuda.current_stream().wait_event(done)  # the last result has reached host memory
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1) / args.steps

    def rate(ms):
        return B * 0.1 / (ms * 1e-3)

    return {"what": "FullSubNet streaming step vs chunk loop", "precision": model.precision, "streams": B,
            "step": {"ms_mean": step_ms, "ms_p50": float(np.percentile(step_times, 50)),
                     "ms_p99": float(np.percentile(step_times, 99)), "steps_timed": len(step_times),
                     "audio_s_per_s": rate(step_ms),
                     "achieved_tflops": MFLOP_PER_STREAM_CHUNK * 1e6 * B / (step_ms * 1e-3) / 1e12},
            "loop": {"ms_per_chunk_step": loop_ms, "utterance_s": args.seconds, "chunks": n_chunks,
                     "utterance_batches_timed": args.rounds * args.reps, "audio_s_per_s": B * args.seconds /
                     (loop_total / (args.rounds * args.reps) * 1e-3)},
            "step_over_loop": step_ms / loop_ms,
            "e2e": {"ms_per_step": e2e_ms, "audio_s_per_s": rate(e2e_ms),
                    "api": "FullSubNet.process_chunk_host(pinned chunk, pinned result)"},
            **info, "data": "synthetic, seed-5 weights"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="1,256,1024")
    ap.add_argument("--precisions", default="fp16,tf32")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--seconds", type=float, default=3.0)
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.steps < 200:
        ap.error("--steps: time at least 200 steps")
    if not torch.cuda.is_available():
        sys.exit("bench_fsn_stream.py needs a CUDA device")
    streams = [int(s) for s in args.streams.split(",")]
    info = card()
    lines = []
    for precision in args.precisions.split(","):
        model = build(precision, max(streams))
        for B in streams:
            line = measure(model, B, args, info)
            print(json.dumps(line), flush=True)
            lines.append(line)
        del model
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
