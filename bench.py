#!/usr/bin/env python
"""Headline benchmark: enhanced audio-seconds per wall-second of the CRN_ELU streaming path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--streams B] [--precision fp32|tf32]
                    [--dump-outputs DIR]

A step advances every concurrent stream by one 3200-sample chunk at hop 1600 (0.1 s of new audio per stream):
STFT -> features -> preconv/encoder -> GRU -> decoder -> cIRM mask -> iSTFT -> overlap-add, with the per-stream causal
state carried in HBM.  Workload = BASELINE.json configs[1]: teacher CRN_ELU, 1024 concurrent synthetic streams per GPU.
Streams are independent, so N GPUs run N x 1024 streams with no data-path collective ("weak" scaling); NCCL is used
only to take the max of the device time over ranks.

`--impl reference` times the UNMODIFIED reference (`oracle/_ref/reference.zip`, packed from /root/reference by
`oracle/build_ref.py`; `CRN_ELU.TemporalCRN.realtime_process` on torch CPU ops, as predict.py:48,92 runs it) on the
host cores, on a bounded sample of the same workload; without the archive it falls back to the oracle restatement.

Besides the headline (fp16 operand mode) the line carries, measured in the same run: `modes` (the same workload in tf32
and exact fp32 mode), `latency` (p50 / p99 chunk latency at 1 and 16 streams), and `configs` -- the other BASELINE.json
configurations: the distilled student at 2048 streams per GPU (configs[2]), FullSubNet on 3 s utterances (configs[3]) and
the training step with its NCCL gradient all-reduce (configs[4]).  `--no-extras` skips them.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

_REAL_STDOUT = sys.stdout
METRIC = "enhanced audio-sec/sec (CRN_ELU streaming)"
UNIT = "audio-s/s"
RING = 16  # distinct hops of input per stream kept in HBM (input ring 1024*3*27200*4 B = 334 MB > 126 MB L2)
DUMP_BYTES = 64 << 20  # --dump-outputs keeps a dump at most this large


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=1024, help="concurrent streams per GPU")
    ap.add_argument("--precision", default=os.environ.get("SE_B200_PRECISION", "fp16"))
    ap.add_argument("--model", default="teacher", choices=["teacher", "student"])
    ap.add_argument("--cpu-streams", type=int, default=16, help="streams in the CPU baseline sample")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU time budget of the cpu_baseline leg")
    ap.add_argument("--latency-steps", type=int, default=1000, help="steps of the p99 chunk-latency pass")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip modes / latency / configs (headline only)")
    ap.add_argument("--student-streams", type=int, default=2048, help="configs[2]: 16384 streams over 8 GPUs")
    ap.add_argument("--fsn-streams", type=int, default=256, help="configs[3]: FullSubNet utterances per GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--profile-step", action="store_true",
                    help="warm up, then run ONE chunk step inside cudaProfilerStart/Stop (for ncu --profile-from-start off) "
                         "and write the kernel labels of that step to gpurun_out/kernel_labels.json")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned to DIR/enhanced.npy "
                         "([streams, 1600] float32 enhanced samples), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    return args


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU while the timed region runs: NVML in-process, back to back with a 5 ms pause (an
    `nvidia-smi -lms` child needs about a second to come up on an 8-GPU box and then misses short timed regions); falls
    back to the nvidia-smi loop when the NVML binding is unavailable."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASON_BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index, uuid=None):
        super().__init__(daemon=True)
        self.index = index
        self.uuid = uuid
        self.samples = []  # [sm_mhz, sm_max_mhz, hw_slowdown, hw_thermal_slowdown, sw_thermal_slowdown, sw_power_cap]
        self.proc = None
        self.stamps = []         # wall-clock time of every NVML sample
        self.window = [None, None]  # [start, end] of the timed region: only samples inside it are reported
        self._halt = threading.Event()

    def _run_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid) if self.uuid else pynvml.nvmlDeviceGetHandleByIndex(self.index)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        while not self._halt.is_set():
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            try:
                bits = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                bits = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.stamps.append(time.time())
            self.samples.append([str(sm), str(mx)] + [("Active" if bits & self.REASON_BITS[n] else "Not Active") for n in
                                                      ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                                       "sw_power_cap")])
            self._halt.wait(0.005)

    def run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self._halt.set()
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        samples = self.samples
        if self.window[0] is not None and len(self.stamps) == len(self.samples):
            lo, hi = self.window[0], self.window[1] if self.window[1] is not None else float("inf")
            inside = [x for x, ts in zip(self.samples, self.stamps) if lo <= ts <= hi]
            samples = inside or samples
        for s in samples:
            try:
                sm.append(int(float(s[0])))
                mx = max(mx, int(float(s[1])))
                for n, v in zip(names, s[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# synthetic input
# ----------------------------------------------------------------------------------------------------------------
def synthetic_signal(n_streams, n_samples):
    """[n_streams, 3, n_samples] float32 noisy 3-mic streams: 32 base mixtures from synth, tiled with per-stream gains."""
    import numpy as np
    from speech_enhancement_mi_b200 import synth
    base, _ = synth.make_mixture(min(n_streams, 32), n_samples)
    reps = (n_streams + base.shape[0] - 1) // base.shape[0]
    sig = np.tile(base, (reps, 1, 1))[:n_streams].copy()
    gains = 0.5 + 0.5 * synth.uniform01(2021, n_streams, stream=7).astype(np.float32)
    sig *= gains[:, None, None]
    return sig


def dump_outputs(path, enhanced):
    """Writes the enhanced samples of the last timed step as path/enhanced.npy (float32).  Above DUMP_BYTES every k-th
    stream is kept: a fixed sample, so that the dumps of two builds line up stream for stream."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    stride = -(-enhanced.nbytes // DUMP_BYTES)
    np.save(os.path.join(path, "enhanced.npy"), np.ascontiguousarray(enhanced[::stride], dtype=np.float32))


def build_model(args, max_streams):
    import torch
    from speech_enhancement_mi_b200 import CRN_ELU, distillation_crn, synth, workload
    cfg = workload.TEACHER if args.model == "teacher" else workload.STUDENT
    cls = CRN_ELU.TemporalCRN if args.model == "teacher" else distillation_crn.TemporalCRN
    model = cls(segment_length=3200, dropout=0.0, precision=args.precision, max_streams=max_streams, **cfg)
    w = synth.make_crn_weights(seed=0, **cfg)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in synth.with_alias_keys(w).items()}, strict=True)
    return model.eval(), cfg


# ----------------------------------------------------------------------------------------------------------------
# CPU legs: the UNMODIFIED reference from oracle/_ref (kind "reference"), else the oracle restatement (kind "port").
# The only places bench.py touches oracle/ -- as the thing timed BESIDE the product, never inside it.
# ----------------------------------------------------------------------------------------------------------------
def _reference_model(args):
    """(model, kind): the reference's own TemporalCRN with the synthetic weights, or None when the archive is absent."""
    import torch
    from oracle import ref_loader
    from speech_enhancement_mi_b200 import synth, workload
    if not ref_loader.available():
        return None
    cfg = workload.TEACHER if args.model == "teacher" else workload.STUDENT
    if args.model == "teacher":
        (mod,) = ref_loader.load(("CRN_ELU",))
        model = mod.TemporalCRN(segment_length=3200, dropout=0.0, **cfg)
    else:
        (mod,) = ref_loader.load(("distillation_crn",))
        model = mod.TemporalCRN(segment_length=3200, dropout=0.0, **cfg)
    w = synth.make_crn_weights(seed=0, **cfg)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in synth.with_alias_keys(w).items()}, strict=True)
    return model.eval()


def _cpu_run(args, n_streams, steps, warmup, budget_s=None):
    """Times the CPU implementation on `n_streams` of the workload's streams.  A step = every stream advanced by one second
    of audio through the reference's public call `realtime_process` (10 chunk hops + its own padding chunks); the port
    advances chunk by chunk.  Returns (audio-s/s, ms per step, steps done, kind, cores, description)."""
    import torch
    from speech_enhancement_mi_b200 import workload
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = _reference_model(args)
    L = 16000
    sig = torch.from_numpy(synthetic_signal(n_streams, L))
    times = []
    with torch.no_grad():
        if ref is not None:
            def step():
                y = ref.realtime_process(sig)
                return y[0] if isinstance(y, tuple) else y
            audio_per_step = n_streams * L / 16000.0
            kind = "reference"
            what = (f"unmodified reference {'CRN_ELU' if args.model == 'teacher' else 'distillation_crn'}.TemporalCRN."
                    f"realtime_process (oracle/_ref/reference.zip) on [{n_streams}, 3, {L}] per step")
        else:
            from oracle.crn_oracle import CRNOracle
            from speech_enhancement_mi_b200 import synth
            cfg = workload.TEACHER if args.model == "teacher" else workload.STUDENT
            w = synth.make_crn_weights(seed=0, **cfg)
            oracle = CRNOracle({k: torch.from_numpy(v) for k, v in w.items()}, segment_length=3200,
                               student=args.model == "student", **cfg)
            state = {"carry": None, "i": 0}

            def step():
                off = (state["i"] % 8) * 1600
                state["i"] += 1
                out, state["carry"] = oracle.stream_step(sig[:, :, off:off + 3200], state["carry"])
                return out
            audio_per_step = n_streams * workload.AUDIO_SEC_PER_STEP
            kind = "port"
            what = f"oracle/crn_oracle.py stream_step (restating CRN_ELU.py:367-509) on {n_streams} streams per step"
        for _ in range(max(warmup, 1)):
            step()
        t_start = time.perf_counter()
        while True:
            t0 = time.perf_counter()
            step()
            times.append(time.perf_counter() - t0)
            if budget_s is None and len(times) >= steps:
                break
            if budget_s is not None and len(times) >= 2 and time.perf_counter() - t_start > budget_s:
                break
    mean = sum(times) / len(times)
    return audio_per_step / mean, mean * 1e3, len(times), kind, cores, what


def cpu_baseline(args, n_streams, budget_s):
    value, ms, n, kind, cores, what = _cpu_run(args, n_streams, steps=0, warmup=1, budget_s=budget_s)
    return {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{n_streams} of the workload's streams, {n} steps, fp32 torch CPU ops with {cores} threads: {what}",
            "ms_per_step": ms}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.cpu_streams
    value, ms, steps, kind, cores, what = _cpu_run(args, n, steps=args.steps, warmup=max(args.warmup, 1))
    sample = f"{n} of the {args.streams} streams per step, {steps} steps, fp32 torch CPU ops with {cores} threads: {what}"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": max(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"CRN_ELU {args.model} batched streaming inference, {args.streams} concurrent synthetic "
                               f"streams per GPU, 3200-sample chunks at hop 1600 (BASELINE.json configs[1])",
                   "streams_per_gpu": args.streams, "precision": "fp32", "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


# ----------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    # stdout carries exactly ONE JSON line: anything a library prints to fd 1 (e.g. the "NCCL version" banner) goes to
    # stderr instead; the result line is written to the saved descriptor
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)

    import ctypes as C

    import torch
    import torch.distributed as dist
    from speech_enhancement_mi_b200 import workload
    from speech_enhancement_mi_b200._native import check, lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200 (no CPU fallback); use --impl reference for the CPU baseline")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = args.streams
    model, cfg = build_model(args, B)
    sig_host = synthetic_signal(B, (RING + 1) * 1600)
    sig = torch.from_numpy(sig_host).to(dev)
    out = torch.empty((B, 1600), dtype=torch.float32, device=dev)

    def chunk_view(i):
        off = (i % RING) * 1600
        return sig[:, :, off:off + 3200]  # strided view: the kernel reads it in place

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    K, W = args.steps, max(args.warmup, 3)
    for i in range(W):
        model.process_chunk(chunk_view(i), out)
    barrier()
    if args.profile_step:
        L = lib()
        labels = ["set_io"]
        for i in range(L.se_crn_num_kernels(model._ctx)):
            name = C.create_string_buffer(96)
            check(L.se_crn_kernel_info(model._ctx, i, name, 96, None, None, None), "kernel_info")
            labels.append(name.value.decode())
        os.makedirs(os.path.join(REPO, "gpurun_out"), exist_ok=True)
        with open(os.path.join(REPO, "gpurun_out", "kernel_labels.json"), "w") as f:
            json.dump({"streams": B, "precision": args.precision, "labels": labels}, f)
        torch.cuda.profiler.start()
        model.process_chunk(chunk_view(W), out)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    try:
        gpu_uuid = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        gpu_uuid = None
    sampler = ClockSampler(local_rank, gpu_uuid)
    sampler.start()
    time.sleep(0.05)
    events = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    barrier()
    sampler.window[0] = time.time()
    events[0].record()
    for k in range(K):
        model.process_chunk(chunk_view(W + k), out)
        events[k + 1].record()
    barrier()
    sampler.window[1] = time.time()
    if args.dump_outputs and rank == 0:  # every rank runs the same streams
        dump_outputs(args.dump_outputs, out.cpu().numpy())
    total_ms = events[0].elapsed_time(events[K])
    lat = sorted(events[k].elapsed_time(events[k + 1]) for k in range(K))
    clocks = sampler.stop()
    # p99 chunk latency (BASELINE.json metric; SURVEY.md section 8(d): >= 1000 steps after warm-up): a separate pass so
    # that the percentile does not rest on the K timed steps alone.  Real-time deadline: 100 ms per chunk step.
    NLAT = max(K, args.latency_steps)
    if NLAT > K:
        lev = [torch.cuda.Event(enable_timing=True) for _ in range(NLAT + 1)]
        lev[0].record()
        for k in range(NLAT):
            model.process_chunk(chunk_view(W + K + k), out)
            lev[k + 1].record()
        torch.cuda.synchronize()
        lat = sorted(lev[k].elapsed_time(lev[k + 1]) for k in range(NLAT))
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / K
    value = world * B * workload.AUDIO_SEC_PER_STEP / (ms_per_step * 1e-3)

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timed region ------------
    e2e = None
    if not args.no_e2e:
        host_in = [torch.from_numpy(sig_host[:, :, (i % RING) * 1600:(i % RING) * 1600 + 3200].copy()).pin_memory()
                   for i in range(4)]
        host_out = [torch.empty((B, 1600), dtype=torch.float32).pin_memory() for _ in range(2)]
        model.reset()

        def e2e_step(i):  # public serving call: pinned host chunk in, pinned host result out, copies on side streams
            return model.process_chunk_host(host_in[i % 4], host_out[i % 2])

        for i in range(W):
            e2e_step(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        done = None
        for i in range(K):
            done = e2e_step(i)
        torch.cuda.current_stream().wait_event(done)  # the last result has reached host memory
        e1.record()
        barrier()
        te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": world * B * workload.AUDIO_SEC_PER_STEP / (float(te.item()) / K * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": B * 3 * 3200 * 4, "d2h_bytes_per_step": B * 1600 * 4,
               "ms_per_step": float(te.item()) / K,
               "api": "TemporalCRN.process_chunk_host(pinned chunk, pinned result): H2D, chunk step and D2H of "
                      "neighbouring steps overlap on three streams over double-buffered staging; every step's input "
                      "crosses PCIe and every step's result is read back inside the timed region"}

    # ---- per-kernel device times (CUDA events inside the library, on the launching stream) and rooflines ------------
    # Every kernel of the chunk step is timed alone (burst: back-to-back launches), with its ALGORITHMIC flops / bytes
    # (SURVEY.md section 8(d), DESIGN.md section 4) from the library's op table.  Kernels of one class (e.g. the 21
    # recurrent steps of a GRU layer) are grouped; `roofline` is the class with the largest share of the step.
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            mp = json.load(f)
        peaks.update({k: mp[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in mp})
        peaks["src"] = "measured"
    except Exception:
        pass
    # DRAM bytes per launch come from an ncu capture of one chunk step (tools/ncu_step_summary.py); they are reported only
    # when that capture was taken on the library this run loads (source hash recorded with the capture)
    traffic, traffic_note = {}, "no ncu capture for this build"
    try:
        from speech_enhancement_mi_b200 import build as native_build
        with open(os.path.join(REPO, "profiles", "ncu_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("source_hash") == native_build.source_hash():
            traffic = tj.get("dram_bytes_per_launch", {})
            traffic_note = f"ncu dram__bytes_read+write per launch, capture {tj.get('capture', '?')} of this build"
        else:
            traffic_note = "profiles/ncu_traffic.json was captured on another build of the library: not reported"
    except Exception:
        pass
    stages, kernels, roofline, step_aggregate = {}, [], None, None
    launches_per_chunk = lib().se_crn_launches_per_chunk(model._ctx)
    if rank == 0:
        import re
        L = lib()
        stage_names = ("stft", "preconv", "encoder", "gru", "decoder", "mask_istft", "roll")
        groups = {}
        for i in range(L.se_crn_num_kernels(model._ctx)):
            name = C.create_string_buffer(96)
            fl, by, stg = C.c_double(0), C.c_double(0), C.c_int(0)
            check(L.se_crn_kernel_info(model._ctx, i, name, 96, C.byref(fl), C.byref(by), C.byref(stg)), "kernel_info")
            ms = C.c_float(0)
            check(L.se_crn_time_kernel(model._ctx, i, B, 5, C.byref(ms)), "se_crn_time_kernel")
            key = re.sub(r"step\d+", "step", name.value.decode())
            g = groups.setdefault(key, {"name": key, "stage": stage_names[stg.value], "launches": 0, "ms_total": 0.0,
                                        "flops": fl.value * B, "bytes": by.value * B})
            g["launches"] += 1
            g["ms_total"] += ms.value
        model.reset()
        tot = sum(g["ms_total"] for g in groups.values())
        tensor_peak = peaks["bf16_tflops"]  # kernels are timed alone: burst figure
        for g in groups.values():
            ms = g["ms_total"] / g["launches"]
            k = {"name": g["name"], "stage": g["stage"], "launches": g["launches"], "ms": ms,
                 "share": g["ms_total"] / tot}
            # the binding floor of a kernel is the LARGER of its two floors: algorithmic flops at the tensor peak,
            # algorithmic bytes at the HBM peak; frac = that floor / measured time (both fractions are reported)
            f_t = g["flops"] / (ms * 1e-3) / 1e12 / tensor_peak
            f_h = g["bytes"] / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"]
            k["frac_tensor"], k["frac_hbm"] = f_t, f_h
            if f_t >= f_h:
                k.update(bound="tensor", achieved=f_t * tensor_peak, peak=tensor_peak, unit="TFLOP/s", frac=f_t)
                if args.precision == "tf32":
                    k["frac_of_tf32_rate"] = 2.0 * f_t
            else:
                k.update(bound="hbm", achieved=f_h * peaks["hbm_gbs"], peak=peaks["hbm_gbs"], unit="GB/s", frac=f_h)
            k["traffic"] = traffic.get(g["name"])
            kernels.append(k)
            st = stages.setdefault(g["stage"], {"ms": 0.0})
            st["ms"] += g["ms_total"]
        for st in stages.values():
            st["share"] = st["ms"] / tot
        # whole-step context for the per-kernel rooflines: algorithmic flops / bytes of ALL kernels over the timed step
        step_flops = sum(g["flops"] * g["launches"] for g in groups.values())
        step_bytes = sum(g["bytes"] * g["launches"] for g in groups.values())
        step_aggregate = {"algorithmic_tflop_per_s": step_flops / (ms_per_step * 1e-3) / 1e12,
                          "frac_of_tensor_peak_sustained": step_flops / (ms_per_step * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
                          "algorithmic_gb_per_s": step_bytes / (ms_per_step * 1e-3) / 1e9,
                          "frac_of_hbm_peak": step_bytes / (ms_per_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
                          "sum_of_kernel_ms": tot}
        # `roofline` = the WORST kernel of the step (lowest fraction of its bound among the kernels that hold >= 2 % of the
        # step), with the whole-step aggregate beside it; the per-kernel list is in `kernels`.
        cand = [k for k in kernels if k["share"] >= 0.02] or kernels
        top = min(cand, key=lambda k: k["frac"])
        roofline = {"kernel": top["name"], "selection": "worst fraction among kernels with >= 2 % of the step",
                    "launches_per_step": top["launches"], "ms_per_launch": top["ms"],
                    "share_of_step": top["share"], "bound": top["bound"], "achieved": top["achieved"],
                    "peak": top["peak"], "unit": top["unit"], "frac": top["frac"], "traffic": top["traffic"],
                    "traffic_source": traffic_note,
                    "peak_source": f"{peaks['src']} ({'bf16/fp16 dense burst; tf32 math runs at half that rate' if top['bound'] == 'tensor' else 'copy bandwidth'})",
                    "step": step_aggregate,
                    "kernels_at_or_above_half_of_bound": sum(1 for k in kernels if k["frac"] >= 0.5),
                    "kernels_total": len(kernels)}
        if "frac_of_tf32_rate" in top:
            roofline["frac_of_tf32_rate"] = top["frac_of_tf32_rate"]

    # ---- the rest of the contract, measured in the same run (every rank takes part: the parts hold barriers) -------
    modes, latency, configs = None, None, None
    if not args.no_extras:
        from tools import bench_parts
        model._destroy_ctx()  # release the headline context now (not whenever the cycle collector runs its destructor)
        del model
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        short = max(3, min(K, 10))
        modes = {"fp16": {"ms_per_step": ms_per_step, "value": value, "unit": UNIT}}
        for prec in ("tf32", "fp32"):
            r = bench_parts.crn_stream(args.model, B, prec, steps=short if prec == "tf32" else max(3, short // 2), dev=dev)
            modes[prec] = {"ms_per_step": r["ms_per_step"], "value": r["value"], "unit": UNIT, "steps": r["steps"],
                           "algorithmic_tflop_per_s": r["algorithmic_tflop_per_s"]}
        modes["note"] = ("same workload and streams; fp32 = exact CUDA-core arithmetic (parity anchor), tf32 = tcgen05 kind::tf32 "
                         "on fp32 storage, fp16 = fp16 operand storage with fp32 accumulation / statistics / state (headline)")
        latency = {}
        for nb in (1, 16):
            r = bench_parts.crn_stream(args.model, nb, args.precision, steps=20, latency_steps=300, dev=dev)
            latency[f"streams_{nb}"] = {k: r[k] for k in ("ms_per_step", "p50_chunk_latency_ms", "p99_chunk_latency_ms",
                                                          "latency_steps", "value")}
        latency["note"] = "device time of one chunk step (CUDA events), real-time deadline 100 ms per step"
        configs = {}
        r = bench_parts.crn_stream("student", args.student_streams, args.precision, steps=short, dev=dev)
        r["roofline"] = {"bound": "tensor", "achieved": r["algorithmic_tflop_per_s"], "peak": peaks["bf16_tflops"],
                         "unit": "TFLOP/s", "frac": r["algorithmic_tflop_per_s"] / peaks["bf16_tflops"],
                         "note": "whole-step algorithmic FLOPs (250.9 MFLOP per stream-chunk) over the step time"}
        r["workload"] = (f"distilled student CRN, {args.student_streams} concurrent streams per GPU "
                         "(BASELINE.json configs[2]: 16384 streams over 8 GPUs)")
        configs["student_streams"] = r
        r = bench_parts.fsn_utterances(args.fsn_streams, seconds=3.0, reps=1, precision="fp16", peak_tflops=peaks["bf16_tflops"],
                                       dev=dev)
        r["workload"] = f"FullSubNet, {args.fsn_streams} synthetic 3 s utterances per GPU, train=False chunk loop (BASELINE.json configs[3])"
        configs["fsn_3s"] = r
        r = bench_parts.train_step(batch=1, seconds=2.0, steps=10, warmup=3, precision="tf32", graph=True, dev=dev)
        r["workload"] = ("CRN_ELU compute_loss training step, one 2 s piece per rank, grad-accum 2, gradient all-reduce over the "
                         "ranks of this run (BASELINE.json configs[4])")
        configs["train_step"] = r
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args, args.cpu_streams, args.cpu_seconds)

    if rank == 0:
        launches = launches_per_chunk + 1  # + the io-descriptor kernel
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "tf32": "tf32", "fp16": "f16"}[args.precision], "data": "synthetic",
            "config": {"workload": f"CRN_ELU {args.model} batched streaming inference, {B} concurrent synthetic "
                                   f"streams per GPU, 3200-sample chunks at hop 1600 (BASELINE.json configs[1])",
                       "streams_per_gpu": B, "precision": args.precision,
                       "l2": f"inputs larger than L2: {RING}-hop input ring of {sig.numel() * 4 / 1e6:.0f} MB and a "
                             f"per-step working set of several GB, both > 126 MB L2"},
            "p99_chunk_latency_ms": lat[min(len(lat) - 1, int(0.99 * len(lat)))],
            "p50_chunk_latency_ms": lat[len(lat) // 2], "latency_steps": len(lat),
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches * K, "roofline": roofline, "step_aggregate": step_aggregate,
            "modes": modes, "latency": latency, "configs": configs, "stages": stages, "kernels": kernels,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
