"""GPU: the CRN streaming step at the stream counts where its launchers split the work, against the CPU oracle.

The persistent GRU kernels (gru_tc_persist.cu, gru_wave.cu) need every CTA of a launch resident at once, so a batch of
more than `tiles_per_wave` 128-stream m-tiles runs as several launches ("waves"), each over a slice of the batch with
its own offsets into the gate inputs, the state histories, the fp32 master state and the counters.  These tests run
batches that need two waves, a ragged last m-tile beside full ones, the tile edges 127 / 128 / 129 / 257 of the GRU and
the GEMMs, a batch smaller than the capacity of its context, and resets of a sub-range of the streams.  A launch guard
(torch.profiler over one eager chunk step) proves that each case ran the kernels it is meant to test."""
import collections
import re

import numpy as np
import pytest
import torch

from common import CONFIGS, TEACHER, TOL, make_model, make_oracle, oracle_stream_steps, si_sdr_db
from oracle import synth

pytestmark = pytest.mark.gpu

D, N = 8, 3   # distinct streams checked against the oracle, chunk steps (carried state from the second one on)
BM = 128      # streams per m-tile of the persistent GRU kernels (BM of gru_tc_persist.cu / gru_wave.cu)
REP_TOL = {"fp32": 2e-5, "tf32": 2e-3, "fp16": 2e-3}  # replica vs original, x peak (as in test_crn_gpu.py)


def tiles_per_wave(H, layers):
    """m-tiles per launch of a persistent GRU kernel: one CTA per SM, `layers` x H/32 CTAs per m-tile
    (launch_gru_tc_persist: one layer per launch; launch_gru_wave: one or two)."""
    return torch.cuda.get_device_properties(0).multi_processor_count // (layers * (H // 32))


def gru_waves(B, H, layers):
    mtiles = (B + BM - 1) // BM
    tpw = tiles_per_wave(H, layers)
    return (mtiles + tpw - 1) // tpw


def profiled_step(model, chunk):
    """One process_chunk under torch.profiler with graph replay off: (output, Counter of kernel name -> launches).
    Graph replay is switched back on afterwards."""
    from torch.profiler import ProfilerActivity, profile
    from speech_enhancement_mi_b200._native import check, lib
    model._ensure_ctx(chunk.shape[0], model._pick_device(chunk), keep_state=True)
    check(lib().se_crn_set_graph(model._ctx, 0), "se_crn_set_graph")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        y = model.process_chunk(chunk)
        torch.cuda.synchronize()
    check(lib().se_crn_set_graph(model._ctx, 1), "se_crn_set_graph")
    counts = collections.Counter(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
    counts = collections.Counter({k: n for k, n in counts.items() if not k.startswith(("Memcpy", "Memset"))})
    # without kernel records every "launched 0 times" below would pass vacuously
    assert counts, "the profiler recorded no kernel launches"
    return y, counts


def launches(counts, kernel):
    """Launches of `kernel` (any template arguments / namespace) in a profiled_step Counter."""
    pat = re.compile(r"\b" + re.escape(kernel) + r"\b")
    return sum(n for name, n in counts.items() if pat.search(name))


def short_counts(counts):
    """Kernel name without namespace and parameter list -> launches, for printing."""
    pat = re.compile(r"(\w+)(<[^()]*>)?\((?!anonymous)")
    out = collections.Counter()
    for name, n in counts.items():
        m = pat.search(name)
        out[m.group(1) + (m.group(2) or "") if m else name] += n
    return dict(sorted(out.items()))


def run_steps(model, chunks, profile_first=False):
    """process_chunk over `chunks` from the model's current state: outputs [B, 1600 * len(chunks)] (and the kernel
    counts of the first step if profile_first)."""
    outs, counts = [], None
    for n, c in enumerate(chunks):
        if n == 0 and profile_first:
            y, counts = profiled_step(model, c.cuda())
        else:
            y = model.process_chunk(c.cuda())
        outs.append(y.cpu().numpy())
    return np.concatenate(outs, axis=-1), counts


@pytest.fixture(scope="module")
def checked():
    """tag -> (chunks [D, 3, 3200] x N, oracle outputs [D, 1600 N], streams on the atan2 branch cut), computed once."""
    cache = {}

    def get(tag):
        if tag not in cache:
            oracle, _ = make_oracle(tag)
            mix, _ = synth.make_mixture(D, 1600 * (N + 1))
            chunks = [torch.from_numpy(mix[:, :, 1600 * n:1600 * n + 3200].copy()) for n in range(N)]
            want, on_cut = oracle_stream_steps(oracle, chunks, make_model(tag, "fp32"))
            cache[tag] = chunks, want, on_cut
        return cache[tag]
    return get


def placement(B, wave_start):
    """Which checked stream each of the B batch positions holds: shuffled replicas, with every checked stream in the
    first m-tile, in the first m-tile of the second wave and in the last (ragged) m-tile as far as those hold D."""
    idx = np.random.default_rng(B).permutation(B) % D
    idx[:D] = np.arange(D)
    if wave_start < B:
        k = min(D, B - wave_start)
        idx[wave_start:wave_start + k] = np.arange(k)
    k = min(D, B - (B - 1) // BM * BM)
    idx[B - k:] = np.arange(k)
    return idx


# (tag, precision, switch, (persistent GRU kernel, layers per launch) or None, B); "wave+k": k streams past the last full
# wave of that kernel on this device (9 x 128 + k for the teacher's H = 512, 18 x 128 + k for the student's two-layer
# H = 128 on 148 SMs)
WAVE_CASES = [
    ("crn_teacher", "fp16", None, ("gru_tc_persist_kernel", 1), "wave+1"),
    ("crn_teacher", "fp16", None, ("gru_tc_persist_kernel", 1), "wave+77"),
    ("crn_teacher", "fp16", ("SE_B200_GRU_WAVE", "2"), ("gru_wave_kernel", 1), "wave+77"),
    ("crn_student", "fp16", None, ("gru_wave_kernel", 2), "wave+1"),
    ("crn_student", "fp16", None, ("gru_wave_kernel", 2), "wave+77"),
]
EDGE_CASES = [("crn_teacher", p, None, ("gru_tc_persist_kernel", 1) if p == "fp16" else None, B)
              for p in ("fp16", "fp32", "tf32") for B in (127, 128, 129, 257)]


def case_id(case):
    tag, precision, switch, _, B = case
    return f"{tag[4:]}-{precision}-{'='.join(switch) if switch else 'default'}-{B if isinstance(B, str) else f'B{B}'}"


@pytest.mark.parametrize("case", WAVE_CASES + EDGE_CASES, ids=case_id)
def test_replicas_across_gru_waves_and_tile_edges_match_oracle(monkeypatch, checked, case):
    """D checked streams against the oracle over N chunk steps; a B-stream batch of their replicas (placement()) must
    reproduce the originals, and after it the same model -- its context now holds B streams -- run on the D streams
    again (B < capacity: the TMA maps built over the capacity, the counters of fewer m-tiles) must reproduce the fresh
    small context.  The first step of the batch is profiled: the persistent GRU kernel of the case must have run
    layers x waves times (>= 2 waves for the "wave+k" batches) and the other persistent form not at all."""
    tag, precision, switch, gru, B = case
    if switch:
        monkeypatch.setenv(*switch)
    chunks, want, on_cut = checked(tag)
    H = CONFIGS[tag][0]["hidden"]
    wave_start = tiles_per_wave(H, gru[1]) * BM if gru else None  # first stream of the second wave
    if isinstance(B, str):
        B = wave_start + int(B.split("+")[1])
    wave_start = min(wave_start or B, B)
    model = make_model(tag, precision)
    tol = TOL[precision]
    peak = max(1.0, float(np.abs(want).max()))
    keep = ~on_cut if precision == "fp32" else np.ones(D, dtype=bool)

    small, _ = run_steps(model, chunks)
    assert np.abs(small - want)[keep].max() < tol["wave_max_abs"] * peak
    assert np.abs(small - want).max() < TOL["fp16"]["wave_max_abs"] * peak  # streams on the cut: still the same signal
    assert si_sdr_db(small[keep][:, 1600:], want[keep][:, 1600:]) > tol["si_sdr_vs_ref_db"]

    idx = placement(B, wave_start)
    model.reset()
    big, counts = run_steps(model, [c[idx] for c in chunks], profile_first=True)
    persist = {k: launches(counts, k) for k in ("gru_tc_persist_kernel", "gru_wave_kernel")}
    print(f"\n{case_id(case)}: B = {B}, persistent GRU launches {persist}, all launches {short_counts(counts)}")
    if gru:
        waves = gru_waves(B, H, gru[1])
        if isinstance(case[4], str):
            assert waves >= 2, (B, waves)
        assert persist.pop(gru[0]) == (2 // gru[1]) * waves, (persist, waves)
    assert not any(persist.values()), persist
    rep_tol = REP_TOL[precision]
    assert np.abs(big - small[idx]).max() < rep_tol * peak
    assert np.abs(big - want[idx])[keep[idx]].max() < tol["wave_max_abs"] * peak

    assert model._ctx_capacity >= B > D
    model.reset()
    shrunk, _ = run_steps(model, chunks)
    assert np.abs(shrunk - small).max() < rep_tol * peak, "D streams on a context grown to B streams"


# (precision, switch): one per layout of the state table (crn.cu "state tables")
RESET_LAYOUTS = [
    ("fp32", None),                            # GEMM-path causal-conv buffers (PreBuf slabs of the pre-convolutions)
    ("tf32", None),
    ("fp16", None),                            # fused pre-convolutions: pre_state; GRU: hseq + fp32 master copy h32
    ("fp16", ("SE_B200_FRONT_MMA", "0")),      # per-layer tensor-core pre-convolutions: pre_h slabs
    ("fp16", ("SE_B200_PRECONV_TC", "0")),     # fp32 CUDA-core pre-convolutions: PreBuf slabs beside fp16 operands
]


@pytest.mark.parametrize("layout", RESET_LAYOUTS, ids=lambda l: f"{l[0]}-{'='.join(l[1]) if l[1] else 'default'}")
def test_partial_state_reset_touches_only_the_given_streams(monkeypatch, layout):
    """se_crn_state_reset(first, count) for a sub-range of the streams (a serving loop whose streams join and leave):
    300 teacher streams run two chunk steps, streams 100 .. 229 (across the m-tile borders at 128 and 256) are reset,
    and two more steps follow.  The reset streams must reproduce a run whose state was fully reset at that point, the
    others the uninterrupted continuation -- bit for bit, since all three runs have the same batch geometry on the same
    context.  Every entry of the state table (causal-conv buffers of every layout, GRU histories, the fp32 master copy
    of the GRU state, the overlap-add carry) must be cleared for exactly that range."""
    from speech_enhancement_mi_b200._native import check, lib
    precision, switch = layout
    if switch:
        monkeypatch.setenv(*switch)
    B, first, count = 300, 100, 130
    mix, _ = synth.make_mixture(B, 1600 * 5)
    chunks = [torch.from_numpy(mix[:, :, 1600 * n:1600 * n + 3200].copy()).cuda() for n in range(4)]
    model = make_model("crn_teacher", precision)

    def run(between):
        model.reset()
        for c in chunks[:2]:
            model.process_chunk(c)
        between()
        return np.concatenate([model.process_chunk(c).cpu().numpy() for c in chunks[2:]], axis=-1)

    y_cont = run(lambda: None)
    y_fresh = run(model.reset)
    y = run(lambda: check(lib().se_crn_state_reset(model._ctx, first, count, None), "se_crn_state_reset"))
    sel = np.zeros(B, dtype=bool)
    sel[first:first + count] = True
    print(f"\n{precision} {switch}: reset streams vs fresh {np.abs(y[sel] - y_fresh[sel]).max():.3e}, "
          f"others vs continuation {np.abs(y[~sel] - y_cont[~sel]).max():.3e}")
    assert np.array_equal(y[~sel], y_cont[~sel])
    assert np.array_equal(y[sel], y_fresh[sel])
    # the carried state matters for every reset stream, or this test would prove nothing
    peak = max(1.0, float(np.abs(y_cont).max()))
    assert np.abs(y_cont[sel] - y_fresh[sel]).max(axis=1).min() > 1e-3 * peak


def enc_tc_levels(mode, channels):
    """Encoder levels (Cin -> Cout, the first one from the 8-channel padded pre-convolution output, crn.cu enc_in) that
    SE_B200_ENC_TC=mode puts on enc_tc_kernel: 32 -> 64 unless 0, 16 -> 32 at 2 only."""
    levels = list(zip([8] + channels[:-1], channels))
    on = {0: [], 1: [(32, 64)], 2: [(16, 32), (32, 64)]}[mode]
    return sum(level in on for level in levels)


@pytest.mark.parametrize("mode", [None, "0", "2"], ids=lambda m: f"SE_B200_ENC_TC={m or 'unset'}")
def test_enc_tc_switch_is_read_per_context(monkeypatch, mode):
    """SE_B200_ENC_TC is read when a context is created, like every other kernel switch: the teacher's chunk step launches
    enc_tc_kernel once per level the setting selects (levels 8 -> 16 -> 32 -> 64 -> 128: none at 0, the 32 -> 64 level
    by default, 16 -> 32 too at 2) whatever contexts the process built before."""
    expected = enc_tc_levels(int(mode or 1), TEACHER["num_channels"])
    assert expected == {None: 1, "0": 0, "2": 2}[mode]
    # an fp16 context built first under another setting
    monkeypatch.setenv("SE_B200_ENC_TC", "0" if mode == "2" else "2")
    make_model("crn_teacher", "fp16").process_chunk(torch.zeros(2, 3, 3200, device="cuda"))
    if mode is None:
        monkeypatch.delenv("SE_B200_ENC_TC")
    else:
        monkeypatch.setenv("SE_B200_ENC_TC", mode)
    model = make_model("crn_teacher", "fp16")
    mix, _ = synth.make_mixture(2, 3200)
    _, counts = profiled_step(model, torch.from_numpy(mix).cuda())
    got = launches(counts, "enc_tc_kernel")
    print(f"\nSE_B200_ENC_TC={mode or 'unset'}: enc_tc_kernel launches per chunk step {got} (expected {expected})")
    assert got == expected
