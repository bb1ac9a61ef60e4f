"""GPU: the FullSubNet chunk loop (fsn.cu on the LSTM step GEMMs of gemm_tc.cu) at serving batch sizes, against the CPU
oracle.

Every LSTM step is one persistent gemm_tc_kernel launch (grid = min(tiles, SMs), tiles = m-tiles x n-tiles) over M = B
rows in the full band and M = B x 201 rows in the sub band, one row per (stream, bin) sequence, in 128-row m-tiles.  The
batches here are large enough that every CTA takes several tiles (the TMEM accumulator hand-off between tiles), that the
CTA-pair form walks many super-tiles and masks the second m-tile of an odd last pair, and that a ragged full-band tile
sits beside full ones.  Each kernel form the switches select runs: gather (template argument 0), TMA (1) and TMA with CTA
pairs (2); a launch guard (torch.profiler over one chunk) proves it.  Also covered: more than one block of the
CumLayerNorm update, a batch smaller than the capacity of its context, 94-chunk streams (past the CumLayerNorm step cap
of 80), the grid-stride loops of the elementwise kernels, and the realtime_process scratch reused across calls with
different stream and chunk counts.  (Resets of a sub-range of the streams on a context larger than the batch:
test_fsn_gpu.py::test_partial_state_reset_touches_only_the_given_streams.)"""
import collections
import os
import re

import numpy as np
import pytest
import torch

from common import FSN_FULL, FSN_SMALL, FSN_TOL_DB, FSN_TOL_REL, GOLDEN, make_fsn, si_sdr_db
from oracle import synth
from oracle.fsn_oracle import FSNOracle, unfold

pytestmark = pytest.mark.gpu

D = 8                  # distinct streams checked against the oracle
L1, L2 = 6400, 3200    # samples: 8 chunks from a reset state (front pad), then 4 more as a flag=True continuation
BM = 128               # rows per m-tile of gemm_tc_kernel
F, T = 201, 21         # bins = sub-band sequences per stream; frames per chunk = LSTM steps per layer and chunk
CFGS = {"full": (FSN_FULL, 5), "small": (FSN_SMALL, 11), "small64": (dict(FSN_SMALL, sb_hidden=64), 11)}
# replica vs original, x max(1, peak).  Streams are independent, but the per-stream CumLayerNorm sums are double atomics
# (fsn_mag_kernel, fsn_scale_fb_kernel, the EPI_RELU_STATS epilogue) whose order and partition depend on where the
# stream sits in the batch.  Measured on one B200 (1000 W power limit): 0, bit-identical, in every case below.  1e-5
# leaves room for a norm mean whose double sum rounds to the neighbouring float; stale norms of the streams past the
# first 128 give 0.10.
REP_TOL = 1e-5


def oracle_for(tag):
    cfg, seed = CFGS[tag]
    return FSNOracle(synth.make_fsn_weights(seed=seed, **cfg), **cfg)


def run_pair(model, mix1, mix2):
    """realtime_process from a reset state, then a flag=True continuation: the two outputs side by side [B, L1 + L2]."""
    a = model.realtime_process(torch.from_numpy(mix1).cuda(), None, flag=False, train=False).cpu().numpy()
    b = model.realtime_process(torch.from_numpy(mix2).cuda(), None, flag=True, train=False).cpu().numpy()
    return np.concatenate([a, b], axis=-1)


def assert_matches_oracle(got, want, what="", sdr=True):
    """The stated tolerances: max-abs error < 2e-2 x max(1, peak) and (sdr) >= 40 dB SI-SDR on every stream."""
    peak = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(got - want).max())
    db = min(si_sdr_db(g, w) for g, w in zip(got, want))
    print(f"{what}: max-abs {err:.3e} (peak {peak:.3g}), worst stream SI-SDR {db:.1f} dB")
    assert err < FSN_TOL_REL * peak, (what, err)
    assert not sdr or db > FSN_TOL_DB, (what, db)


@pytest.fixture(scope="module")
def checked():
    """tag -> (mixture [D, 3, L1], continuation [D, 3, L2], oracle outputs [D, L1 + L2]), computed once."""
    cache = {}

    def get(tag):
        if tag not in cache:
            mix1, _ = synth.make_mixture(D, L1)
            mix2, _ = synth.make_mixture(D, L2, first_stream=100)
            o = oracle_for(tag)
            with torch.no_grad():
                w1, _ = o.realtime_process(torch.from_numpy(mix1))
                w2, _ = o.realtime_process(torch.from_numpy(mix2), flag=True)
            cache[tag] = mix1, mix2, np.concatenate([w1.numpy(), w2.numpy()], axis=-1)
        return cache[tag]
    return get


def lstm_geometry(cfg, B):
    """Tiles of the LSTM step GEMMs by the rules of fsn.cu build_lstm (64 hidden units x 4 gates = 256 columns per tile
    where the hidden size allows it, 32 x 4 with SE_B200_FSN_WIDE=0) and gemm_tc.cu (128-row m-tiles, grid = min(tiles,
    SMs); a CTA pair takes a super-tile of two m-tiles, grid = min(super-tiles, SMs / 2) clusters)."""
    wide = int(os.environ.get("SE_B200_FSN_WIDE", "1")) != 0

    def bn(H):
        return 256 if H % 64 == 0 and wide else 128

    g = dict(sms=torch.cuda.get_device_properties(0).multi_processor_count,
             fb_mt=-(-B // BM), fb_nt=4 * cfg["fb_hidden"] // bn(cfg["fb_hidden"]),
             sb_mt=-(-B * F // BM), sb_nt=4 * cfg["sb_hidden"] // bn(cfg["sb_hidden"]),
             norm_blocks=-(-B // 128))
    g["sb_tiles"] = g["sb_mt"] * g["sb_nt"]
    g["sb_super"] = -(-g["sb_mt"] // 2) * g["sb_nt"]
    return g


GEMM = re.compile(r"gemm_tc_kernel<([^<>]*)>")


def profiled_forward(model, B):
    """One forward chunk of B streams under torch.profiler (the chunk runs as the context's CUDA graph):
    Counter of gemm_tc_kernel launches by their last template argument (0 gather, 1 TMA, 2 TMA + CTA pair)."""
    from torch.profiler import ProfilerActivity, profile
    x = torch.randn(B, 2 * model.num_mics, F, T, generator=torch.Generator().manual_seed(B)).cuda()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        model.forward(x)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    names = [n for n in names if not n.startswith(("Memcpy", "Memset"))]
    # without kernel records every "launched 0 times" below would pass vacuously
    assert names, "the profiler recorded no kernel launches"
    forms = collections.Counter()
    for n in names:
        m = GEMM.search(n)
        if m:
            forms[int(m.group(1).split(",")[-1])] += 1
    return forms


# (tag, precision, switches, B, forms of the sub-band LSTM steps of layer 0 / layer 1: 0 gather, 1 TMA, 2 TMA + pair)
CASES = [
    # 201 m-tiles, odd and all full: the second CTA of the last pair is fully masked
    ("full", "fp16", {}, 128, (2, 2)),
    # ragged full-band tile beside a full one, 2 CumLayerNorm blocks; 203 (odd) / 404 sub-band m-tiles, ragged last one
    ("full", "fp16", {}, 129, (2, 2)),
    ("full", "fp16", {}, 257, (2, 2)),
    ("full", "fp16", {}, 256, (2, 2)),  # the benchmark shape (bench.py configs[3])
    # 128-column tiles: layer 0 (K = 64 + 384 = 448 < 576) stays single-CTA TMA, layer 1 (K = 768) is a pair
    ("full", "fp16", {"SE_B200_FSN_WIDE": "0"}, 129, (1, 2)),
    ("full", "fp16", {"SE_B200_TMA_PAIR": "0"}, 129, (1, 1)),
    # forced pairs: with 128-column tiles layer 0 becomes a pair too
    ("full", "fp16", {"SE_B200_FSN_WIDE": "0", "SE_B200_TMA_PAIR": "2"}, 129, (2, 2)),
    ("full", "fp16", {"SE_B200_FSN_TMA": "0"}, 129, (0, 0)),  # fp16 cp.async gather form
    *[("full", "tf32", {}, B, (0, 0)) for B in (127, 128, 129, 257)],
    ("small64", "fp16", {}, 129, (2, 2)),  # the smallest fp16-legal sub-band size
]


def case_id(case):
    tag, precision, env, B, _ = case
    sw = ",".join(f"{k[8:]}={v}" for k, v in env.items()) or "default"
    return f"{tag}-{precision}-{sw}-B{B}"


def placement(B):
    """Which checked stream each of the B batch positions holds: shuffled replicas, with the D originals in order at the
    start (first m-tiles) and at the end (ragged last m-tiles)."""
    idx = np.random.default_rng(B).permutation(B) % D
    idx[:D] = np.arange(D)
    idx[B - D:] = np.arange(D)
    return idx


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_replicas_at_serving_batch_sizes_match_oracle(monkeypatch, checked, case):
    """D checked streams against the oracle; a B-stream batch of their replicas (placement()) must reproduce the
    originals at every batch position, and after it the same model -- its context now holds B streams -- run on the D
    streams again must reproduce the fresh small context.  One forward chunk of the batch is profiled: the LSTM step
    launches must be in the forms of the case."""
    tag, precision, env, B, forms = case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    cfg, seed = CFGS[tag]
    mix1, mix2, want = checked(tag)
    peak = max(1.0, float(np.abs(want).max()))
    model = make_fsn(cfg, seed, precision=precision)

    small = run_pair(model, mix1, mix2)
    assert_matches_oracle(small, want, f"{case_id(case)}: {D} streams vs oracle")

    g = lstm_geometry(cfg, B)
    print(f"{case_id(case)}: {g}")
    assert g["sb_tiles"] > g["sms"] and g["sb_super"] > g["sms"] // 2, g  # every CTA / cluster takes several tiles
    if B == BM:
        assert B * F % BM == 0 and g["sb_mt"] % 2 == 1, g  # all m-tiles full; the last pair's second CTA has no rows
    if B % BM:
        assert B * F % BM != 0  # ragged last sub-band m-tile
    if B > BM and B % BM:
        assert g["fb_mt"] >= 2 and g["norm_blocks"] >= 2, g  # ragged full-band tile beside full ones

    idx = placement(B)
    big = run_pair(model, mix1[idx], mix2[idx])
    spread = float(np.abs(big - small[idx]).max())
    print(f"{case_id(case)}: replicas vs originals max-abs {spread:.3e}")
    assert spread < REP_TOL * peak
    assert np.abs(big - want[idx]).max() < FSN_TOL_REL * peak

    got = profiled_forward(model, B)
    expected = {0: 2 * T + 2 + T * forms.count(0), 1: T * forms.count(1), 2: T * forms.count(2)}
    print(f"{case_id(case)}: gemm_tc_kernel launches per chunk by form {dict(got)}, expected {expected}")
    assert {k: got.get(k, 0) for k in expected} == expected
    assert sum(got.values()) == sum(expected.values())

    assert model._ctx_capacity >= B > D
    shrunk = run_pair(model, mix1, mix2)
    assert np.abs(shrunk - small).max() < REP_TOL * peak, "D streams on a context grown to B streams"


# realtime_process calls (streams, samples, train) on ONE model; the first five have no max_streams
SCRATCH_SEQS = [
    (None, [(4, 4000, False), (1, 48000, False), (4, 4000, False)]),  # 6 / 34 / 6 chunks: more streams, fewer rows
    (None, [(4, 4000, True), (1, 48000, True), (4, 4000, True)]),
    (None, [(4, 4000, True), (1, 48000, False), (4, 4000, True)]),
    (None, [(4, 4000, False), (1, 48000, True), (4, 4000, False)]),
    (8, [(4, 4000, False), (1, 48000, False), (8, 1600, False)]),
    # train=True with fewer rows (6) than the capacity (8), then the chunk loop over all 8 streams (4 chunks)
    (8, [(1, 48000, False), (1, 4000, True), (8, 1600, False)]),
]


@pytest.mark.parametrize("max_streams,calls", SCRATCH_SEQS,
                         ids=lambda v: "cap" + str(v) if not isinstance(v, list) else
                         "-".join(f"{b}x{n}{'T' if t else 'F'}" for b, n, t in v))
def test_scratch_reused_across_calls_of_other_stream_and_chunk_counts(max_streams, calls):
    """se_fsn_realtime_process keeps its scratch across calls and grows it on demand.  A call with more streams but fewer
    chunks than an earlier one (a predict loop over files of mixed counts and lengths) must find scratch large enough for
    its streams: every output of one model over the sequence equals, bit for bit, the same call on a fresh model of the
    same capacity."""
    cfg, seed = CFGS["small"]
    model = make_fsn(cfg, seed, max_streams=max_streams)
    cap = max([b for b, _, _ in calls] + [max_streams or 0])
    ctx = None
    for n, (B, L, train) in enumerate(calls):
        mix, _ = synth.make_mixture(B, L, first_stream=10 * n)
        x = torch.from_numpy(mix).cuda()
        y = model.realtime_process(x, None, flag=False, train=train).cpu().numpy()
        assert model._ctx_capacity == cap and (ctx is None or model._ctx.value == ctx)  # one context, its scratch kept
        ctx = model._ctx.value
        fresh = make_fsn(cfg, seed, max_streams=cap)
        y_fresh = fresh.realtime_process(x, None, flag=False, train=train).cpu().numpy()
        del fresh
        assert np.array_equal(y, y_fresh), (n, B, L, train, float(np.abs(y - y_fresh).max()))


@pytest.mark.parametrize("tag,precision", [("small", "tf32"), ("small64", "fp16")])
def test_long_stream_past_the_norm_step_cap_matches_oracle(tag, precision):
    """Two 9 s streams = 94 chunks: the CumLayerNorm step saturates at 80 (fullsubnet.py:184-201) and the LSTM state is
    carried through every chunk.  Against the oracle on the whole signal and on its last second."""
    from speech_enhancement_mi_b200._native import chunk_grid
    L = 9 * 16000
    assert chunk_grid(L + 1600, 3200)[1] > 80
    cfg, seed = CFGS[tag]
    mix, _ = synth.make_mixture(2, L)
    x = torch.from_numpy(mix)
    with torch.no_grad():
        want, _ = oracle_for(tag).realtime_process(x)
    want = want.numpy()
    got = make_fsn(cfg, seed, precision=precision).realtime_process(x.cuda(), None, flag=False, train=False)
    got = got.cpu().numpy()
    assert_matches_oracle(got, want, f"{tag} {precision} 9 s")
    assert_matches_oracle(got[:, -16000:], want[:, -16000:], f"{tag} {precision} last second")


def test_unfold_grid_stride_loop_bit_exact():
    """se_unfold's grid is capped at 148 x 32 blocks of 256 threads: 4.2 M outputs take several trips of its loop."""
    from speech_enhancement_mi_b200.fullsubnet import BaseModel
    x = torch.randn(16, 2, 201, 21, generator=torch.Generator().manual_seed(0))
    want = unfold(x, 15).numpy()
    assert want.size > 148 * 32 * 256 * 3
    assert np.array_equal(BaseModel.unfold(x.cuda(), 15).cpu().numpy(), want)


def test_stft_trans_grid_stride_loop_matches_oracle():
    """se_fsn_planes' grid is capped at 148 x 32 blocks of 256 threads: 128 x 3 chunks are 1.6 M spectrum values."""
    R = 128
    mix, _ = synth.make_mixture(R, 3200)
    x = torch.from_numpy(mix)
    assert R * 3 * F * T > 148 * 32 * 256
    got = make_fsn(*CFGS["small"]).stft_trans(x.cuda()).cpu()
    want = oracle_for("small").stft_trans(x)
    assert got.shape == want.shape
    assert (got - want).abs().max() < 1e-6 * want.abs().max()


def test_whole_utterance_train_true_replicated_matches_reference():
    """train=True (all chunks as one forward) at 129 streams: the two streams of the fsn_small_whole fixture (the
    unmodified reference; the oracle has no train=True form) replicated, a ragged full-band tile and 774 chunk-rows
    through the grid-stride loop of se_fsn_apply_mask.  Every replica must reproduce the fixture, and the two-stream run
    of the same model."""
    z = np.load(os.path.join(GOLDEN, "fsn_small_whole.npz"))
    cfg, seed = CFGS["small"]
    n, L = int(z["meta"][1]), int(z["meta"][2])
    mix, _ = synth.make_mixture(n, L)
    mix2, _ = synth.make_mixture(n, L // 2, first_stream=100)
    model = make_fsn(cfg, seed)
    small = [model.realtime_process(torch.from_numpy(m).cuda(), None, flag=f, train=True).cpu().numpy()
             for m, f in ((mix, False), (mix2, True))]
    idx = np.arange(129) % n
    big = [model.realtime_process(torch.from_numpy(m[idx]).cuda(), None, flag=f, train=True).cpu().numpy()
           for m, f in ((mix, False), (mix2, True))]
    assert model._ctx_capacity == 129
    for key, s, b in (("out", small[0], big[0]), ("out_cont", small[1], big[1])):
        ref = z[key][idx]
        peak = max(1.0, float(np.abs(ref).max()))
        print(f"train=True {key}: replicas vs two-stream run {np.abs(b - s[idx]).max():.3e}")
        assert np.abs(b - s[idx]).max() < REP_TOL * peak
        # the continuation is held to the max-abs tolerance only, as in test_fsn_gpu.py
        assert_matches_oracle(b, ref, f"train=True {key} vs reference", sdr=key == "out")
