"""GPU: the FullSubNet streaming step, se_fsn_process_chunk behind FullSubNet.process_chunk / process_chunk_host (one
3200-sample chunk per stream in, 1600 enhanced samples out; STFT, chunk network, mask, iSTFT and the overlap-add with
a carried half on the device in one CUDA-graph replay).

Chunks here are cut the way realtime_process(flag=False) cuts a signal: 1600 zeros in front, then the reference
segmentation.  Step n returns the first half of chunk n overlap-added with the second half of chunk n-1, so the outputs
of steps 1 .. N-1 joined are the realtime_process output with the 1600-sample front pad still in front."""
import collections

import numpy as np
import pytest
import torch

from common import FSN_FULL, FSN_SMALL, FSN_TOL_DB, FSN_TOL_REL, make_fsn, si_sdr_db
from oracle import crn_oracle, synth
from oracle.fsn_oracle import FSNOracle

pytestmark = pytest.mark.gpu

K, P = 3200, 1600
# Step vs realtime_process on the same streams, and a replica vs its original, x max(1, peak): both run the same
# kernels; the only expected difference is the order of the double-atomic CumLayerNorm sums (REP_TOL of
# test_fsn_stream_counts_gpu.py)
REP_TOL = 1e-5
CFGS = {"full": (FSN_FULL, 5), "small": (FSN_SMALL, 11),
        # fp16 operands need 64-unit sub-band tiles (the TMA / CTA-pair path of the LSTM steps)
        "small64": (dict(FSN_SMALL, sb_hidden=64), 11)}
D = 8  # distinct streams checked against the oracle


def chunks_of(mix):
    """[B, M, L] numpy -> [B, N, M, K] on the device: the front pad of realtime_process(flag=False), then the
    reference segmentation."""
    B, M, _ = mix.shape
    xp = torch.cat([torch.zeros(B, M, P), torch.from_numpy(mix)], dim=-1)
    seg, _ = crn_oracle.segmentation(xp, K)
    return seg.reshape(B, -1, M, K).cuda()


def stream(model, seg, L=None):
    """process_chunk over every chunk of seg [B, N, M, K] (each a strided view of seg); L: the signal's samples
    [B, L] as realtime_process returns them, else the raw step outputs [B, N * 1600]."""
    outs = [model.process_chunk(seg[:, n]).clone() for n in range(seg.shape[1])]
    if L is None:
        return torch.cat(outs, dim=-1).cpu().numpy()
    return torch.cat(outs[1:], dim=-1)[:, P:P + L].cpu().numpy()


def peak_of(x):
    return max(1.0, float(np.abs(x).max()))


@pytest.mark.parametrize("tag,precision", [("small", "tf32"), ("small", "3xtf32"), ("small64", "fp16"),
                                           ("full", "tf32"), ("full", "fp16")])
def test_steps_equal_realtime_process(tag, precision):
    cfg, seed = CFGS[tag]
    B, L = 3, 8000
    mix, _ = synth.make_mixture(B, L)
    model = make_fsn(cfg, seed, precision=precision)
    ref = model.realtime_process(torch.from_numpy(mix).cuda(), None, flag=False, train=False).cpu().numpy()
    model.reset_state(B)
    got = stream(model, chunks_of(mix), L)
    err = float(np.abs(got - ref).max())
    print(f"{tag} {precision}: process_chunk steps vs realtime_process max-abs {err:.3e} (peak {peak_of(ref):.3g})")
    assert err <= REP_TOL * peak_of(ref)


def assert_matches_oracle(got, want, what):
    peak = peak_of(want)
    err = float(np.abs(got - want).max())
    db = min(si_sdr_db(g, w) for g, w in zip(got, want))
    print(f"{what}: max-abs {err:.3e} (peak {peak:.3g}), worst stream SI-SDR {db:.1f} dB")
    assert err < FSN_TOL_REL * peak, (what, err)
    assert db > FSN_TOL_DB, (what, db)


@pytest.fixture(scope="module")
def checked():
    """(tag, streams, samples) -> (mixture, oracle realtime_process output), computed once."""
    cache = {}

    def get(tag, B, L):
        if (tag, B, L) not in cache:
            cfg, seed = CFGS[tag]
            mix, _ = synth.make_mixture(B, L)
            with torch.no_grad():
                want, _ = FSNOracle(synth.make_fsn_weights(seed=seed, **cfg), **cfg).realtime_process(
                    torch.from_numpy(mix))
            cache[tag, B, L] = mix, want.numpy()
        return cache[tag, B, L]
    return get


# 1 s = 14 chunks; 9 s = 94 chunks, past the CumLayerNorm step cap of 80 (fullsubnet.py:184-201)
@pytest.mark.parametrize("tag,precision,B,L", [("small", "tf32", D, 16000), ("small64", "fp16", D, 16000),
                                               ("small", "tf32", 2, 9 * 16000)])
def test_steps_match_oracle(checked, tag, precision, B, L):
    mix, want = checked(tag, B, L)
    seg = chunks_of(mix)
    assert seg.shape[1] >= (82 if L > 16000 else 12)
    got = stream(make_fsn(*CFGS[tag], precision=precision), seg, L)
    assert_matches_oracle(got, want, f"{tag} {precision} {B} x {seg.shape[1]} chunks")
    if L > 16000:
        assert_matches_oracle(got[:, -16000:], want[:, -16000:], f"{tag} {precision} last second")


def test_serving_batch_replicas_and_smaller_batch_leave_other_streams_alone(checked):
    """300 replicas of the D oracle-checked streams on a context of 512: every replica reproduces its original.  A second
    model runs the same streams, but a few steps in the middle with only the first Bs streams: those continue, and the
    others, continued afterwards, must produce exactly what they produce without the pause."""
    mix, want = checked("small", D, 16000)
    L = mix.shape[-1]
    peak = peak_of(want)
    small = stream(make_fsn(*CFGS["small"]), chunks_of(mix), L)
    assert_matches_oracle(small, want, f"{D} streams")

    Bb, Bs, h, j = 300, 100, 5, 3
    idx = np.random.default_rng(Bb).permutation(Bb) % D
    idx[:D] = np.arange(D)
    idx[Bb - D:] = np.arange(D)
    seg = chunks_of(mix[idx])
    N = seg.shape[1]
    model = make_fsn(*CFGS["small"], max_streams=512)
    ref = stream(model, seg)  # [Bb, N * P]
    assert model._ctx_capacity == 512
    big = ref.reshape(Bb, N, P)[:, 1:].reshape(Bb, -1)[:, P:P + L]
    spread = float(np.abs(big - small[idx]).max())
    print(f"{Bb} replicas on a context of 512 vs the {D} originals: max-abs {spread:.3e}")
    assert spread < REP_TOL * peak
    assert np.abs(big - want[idx]).max() < FSN_TOL_REL * peak

    # chunks 0..h-1 for all streams; h..h+j-1 for streams [0, Bs) only; then all streams, each at its own next chunk
    model = make_fsn(*CFGS["small"], max_streams=512)
    outs = [[] for _ in range(Bb)]
    rows = torch.arange(Bb, device=seg.device)
    pos = torch.zeros(Bb, dtype=torch.long, device=seg.device)

    def step(B):
        y = model.process_chunk(seg[rows[:B], pos[:B]]).cpu().numpy()
        for r in range(B):
            outs[r].append(y[r])
        pos[:B] += 1

    for _ in range(h):
        step(Bb)
    for _ in range(j):
        step(Bs)
    for _ in range(N - h - j):
        step(Bb)
    for r in range(Bb):
        got = np.concatenate(outs[r])
        assert got.shape[0] == (N if r < Bs else N - j) * P
        if r < Bs:  # steps of two batch sizes: the CumLayerNorm sums may be added in another order
            assert np.abs(got - ref[r]).max() < REP_TOL * peak, r
        else:
            assert np.array_equal(got, ref[r, :got.shape[0]]), r


def test_partial_reset_clears_state_and_carry_of_the_given_streams_only():
    """se_fsn_reset_state(first, count) between two steps on a context larger than the batch.  The continuation starts
    with a chunk of zeros: its enhanced spectrum is exactly zero, so that step returns the carried half / 2 -- zero for a
    reset stream.  Reset streams must reproduce a fresh model bit for bit, the others the uninterrupted run."""
    from speech_enhancement_mi_b200._native import check, lib
    B, cap, first, count, h = 6, 16, 1, 3, 4
    mix, _ = synth.make_mixture(B, 1600 * 9)
    seg = chunks_of(mix)
    cont = torch.cat([torch.zeros_like(seg[:, :1]), seg[:, h:]], dim=1)

    def run(between):
        m = make_fsn(*CFGS["small"], max_streams=cap)
        if between is not None:
            stream(m, seg[:, :h])
            between(m)
        return stream(m, cont)

    y_cont = run(lambda m: None)
    y_fresh = run(None)
    y = run(lambda m: check(lib().se_fsn_reset_state(m._ctx, first, count, None), "se_fsn_reset_state"))
    sel = np.zeros(B, dtype=bool)
    sel[first:first + count] = True
    assert np.array_equal(y[~sel], y_cont[~sel])
    assert np.array_equal(y[sel], y_fresh[sel])
    # not vacuous: the carry and the rest of the state both change the output of every stream
    assert np.all(y_fresh[:, :P] == 0)
    assert np.abs(y_cont[:, :P]).max(axis=1).min() > 1e-4
    assert np.abs(y_cont[:, P:] - y_fresh[:, P:]).max(axis=1).min() > 1e-4


def test_strided_input_and_output_are_bitwise_equal_to_contiguous():
    B, M = 4, 3
    mix, _ = synth.make_mixture(B, 1600 * 5)
    seg = chunks_of(mix)
    ma, mb = make_fsn(*CFGS["small"]), make_fsn(*CFGS["small"])
    for n in range(seg.shape[1]):
        want = ma.process_chunk(seg[:, n].contiguous()).cpu().numpy()
        # stream and microphone strides larger than contiguous, first sample at an odd offset (no 16-byte loads)
        buf = torch.full((B, M + 2, K + 37), float("nan"), device="cuda")
        x = buf[:, 1:1 + M, 5:5 + K]
        x.copy_(seg[:, n])
        obuf = torch.full((B, P + 100), float("nan"), device="cuda")
        out = obuf[:, 50:50 + P]
        assert x.stride() == ((M + 2) * (K + 37), K + 37, 1) and out.stride() == (P + 100, 1)
        assert mb.process_chunk(x, out) is out
        assert np.array_equal(out.cpu().numpy(), want), n
        assert torch.isnan(obuf[:, :50]).all() and torch.isnan(obuf[:, 50 + P:]).all()


def test_pipelined_host_steps_equal_device_steps():
    """process_chunk_host (pinned host buffers, copies on side streams, double-buffered staging) returns exactly what
    process_chunk returns for the same chunks, also when many steps are in flight."""
    model = make_fsn(*CFGS["small"])
    B, N = 4, 9
    mix, _ = synth.make_mixture(B, 1600 * (N + 1))
    chunks = [torch.from_numpy(mix[:, :, 1600 * n:1600 * n + 3200].copy()) for n in range(N)]
    want = [model.process_chunk(c.cuda()).cpu().numpy() for c in chunks]
    model.reset_state(B)
    pinned = [c.pin_memory() for c in chunks]
    outs = [torch.empty((B, 1600), dtype=torch.float32).pin_memory() for _ in range(N)]
    events = [model.process_chunk_host(pinned[n], outs[n]) for n in range(N)]  # no synchronisation in between
    for n in range(N):
        events[n].synchronize()
        assert np.array_equal(outs[n].numpy(), want[n]), n


def test_interleaved_paths_do_not_leak_into_each_other():
    """process_chunk, realtime_process and forward on ONE context: each call equals the same call (or sequence) on a
    fresh model.  realtime_process(flag=False) resets the streams it runs, carry included."""
    B = 3
    mix, _ = synth.make_mixture(B, 8000)
    x = torch.from_numpy(mix).cuda()
    seg = chunks_of(mix)
    spec = torch.randn(B, 6, 201, 21, generator=torch.Generator().manual_seed(3)).cuda()
    fresh = lambda: make_fsn(*CFGS["small"])  # noqa: E731
    m = fresh()
    stream(m, seg[:, :3])
    got = m.realtime_process(x, None, flag=False, train=False).cpu().numpy()
    assert np.array_equal(got, fresh().realtime_process(x, None, flag=False, train=False).cpu().numpy())
    m.reset_state(B)
    assert np.array_equal(m.forward(spec).cpu().numpy(), fresh().forward(spec).cpu().numpy())
    m.reset_state(B)
    assert np.array_equal(stream(m, seg), stream(fresh(), seg))


def kernel_launches(fn):
    """Counter of the CUDA kernels fn launches (graph replays included) under torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    names = [n for n in names if not n.startswith(("Memcpy", "Memset"))]
    assert names, "the profiler recorded no kernel launches"
    counts = collections.Counter()
    for n in names:
        for k in ("gemm_tc_kernel", "stft_features_kernel", "mask_istft_kernel"):
            counts[k] += k in n
    return counts


@pytest.mark.parametrize("tag,precision", [("small", "tf32"), ("small64", "fp16")])
def test_step_launches_the_network_of_forward_and_one_stft_and_istft(tag, precision):
    B = 5
    model = make_fsn(*CFGS[tag], precision=precision)
    spec = torch.randn(B, 6, 201, 21, generator=torch.Generator().manual_seed(B)).cuda()
    chunk = torch.randn(B, 3, K, generator=torch.Generator().manual_seed(1)).cuda()
    model.forward(spec)
    model.process_chunk(chunk)  # both graphs captured outside the profiled window
    fwd = kernel_launches(lambda: model.forward(spec))
    step = kernel_launches(lambda: model.process_chunk(chunk))
    print(f"{tag} {precision}: forward {dict(fwd)}, process_chunk {dict(step)}")
    assert fwd["gemm_tc_kernel"] > 0 and step["gemm_tc_kernel"] == fwd["gemm_tc_kernel"]
    assert step["stft_features_kernel"] == 1 and step["mask_istft_kernel"] == 1


def test_errors():
    from speech_enhancement_mi_b200._native import lib
    model = make_fsn(*CFGS["small"])
    with pytest.raises(ValueError):
        model.process_chunk(torch.zeros(2, 3, K))  # CPU tensor
    with pytest.raises(ValueError):
        model.process_chunk(torch.zeros(2, 2, K, device="cuda"))
    with pytest.raises(ValueError):
        model.process_chunk(torch.zeros(2, 3, K - 1, device="cuda"))
    model.process_chunk(torch.zeros(2, 3, K, device="cuda"))
    with pytest.raises(RuntimeError, match="stream state would be lost"):
        model.process_chunk(torch.zeros(3, 3, K, device="cuda"))
    x = torch.zeros(3, 3, K, device="cuda")
    out = torch.zeros(3, P, device="cuda")
    cap = model._ctx_capacity
    assert cap == 2
    rc = lib().se_fsn_process_chunk(model._ctx, x.data_ptr(), 3 * K, K, out.data_ptr(), P, cap + 1, None)
    assert rc != 0 and b"max_streams" in lib().se_last_error()
    assert lib().se_fsn_process_chunk(model._ctx, None, 3 * K, K, out.data_ptr(), P, 1, None) != 0
    assert lib().se_fsn_process_chunk(model._ctx, x.data_ptr(), 3 * K, K, out.data_ptr(), P, 0, None) == 0
