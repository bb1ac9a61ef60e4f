"""GPU parity tests proper: the CUDA path (through the C-ABI behind the reference's model API) against the oracle, the
committed reference fixtures, and size-independent properties.  Tolerances are the stated ones in tests/common.py."""
import numpy as np
import pytest
import torch

from common import CONFIGS, TOL, load_golden, make_model, make_oracle, oracle_stream_steps, rel_err, si_sdr_db
from oracle import crn_oracle, synth

pytestmark = pytest.mark.gpu


def ramp(L):
    r = torch.arange(1, L + 1, dtype=torch.float32).reshape(1, 1, L).repeat(2, 3, 1)
    r[1] += 100000
    r[:, 1] += 0.25
    r[:, 2] += 0.5
    return r


@pytest.mark.parametrize("L", [1, 1599, 1600, 1601, 3199, 3200, 3201, 4000, 9600])
def test_segmentation_over_add_bit_exact(L):
    """Integer index work: bit-exact against the reference fixtures / oracle, incl. the ragged edge lengths."""
    from speech_enhancement_mi_b200 import utility
    g = load_golden("framing")
    x = ramp(L)
    seg, gap = utility.segmentation(x.cuda(), 3200)
    seg_o, gap_o = crn_oracle.segmentation(x, 3200)
    assert gap == gap_o
    assert np.array_equal(seg.cpu().numpy(), seg_o.numpy())
    N = seg.shape[0] // 2
    if N >= 2:
        chunks = seg[:, 0].reshape(2, N, 3200)
        ola = utility.over_add(chunks, gap).cpu().numpy()
        ola_o = crn_oracle.over_add(seg_o[:, 0].reshape(2, N, 3200), gap_o).numpy()
        assert np.array_equal(ola, ola_o)
        if L in (1601, 4000):
            assert np.array_equal(seg.cpu().numpy(), g[f"seg_{L}"])
            assert np.array_equal(ola, g[f"ola_{L}"])


def test_stft_istft_against_reference_fixture():
    g = load_golden("crn_teacher")
    model = make_model("crn_small")
    oracle, _ = make_oracle("crn_small")
    B, L = int(g["meta"][1]), int(g["meta"][2])
    mix, _ = synth.make_mixture(B, L)
    x = torch.cat([torch.zeros(B, 3, 1600), torch.from_numpy(mix)], dim=-1)
    seg, _ = crn_oracle.segmentation(x, 3200)
    N = seg.shape[0] // B
    spec = model.stft_trans(seg.cuda()).cpu().numpy()
    assert spec.shape == (B * N, 3, 201, 21, 2)
    want = g["spec_chunk1"]
    got = spec.reshape(B, N, 3, 201, 21, 2)[:, 1]
    assert rel_err(got, want) < 1e-5  # framing bit-exact, fp32 FFT
    ist = model.istft_trans(torch.from_numpy(g["fwd_chunk1"]).cuda()).cpu().numpy()
    assert rel_err(ist, g["istft_chunk1"]) < 1e-5
    # identity: iSTFT(STFT(chunk)) == chunk (mask = 1), a size-independent property
    chunk = seg[:4]
    back = model.istft_trans(model.stft_trans(chunk.cuda())[:, 0].contiguous()).cpu().numpy()
    assert np.abs(back - chunk[:, 0].numpy()).max() < 1e-5
    # zero chunk (empty input edge case)
    z = model.stft_trans(torch.zeros(1, 3, 3200).cuda()).cpu().numpy()
    assert np.all(z == 0)


@pytest.mark.parametrize("precision", ["fp32", "tf32", "fp16"])
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_forward_chunk_matches_reference(tag, precision):
    g = load_golden(tag)
    tol = TOL[precision]
    model = make_model(tag, precision)
    out = model.forward(torch.from_numpy(g["spec_chunk1"]).cuda())
    out = out[0] if isinstance(out, tuple) else out
    assert rel_err(out.cpu().numpy(), g["fwd_chunk1"]) < tol["spec_rel"]


@pytest.mark.parametrize("chunk_batch", [False, True])
@pytest.mark.parametrize("precision", ["fp32", "tf32", "fp16"])
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_realtime_process_matches_reference(tag, precision, chunk_batch):
    """chunk_batch=False: the serial chunk loop (se_crn_realtime_process); True: every layer once over all chunks, only
    the GRU serial (chunk-major forward; offline files with few streams).  fp32: CUDA-core exact mode.  tf32: tcgen05 tensor cores (operands truncated to TF32, fp32 accumulate in TMEM);
    stated tolerances: tests/common.py TOL (for context, BASELINE.md section 3: the reference under its own bf16 autocast
    sits at 3.2e-2 x peak / 42 dB)."""
    g = load_golden(tag)
    tol = TOL[precision]
    if chunk_batch and precision == "fp16":
        pytest.skip("fp16 operand storage exists only on the streaming path")
    model = make_model(tag, precision)
    model.chunk_batch = chunk_batch
    B, L = int(g["meta"][1]), int(g["meta"][2])
    mix, _ = synth.make_mixture(B, L)
    y = model.realtime_process(torch.from_numpy(mix).cuda())
    assert model._state_owner == ("chunk-batch" if chunk_batch else "stream")
    y = (y[0] if isinstance(y, tuple) else y).cpu().numpy()
    assert y.shape == g["out"].shape
    assert np.abs(y - g["out"]).max() < tol["wave_max_abs"] * max(1.0, np.abs(g["out"]).max())
    assert si_sdr_db(y, g["out"]) > tol["si_sdr_vs_ref_db"]
    if "out_cont" in g:  # flag=True continuation keeps the causal-conv / GRU state (CRN_ELU.py:474,480)
        mix2, _ = synth.make_mixture(B, L // 2, first_stream=100)
        y2 = model.realtime_process(torch.from_numpy(mix2).cuda(), True).cpu().numpy()
        assert np.abs(y2 - g["out_cont"]).max() < tol["wave_max_abs"] * max(1.0, np.abs(g["out_cont"]).max())
    # CPU tensors in / out (predict.py:48,59-62): host<->device copies inside the native call
    yh = model.realtime_process(torch.from_numpy(mix))
    yh = (yh[0] if isinstance(yh, tuple) else yh).numpy()
    assert not torch.is_tensor(yh) and np.abs(yh - y).max() < 1e-6


def test_streams_are_independent_and_shardable():
    """Batch of B equals B batches of 1 (sharding streams across GPUs changes nothing; SURVEY.md section 8(e)).
    Not bit-identical: GEMM tiles straddle stream boundaries differently and the GlobalLayerNorm statistics are
    accumulated with atomics, so the last bits depend on the batch; the reference itself is batch-independent only
    to 5e-7 (SURVEY.md section 3.1)."""
    model = make_model("crn_small")
    mix, _ = synth.make_mixture(5, 6000)
    x = torch.from_numpy(mix).cuda()
    y = model.realtime_process(x).cpu().numpy()
    for b in (0, 3, 4):
        yb = model.realtime_process(x[b:b + 1]).cpu().numpy()
        assert np.abs(yb[0] - y[b]).max() < 2e-5


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_true_streaming_steps_equal_realtime_process(precision):
    """process_chunk (the streaming step the bench times) reproduces realtime_process sample for sample."""
    model = make_model("crn_small", precision)
    B, L = 3, 8000
    mix, _ = synth.make_mixture(B, L)
    x = torch.from_numpy(mix).cuda()
    ref = model.realtime_process(x).cpu().numpy()  # fp32: the chunk-batched forward; fp16: the serial chunk loop
    xp = torch.cat([torch.zeros(B, 3, 1600), torch.from_numpy(mix)], dim=-1)
    seg, gap = crn_oracle.segmentation(xp, 3200)
    N = seg.shape[0] // B
    seg = seg.reshape(B, N, 3, 3200).cuda()
    model.reset()
    outs = [model.process_chunk(seg[:, n].contiguous()).clone() for n in range(N)]
    y = torch.cat(outs[1:], dim=-1)[:, 1600:1600 + L].cpu().numpy()
    assert np.abs(y - ref).max() < 2e-5


def test_pipelined_host_steps_equal_device_steps():
    """process_chunk_host (pinned host buffers, copies on side streams, double-buffered staging) returns exactly what
    process_chunk returns for the same chunks, also when many steps are in flight."""
    model = make_model("crn_small", "fp32")
    B, N = 4, 9
    mix, _ = synth.make_mixture(B, 1600 * (N + 1))
    chunks = [torch.from_numpy(mix[:, :, 1600 * n:1600 * n + 3200].copy()) for n in range(N)]
    model.reset()
    want = [model.process_chunk(c.cuda()).cpu().numpy() for c in chunks]
    model.reset()
    pinned = [c.pin_memory() for c in chunks]
    outs = [torch.empty((B, 1600), dtype=torch.float32).pin_memory() for _ in range(N)]
    events = [model.process_chunk_host(pinned[n], outs[n]) for n in range(N)]  # no synchronisation in between
    for n in range(N):
        events[n].synchronize()
        assert np.array_equal(outs[n].numpy(), want[n]), n


def test_graph_and_eager_agree_and_reset_restores():
    from speech_enhancement_mi_b200._native import check, lib
    model = make_model("crn_small")
    model.chunk_batch = False  # the CUDA-graph replay belongs to the streaming chunk loop
    mix, _ = synth.make_mixture(2, 5000)
    x = torch.from_numpy(mix).cuda()
    y1 = model.realtime_process(x).cpu().numpy()
    check(lib().se_crn_set_graph(model._ctx, 0))
    y2 = model.realtime_process(x).cpu().numpy()
    assert np.abs(y1 - y2).max() < 2e-5


def test_weights_rebind_after_update():
    model = make_model("crn_small")
    mix, _ = synth.make_mixture(1, 4000)
    x = torch.from_numpy(mix).cuda()
    y1 = model.realtime_process(x).cpu().numpy()
    with torch.no_grad():
        model.deconvlist[-1].conv.bias.add_(0.5)
    y2 = model.realtime_process(x).cpu().numpy()
    assert np.abs(y1 - y2).max() > 1e-4
    model.cuda()
    y3 = model.realtime_process(x).cpu().numpy()
    assert np.abs(y2 - y3).max() < 2e-5


@pytest.mark.parametrize("tc", ["1", "0"])
def test_fp16_preconv_variants_match_reference(monkeypatch, tc):
    """fp16 mode runs the pre-convolutions on the tensor cores (preconv_tc.cu: implicit convolution through no-swizzle
    UMMA descriptors over the channels-last input resident in shared memory); SE_B200_PRECONV_TC=0 keeps the fp32
    CUDA-core kernel.  Both against the reference fixture at the stated fp16 tolerance, incl. the carried state."""
    monkeypatch.setenv("SE_B200_PRECONV_TC", tc)
    for tag in ("crn_small", "crn_teacher"):
        g = load_golden(tag)
        tol = TOL["fp16"]
        model = make_model(tag, "fp16")
        B, L = int(g["meta"][1]), int(g["meta"][2])
        mix, _ = synth.make_mixture(B, L)
        y = model.realtime_process(torch.from_numpy(mix).cuda()).cpu().numpy()
        assert np.abs(y - g["out"]).max() < tol["wave_max_abs"] * max(1.0, np.abs(g["out"]).max())
        assert si_sdr_db(y, g["out"]) > tol["si_sdr_vs_ref_db"]
        mix2, _ = synth.make_mixture(B, L // 2, first_stream=100)
        y2 = model.realtime_process(torch.from_numpy(mix2).cuda(), True).cpu().numpy()  # carried state across calls
        assert np.abs(y2 - g["out_cont"]).max() < tol["wave_max_abs"] * max(1.0, np.abs(g["out_cont"]).max())


@pytest.mark.parametrize("variant", ["mma", "cuda_cores", "gemm"])
def test_fp16_small_layer_variants_match_reference(monkeypatch, variant):
    """The last transposed convolution and the 8/16/32-channel skip 1x1 pairs run on warp-level mma.sync kernels in fp16
    mode (small_layers.cu); SE_B200_SMALL_MMA=0 keeps the CUDA-core generation, SE_B200_SMALL_LAYERS=0 the tcgen05 GEMM
    path.  All three against the reference fixtures (small / teacher / student shapes) at the stated fp16 tolerance."""
    if variant == "cuda_cores":
        monkeypatch.setenv("SE_B200_SMALL_MMA", "0")
    elif variant == "gemm":
        monkeypatch.setenv("SE_B200_SMALL_LAYERS", "0")
    for tag in CONFIGS:
        g = load_golden(tag)
        tol = TOL["fp16"]
        model = make_model(tag, "fp16")
        B, L = int(g["meta"][1]), int(g["meta"][2])
        mix, _ = synth.make_mixture(B, L)
        y = model.realtime_process(torch.from_numpy(mix).cuda())
        y = (y[0] if isinstance(y, tuple) else y).cpu().numpy()
        assert np.abs(y - g["out"]).max() < tol["wave_max_abs"] * max(1.0, np.abs(g["out"]).max()), tag
        assert si_sdr_db(y, g["out"]) > tol["si_sdr_vs_ref_db"], tag


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_full_size_1024_streams_replicas_match_oracle_checked_streams(precision):
    """BASELINE configs[1] size (teacher, 1024 concurrent streams, the bench's precision): 8 distinct streams are checked
    against the oracle over 4 chunk steps; the 1024-stream batch holds 128 shuffled replicas of each, and every replica
    must reproduce its original -- all m-tiles, stream groups and persistent-kernel CTAs of the full-size launch compute
    the same function as the small launch the oracle can afford to check."""
    oracle, _ = make_oracle("crn_teacher")
    model = make_model("crn_teacher", precision)
    D, B, N = 8, 1024, 4
    mix, _ = synth.make_mixture(D, 1600 * (N + 1))
    chunks = [torch.from_numpy(mix[:, :, 1600 * n:1600 * n + 3200].copy()) for n in range(N)]
    # streams on the atan2 branch cut of the phase feature are left out of the tight check (common.oracle_stream_steps)
    want, on_cut = oracle_stream_steps(oracle, chunks, model)
    keep = ~on_cut
    model.reset()
    small = np.concatenate([model.process_chunk(c.cuda()).cpu().numpy() for c in chunks], axis=-1)
    tol = TOL[precision]
    peak = max(1.0, float(np.abs(want).max()))
    assert np.abs(small - want)[keep].max() < tol["wave_max_abs"] * peak
    assert np.abs(small - want).max() < TOL["fp16"]["wave_max_abs"] * peak  # streams on the cut: still the same signal
    assert si_sdr_db(small[keep][:, 1600:], want[keep][:, 1600:]) > tol["si_sdr_vs_ref_db"]
    perm = torch.from_numpy(np.random.default_rng(5).permutation(B) % D)
    model.reset()
    big = np.concatenate([model.process_chunk(c[perm].cuda()).cpu().numpy() for c in chunks], axis=-1)
    # replicas differ from the small launch only through the order of the GLN statistics atomics (fp64) and tile borders
    rep_tol = 2e-5 if precision == "fp32" else 2e-3
    assert np.abs(big - small[perm.numpy()]).max() < rep_tol * peak
    assert np.abs(big - want[perm.numpy()])[keep[perm.numpy()]].max() < tol["wave_max_abs"] * peak


@pytest.mark.parametrize("switch,value", [("SE_B200_FRONT_MMA", "0"), ("SE_B200_ENC_MMA", "0"), ("SE_B200_TMA", "0"),
                                          ("SE_B200_DEC_MMA", "0"), ("SE_B200_TMA_PAIR", "0"), ("SE_B200_TMA_PAIR", "2"),
                                          ("SE_B200_GRU_WAVE", "0"), ("SE_B200_GRU_WAVE", "2"), ("SE_B200_ENC_TC", "0"),
                                          ("SE_B200_ENC_TC", "2"), ("SE_B200_GRU_PERSIST", "0"), ("SE_B200_B2B", "0")])
def test_fp16_round2_kernel_switches_match_reference(monkeypatch, switch, value):
    """Round-2 kernels against the kernels they replace: the fused pre-convolutions / small-channel encoder and decoder
    blocks (front_mma.cu, back_mma.cu: warp-level mma.sync on SMEM-resident streams), the TMA operand delivery and the
    CTA-pair mode of the tcgen05 GEMM, the wavefront GRU (gru_wave.cu) and the implicit-GEMM encoder block (enc_tc.cu),
    plus two earlier fallbacks: the GRU recurrence as one GEMM launch per step instead of a persistent kernel and the
    32- / 64-channel gates as separate GEMMs instead of the back-to-back one.
    The default path is covered by every other test; here each switch is turned OFF (0) or to its opt-in alternative (2:
    pair mode for every TMA GEMM, the one-layer form of the wavefront kernel, enc_tc for 16 -> 32 channels too) and that
    path must still meet the fixtures (all three configurations, incl. the carried state of a flag=True continuation).
    Every switch is read when a context is created, so it takes effect whatever contexts earlier tests built
    (test_stream_counts_gpu.py counts the enc_tc launches per setting)."""
    monkeypatch.setenv(switch, value)
    for tag in CONFIGS:
        g = load_golden(tag)
        tol = TOL["fp16"]
        model = make_model(tag, "fp16")
        B, L = int(g["meta"][1]), int(g["meta"][2])
        mix, _ = synth.make_mixture(B, L)
        y = model.realtime_process(torch.from_numpy(mix).cuda())
        y = (y[0] if isinstance(y, tuple) else y).cpu().numpy()
        assert np.abs(y - g["out"]).max() < tol["wave_max_abs"] * max(1.0, np.abs(g["out"]).max()), tag
        assert si_sdr_db(y, g["out"]) > tol["si_sdr_vs_ref_db"], tag
        if "out_cont" in g:
            mix2, _ = synth.make_mixture(B, L // 2, first_stream=100)
            y2 = model.realtime_process(torch.from_numpy(mix2).cuda(), True).cpu().numpy()
            assert np.abs(y2 - g["out_cont"]).max() < tol["wave_max_abs"] * max(1.0, np.abs(g["out_cont"]).max()), tag


def test_full_size_2048_student_streams_replicas_match_oracle_checked_streams():
    """BASELINE configs[2] per-GPU size (distilled student, 16384 streams over 8 GPUs = 2048 per GPU, fp16 operands): 8
    distinct streams are checked against the oracle over 3 chunk steps, the 2048-stream batch holds 256 shuffled replicas
    of each and every replica must reproduce its original (all 16 m-tiles of the two-layer wavefront GRU kernel, all
    stream-CTAs of the front-end kernels, all tiles of the TMA GEMMs).  On a 148-SM B200 the 16 m-tiles fit ONE launch
    of that kernel; batches that need a second wave are in test_stream_counts_gpu.py."""
    oracle, _ = make_oracle("crn_student")
    model = make_model("crn_student", "fp16")
    D, B, N = 8, 2048, 3
    mix, _ = synth.make_mixture(D, 1600 * (N + 1))
    chunks = [torch.from_numpy(mix[:, :, 1600 * n:1600 * n + 3200].copy()) for n in range(N)]
    with torch.no_grad():
        oracle.reset()
        state, want = None, []
        for c in chunks:
            y, state = oracle.stream_step(c, state)
            want.append(y.numpy())
    want = np.concatenate(want, axis=-1)
    tol = TOL["fp16"]
    peak = max(1.0, float(np.abs(want).max()))
    model.reset()
    small = np.concatenate([model.process_chunk(c.cuda()).cpu().numpy() for c in chunks], axis=-1)
    assert np.abs(small - want).max() < tol["wave_max_abs"] * peak
    perm = torch.from_numpy(np.random.default_rng(11).permutation(B) % D)
    model.reset()
    big = np.concatenate([model.process_chunk(c[perm].cuda()).cpu().numpy() for c in chunks], axis=-1)
    assert np.abs(big - small[perm.numpy()]).max() < 2e-3 * peak
    assert np.abs(big - want[perm.numpy()]).max() < tol["wave_max_abs"] * peak


def test_cirm_clamp_edge_through_the_fused_mask_kernel_and_fsn_apply_mask():
    """decompress_cIRM (utility.py:439-442) at and beyond the clamp |m| >= 9.9 -- values random-init weights never produce
    -- through BOTH product kernels that contain it: the fused mask stage of the CRN chunk step (se_debug_mask_spectrum:
    the mask kernel with an identity GlobalLayerNorm in front) and FullSubNet's se_fsn_apply_mask.  With a mic-0 spectrum
    of 1 + 0j the enhanced spectrum IS the decompressed mask; reference: utility.decompress_cIRM on linspace(-12, 12)
    from framing.npz (generated by the unmodified reference)."""
    import ctypes as C
    from speech_enhancement_mi_b200._native import check, lib
    g = load_golden("framing")
    m_in, want = g["cirm_in"], g["cirm_out"]  # 4001 values in [-12, 12]
    assert np.abs(m_in).max() >= 11.9 and (np.abs(m_in) >= 9.9).sum() > 500
    F, T = 201, 21
    n = F * T * 2
    reps = (n + m_in.size - 1) // m_in.size
    flat = np.tile(m_in, reps)[:n].astype(np.float32)
    flat_want = np.tile(want, reps)[:n].astype(np.float32)
    lim = 10.0 * np.log((10 + 9.9) / (10 - 9.9))
    assert abs(np.abs(flat_want).max() - lim) < 1e-3  # the fixture saturates at 10 ln(199)
    # ---- CRN fused mask kernel: mask [B, T, F, 2] -> spec [B, F, T, 2]
    model = make_model("crn_small", "fp32")
    model.forward(torch.zeros(1, 3, F, T, 2).cuda())  # creates the context
    mask = torch.from_numpy(flat.reshape(1, T, F, 2)).cuda()
    noisy = torch.zeros(1, T, F, 2, device="cuda")
    noisy[..., 0] = 1.0
    out = torch.empty(1, F, T, 2, device="cuda")
    check(lib().se_debug_mask_spectrum(model._ctx, mask.data_ptr(), noisy.data_ptr(), out.data_ptr(), 1),
          "se_debug_mask_spectrum")
    got = out.cpu().numpy().transpose(0, 2, 1, 3).reshape(-1)  # back to [T, F, 2] order
    assert np.isfinite(got).all()
    # identity norm: (m - 0) / (sqrt(1 + 1e-8) + 1e-8) moves m by 1.5e-8 relative; d/dm of the decompression is <= 100
    assert np.abs(got - flat_want).max() <= 2e-4 * lim
    assert np.abs(np.abs(got).max() - lim) < 1e-3
    # ---- FullSubNet: crm [R, 2, F, T], x [R, 2, F, T] -> [R, F, T, 2]
    crm = torch.from_numpy(flat.reshape(1, 2, F, T)).cuda()
    x = torch.zeros(1, 2, F, T, device="cuda")
    x[:, 0] = 1.0
    out2 = torch.empty(1, F, T, 2, device="cuda")
    check(lib().se_fsn_apply_mask(crm.data_ptr(), x.data_ptr(), out2.data_ptr(), 1, F, T, None), "se_fsn_apply_mask")
    got2 = out2.cpu().numpy().transpose(0, 3, 1, 2).reshape(-1)  # [2, F, T] order of crm
    assert np.isfinite(got2).all()
    assert np.abs(got2 - flat_want).max() <= 1e-4 * lim
