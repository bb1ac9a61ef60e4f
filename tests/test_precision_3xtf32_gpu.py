"""precision="3xtf32": every tensor-core GEMM of the CRN and FullSubNet paths in the split form of gemm_tc.cu
(gemm_tc3x_kernel: fp32 operands held as a tf32 head and a tf32 tail, lo.hi + hi.lo + hi.hi per K step, exact-mode
epilogue math).  The mode claims the accuracy of the fp32 exact mode, so the CRN checks run at TOL["fp32"], not
loosened, and a launch guard proves that no GEMM fell back to the single-pass tf32 kernel behind a passing parity check.

FullSubNet has no fp32 CUDA-core mode to borrow a tolerance from.  Its stated tolerances are about 4-5x the error
measured on one B200 (1000 W power limit) against the reference fixtures; see FSN_3X_TOL_REL / FSN_3X_TOL_DB."""
import collections
import re

import numpy as np
import pytest
import torch

from common import (CONFIGS, FSN_FULL, FSN_SMALL, GOLDEN, TOL, load_golden, make_fsn, make_model, make_oracle,
                    oracle_stream_steps, rel_err, si_sdr_db)
from oracle import synth
from test_stream_counts_gpu import launches, profiled_step
from test_train_gpu import _report, _step

pytestmark = pytest.mark.gpu

TOLX = TOL["fp32"]
# FullSubNet in 3xtf32 against the reference fixtures: max-abs error on mask and waveform relative to max(1, peak), and
# SI-SDR against the reference waveform.  Measured on one NVIDIA B200 (1000 W power limit), worst case over the tests
# below: 1.3e-6 x peak (fsn_full forward chunk; waveforms 3.3e-7 .. 7.5e-7) and 108.7 dB (fsn_full waveform).  The
# tolerances are about 4.6x that error (6e-6) and 14 dB below it (94 dB).  For comparison, the CRN in this mode measured
# 2.0e-6 .. 1.1e-5 x peak and >= 106 dB against its fixtures, inside TOL["fp32"].
FSN_3X_TOL_REL, FSN_3X_TOL_DB = 6e-6, 94.0


# ---- CRN: the reference fixtures -------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_forward_chunk_matches_reference(tag):
    g = load_golden(tag)
    model = make_model(tag, "3xtf32")
    out = model.forward(torch.from_numpy(g["spec_chunk1"]).cuda())
    out = out[0] if isinstance(out, tuple) else out
    err = rel_err(out.cpu().numpy(), g["fwd_chunk1"])
    print(f"{tag}: forward chunk rel err {err:.3e}")
    assert err < TOLX["spec_rel"]


@pytest.mark.parametrize("chunk_batch", [False, True])
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_realtime_process_matches_reference(tag, chunk_batch):
    """chunk_batch=False: the serial chunk loop; True: the chunk-major forward of the training context (offline files
    with few streams), whose GEMMs split too."""
    g = load_golden(tag)
    model = make_model(tag, "3xtf32")
    model.chunk_batch = chunk_batch
    B, L = int(g["meta"][1]), int(g["meta"][2])
    mix, _ = synth.make_mixture(B, L)
    y = model.realtime_process(torch.from_numpy(mix).cuda())
    assert model._state_owner == ("chunk-batch" if chunk_batch else "stream")
    y = (y[0] if isinstance(y, tuple) else y).cpu().numpy()
    assert y.shape == g["out"].shape
    peak = max(1.0, np.abs(g["out"]).max())
    print(f"{tag}: max-abs {np.abs(y - g['out']).max() / peak:.3e} x peak, SI-SDR {si_sdr_db(y, g['out']):.1f} dB")
    assert np.abs(y - g["out"]).max() < TOLX["wave_max_abs"] * peak
    assert si_sdr_db(y, g["out"]) > TOLX["si_sdr_vs_ref_db"]
    if "out_cont" in g:  # flag=True continuation keeps the causal-conv / GRU state
        mix2, _ = synth.make_mixture(B, L // 2, first_stream=100)
        y2 = model.realtime_process(torch.from_numpy(mix2).cuda(), True)
        y2 = (y2[0] if isinstance(y2, tuple) else y2).cpu().numpy()
        assert np.abs(y2 - g["out_cont"]).max() < TOLX["wave_max_abs"] * max(1.0, np.abs(g["out_cont"]).max())


# ---- CRN: full size and ragged tiles against the oracle ---------------------------------------------------------------
def checked_streams(D, N):
    oracle, _ = make_oracle("crn_teacher")
    model = make_model("crn_teacher", "3xtf32")
    mix, _ = synth.make_mixture(D, 1600 * (N + 1))
    chunks = [torch.from_numpy(mix[:, :, 1600 * n:1600 * n + 3200].copy()) for n in range(N)]
    # streams on the atan2 branch cut of the phase feature are left out of the tight check (common.oracle_stream_steps)
    want, on_cut = oracle_stream_steps(oracle, chunks, model)
    model.reset()
    small = np.concatenate([model.process_chunk(c.cuda()).cpu().numpy() for c in chunks], axis=-1)
    keep = ~on_cut
    peak = max(1.0, float(np.abs(want).max()))
    print(f"8 checked streams vs oracle: max-abs {np.abs(small - want)[keep].max() / peak:.3e} x peak")
    assert np.abs(small - want)[keep].max() < TOLX["wave_max_abs"] * peak
    assert np.abs(small - want).max() < TOL["fp16"]["wave_max_abs"] * peak  # streams on the cut: still the same signal
    assert si_sdr_db(small[keep][:, 1600:], want[keep][:, 1600:]) > TOLX["si_sdr_vs_ref_db"]
    return model, chunks, want, keep, small, peak


def test_full_size_1024_streams_replicas_match_oracle_checked_streams():
    """1024 teacher streams (the benchmark size): 128 shuffled replicas of each of 8 oracle-checked streams; every
    replica must reproduce its original, and the originals the oracle, at the fp32 tolerance."""
    D, B, N = 8, 1024, 4
    model, chunks, want, keep, small, peak = checked_streams(D, N)
    perm = torch.from_numpy(np.random.default_rng(5).permutation(B) % D)
    model.reset()
    big = np.concatenate([model.process_chunk(c[perm].cuda()).cpu().numpy() for c in chunks], axis=-1)
    # replicas differ from the small launch only through the order of the GLN statistics atomics (fp64) and tile borders
    assert np.abs(big - small[perm.numpy()]).max() < 2e-5 * peak
    assert np.abs(big - want[perm.numpy()])[keep[perm.numpy()]].max() < TOLX["wave_max_abs"] * peak


@pytest.mark.parametrize("B", [129, 257])
def test_ragged_last_tile_replicas_match_checked_streams(B):
    """129 / 257 streams: the row = stream GEMMs (GRU projections and cells) end in a partial m-tile of 1 row.  The 8
    checked streams sit first and last (in the ragged tile), shuffled replicas in between."""
    D, N = 8, 3
    model, chunks, want, keep, small, peak = checked_streams(D, N)
    idx = np.random.default_rng(B).permutation(B) % D
    idx[:D] = np.arange(D)
    idx[B - D:] = np.arange(D)
    model.reset()
    big = np.concatenate([model.process_chunk(c[torch.from_numpy(idx)].cuda()).cpu().numpy() for c in chunks], axis=-1)
    assert np.abs(big - small[idx]).max() < 2e-5 * peak
    assert np.abs(big - want[idx])[keep[idx]].max() < TOLX["wave_max_abs"] * peak


# ---- launch guard -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_split_form_replaces_every_tf32_gemm(tag):
    """One eager chunk step in each mode: 3xtf32 launches gemm_tc3x_kernel exactly where tf32 launches gemm_tc_kernel,
    never gemm_tc_kernel itself, and the CUDA-core gemm_fp32_kernel exactly as often as tf32 does."""
    mix, _ = synth.make_mixture(8, 3200)
    chunk = torch.from_numpy(mix).cuda()
    counts = {}
    for precision in ("tf32", "3xtf32"):
        model = make_model(tag, precision)
        _, c = profiled_step(model, chunk)
        counts[precision] = {k: launches(c, k) for k in ("gemm_tc_kernel", "gemm_tc3x_kernel", "gemm_fp32_kernel")}
    print(f"{tag}: {counts}")
    assert counts["tf32"]["gemm_tc_kernel"] > 0
    assert counts["3xtf32"]["gemm_tc3x_kernel"] == counts["tf32"]["gemm_tc_kernel"]
    assert counts["3xtf32"]["gemm_tc_kernel"] == 0
    assert counts["3xtf32"]["gemm_fp32_kernel"] == counts["tf32"]["gemm_fp32_kernel"]


def fsn_gemm_launches(model, B):
    """One FullSubNet forward chunk (its CUDA graph) under torch.profiler: launches of the two GEMM kernel names."""
    from torch.profiler import ProfilerActivity, profile
    x = torch.randn(B, 2 * model.num_mics, 201, 21, generator=torch.Generator().manual_seed(B)).cuda()
    model.reset_state(B)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        model.forward(x)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names, "the profiler recorded no kernel launches"
    out = collections.Counter()
    for n in names:
        for k in ("gemm_tc_kernel", "gemm_tc3x_kernel"):
            if re.search(r"\b" + k + r"\b", n):
                out[k] += 1
    return out


def test_fsn_split_form_replaces_every_tf32_gemm():
    counts = {p: fsn_gemm_launches(make_fsn(FSN_SMALL, 11, precision=p), 4) for p in ("tf32", "3xtf32")}
    print(counts)
    assert counts["tf32"]["gemm_tc_kernel"] > 0
    assert counts["3xtf32"]["gemm_tc3x_kernel"] == counts["tf32"]["gemm_tc_kernel"]
    assert counts["3xtf32"]["gemm_tc_kernel"] == 0


# ---- CRN training step --------------------------------------------------------------------------------------------------
def test_small_train_step_matches_reference():
    """The thresholds of the fp32 training tests (test_train_gpu.py): forward GEMMs in the split form, the backward in
    its 3xTF32 mma.sync form (the default beside an fp32-accurate forward)."""
    g = np.load(f"{GOLDEN}/train_grads.npz")
    model = make_model("crn_small", precision="3xtf32").cuda().train()
    mix, src = synth.make_mixture(2, 8000)
    pred, dpred, losses, grads = _step(model, mix, src, [8000, 6500], False)
    assert rel_err(pred, g["small_pred"]) < 2e-4
    assert np.allclose(losses, g["small_loss"], atol=2e-3)
    assert rel_err(dpred, g["small_dpred"]) < 4e-3
    _report(grads, g, "small_grad/", 1e-3)
    mix2, src2 = synth.make_mixture(2, 4800, first_stream=100)
    pred, dpred, losses, grads = _step(model, mix2, src2, [4800, 4800], True)
    assert rel_err(pred, g["small_cont_pred"]) < 2e-4
    assert np.allclose(losses, g["small_cont_loss"], atol=2e-3)
    _report(grads, g, "small_cont_grad/", 1e-3)


def test_teacher_train_step_matches_reference():
    g = np.load(f"{GOLDEN}/train_grads.npz")
    model = make_model("crn_teacher", precision="3xtf32").cuda().train()
    mix, src = synth.make_mixture(1, 6400)
    pred, dpred, losses, grads = _step(model, mix, src, [6400], False)
    assert rel_err(pred, g["teacher_pred"]) < 2e-4
    assert np.allclose(losses, g["teacher_loss"], atol=2e-3)
    assert rel_err(dpred, g["teacher_dpred"]) < 4e-3
    bad = []
    for k in [k[len("teacher_gnorm/"):] for k in g.files if k.startswith("teacher_gnorm/")]:
        gn = float(g["teacher_gnorm/" + k])
        if abs(float(np.linalg.norm(grads[k].astype(np.float64))) - gn) > 1e-3 * gn + 1e-9:
            bad.append((k, "norm"))
        head = g["teacher_ghead/" + k]
        if np.abs(grads[k].reshape(-1)[:64] - head).max() > 1e-3 * (np.abs(grads[k]).max() + 1e-30):
            bad.append((k, "head"))
    assert not bad, bad


# ---- FullSubNet -----------------------------------------------------------------------------------------------------------
def fsn_check(what, got, want, sdr=True):
    peak = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(got - want).max()) / peak
    db = si_sdr_db(got, want) if sdr else float("inf")
    print(f"{what}: max-abs {err:.3e} x peak" + (f", SI-SDR {db:.1f} dB" if sdr else ""))
    assert err < FSN_3X_TOL_REL, (what, err)
    assert db > FSN_3X_TOL_DB, (what, db)


@pytest.mark.parametrize("tag,cfg,seed", [("fsn_small", FSN_SMALL, 11), ("fsn_full", FSN_FULL, 5)])
def test_fsn_forward_chunk_matches_reference(tag, cfg, seed):
    g = load_golden(tag)
    m = make_fsn(cfg, seed, precision="3xtf32")
    x1 = torch.from_numpy(g["x_chunk1"]).cuda()
    m.reset_state(x1.shape[0])
    f1 = m.forward(x1).cpu().numpy()
    f2 = m.forward(x1).cpu().numpy()  # running CumLayerNorm mean + carried LSTM state
    fsn_check(f"{tag} forward chunk", f1, g["fwd_chunk1"], sdr=False)
    fsn_check(f"{tag} forward chunk again", f2, g["fwd_chunk1_again"], sdr=False)


def test_fsn_realtime_process_matches_reference():
    g = load_golden("fsn_small")
    m = make_fsn(FSN_SMALL, 11, precision="3xtf32")
    B, L = int(g["meta"][1]), int(g["meta"][2])
    mix, src = synth.make_mixture(B, L)
    s3 = torch.from_numpy(np.repeat(src[:, None, :], 3, axis=1).copy())
    pred, crm, _, _ = m.realtime_process(torch.from_numpy(mix).cuda(), s3.cuda(), flag=False, train=False)
    fsn_check("fsn_small mask", crm.cpu().numpy(), g["crm"], sdr=False)
    fsn_check("fsn_small wave", pred.cpu().numpy(), g["out"])
    mix2, _ = synth.make_mixture(B, L // 2, first_stream=100)
    p2 = m.realtime_process(torch.from_numpy(mix2).cuda(), None, flag=True, train=False).cpu().numpy()
    fsn_check("fsn_small wave, flag=True", p2, g["out_cont"])


def test_fsn_full_config_realtime_process_matches_reference():
    g = load_golden("fsn_full")
    m = make_fsn(FSN_FULL, 5, precision="3xtf32")
    _, B, L = [int(v) for v in g["meta"]]
    mix, _ = synth.make_mixture(B, L)
    pred = m.realtime_process(torch.from_numpy(mix).cuda(), None, flag=False, train=False).cpu().numpy()
    fsn_check("fsn_full wave", pred, g["out"])


def test_fsn_whole_utterance_train_true_matches_reference():
    g = load_golden("fsn_small_whole")
    m = make_fsn(FSN_SMALL, 11, precision="3xtf32")
    B, L = int(g["meta"][1]), int(g["meta"][2])
    mix, src = synth.make_mixture(B, L)
    s3 = torch.from_numpy(np.repeat(src[:, None, :], 3, axis=1).copy())
    pred, crm, _, _ = m.realtime_process(torch.from_numpy(mix).cuda(), s3.cuda(), flag=False, train=True)
    fsn_check("fsn_small_whole mask", crm.cpu().numpy(), g["crm"], sdr=False)
    fsn_check("fsn_small_whole wave", pred.cpu().numpy(), g["out"])
    mix2, _ = synth.make_mixture(B, L // 2, first_stream=100)
    p2 = m.realtime_process(torch.from_numpy(mix2).cuda(), None, flag=True, train=True).cpu().numpy()
    fsn_check("fsn_small_whole wave, flag=True", p2, g["out_cont"])
