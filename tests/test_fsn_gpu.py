"""GPU parity of the FullSubNet chunk path (se_fsn_* behind speech_enhancement_mi_b200.fullsubnet) against fixtures of
the unmodified reference (fp32 CPU run) and the oracle.  The LSTM GEMMs run on TF32 tensor cores (fp32 accumulate, fp32
cell state): stated tolerance = 2e-2 x peak on mask / waveform and >= 40 dB SI-SDR against the reference waveform; the
integer index work (unfold) is bit-exact."""
import os

import numpy as np
import pytest
import torch

from common import FSN_FULL, FSN_SMALL, FSN_TOL_DB, FSN_TOL_REL, GOLDEN, rel_err, si_sdr_db
from common import make_fsn as make
from oracle import synth
from oracle.fsn_oracle import FSNOracle, unfold

pytestmark = pytest.mark.gpu

TOL_REL, TOL_DB = FSN_TOL_REL, FSN_TOL_DB


def load(tag):
    z = np.load(os.path.join(GOLDEN, f"{tag}.npz"))
    return {k: z[k] for k in z.files}


def test_unfold_bit_exact():
    from speech_enhancement_mi_b200.fullsubnet import BaseModel
    g = load("fsn_small")
    x = torch.from_numpy(g["unfold_in"]).cuda()
    assert np.array_equal(BaseModel.unfold(x, 2).cpu().numpy(), g["unfold_out"])
    assert np.array_equal(BaseModel.unfold(x, 0).cpu().numpy(), g["unfold0_out"])
    big = torch.randn(2, 1, 201, 21)
    assert np.array_equal(BaseModel.unfold(big.cuda(), 15).cpu().numpy(), unfold(big, 15).numpy())


@pytest.mark.parametrize("tag,cfg,seed", [("fsn_small", FSN_SMALL, 11), ("fsn_full", FSN_FULL, 5)])
def test_forward_chunk_matches_reference(tag, cfg, seed):
    g = load(tag)
    m = make(cfg, seed)
    x1 = torch.from_numpy(g["x_chunk1"]).cuda()
    m.reset_state(x1.shape[0])
    f1 = m.forward(x1).cpu().numpy()
    f2 = m.forward(x1).cpu().numpy()  # running CumLayerNorm mean + carried LSTM state
    assert rel_err(f1, g["fwd_chunk1"]) < TOL_REL
    assert rel_err(f2, g["fwd_chunk1_again"]) < TOL_REL


def test_fp16_subband_operands_match_reference():
    """SE_PRECISION_FP16: sub-band LSTM operands stored as fp16 (the reference's own CUDA path runs under fp16 autocast,
    fullsubnet.py:943); same stated tolerance as the tf32 mode, on the full-size configuration."""
    g = load("fsn_full")
    m = make(FSN_FULL, 5, precision="fp16")
    x1 = torch.from_numpy(g["x_chunk1"]).cuda()
    m.reset_state(x1.shape[0])
    f1 = m.forward(x1).cpu().numpy()
    f2 = m.forward(x1).cpu().numpy()
    assert rel_err(f1, g["fwd_chunk1"]) < TOL_REL
    assert rel_err(f2, g["fwd_chunk1_again"]) < TOL_REL
    seed, B, L = [int(v) for v in g["meta"]]
    mix, src = synth.make_mixture(B, L)
    pred = m.realtime_process(torch.from_numpy(mix).cuda(), None, flag=False, train=False)[0].cpu().numpy()
    assert np.abs(pred - g["out"]).max() < TOL_REL * max(1.0, np.abs(g["out"]).max())
    assert si_sdr_db(pred, g["out"]) > TOL_DB


def test_realtime_process_matches_reference():
    g = load("fsn_small")
    m = make(FSN_SMALL, 11)
    B, L = int(g["meta"][1]), int(g["meta"][2])
    mix, src = synth.make_mixture(B, L)
    s3 = torch.from_numpy(np.repeat(src[:, None, :], 3, axis=1).copy())
    pred, crm, sf, xf = m.realtime_process(torch.from_numpy(mix).cuda(), s3.cuda(), flag=False, train=False)
    pred = pred.cpu().numpy()
    assert pred.shape == g["out"].shape
    assert rel_err(crm.cpu().numpy(), g["crm"]) < TOL_REL
    assert rel_err(sf.cpu().numpy(), g["sf"]) < 1e-5 and rel_err(xf.cpu().numpy(), g["xf"]) < 1e-5
    assert np.abs(pred - g["out"]).max() < TOL_REL * max(1.0, np.abs(g["out"]).max())
    assert si_sdr_db(pred, g["out"]) > TOL_DB
    mix2, _ = synth.make_mixture(B, L // 2, first_stream=100)
    p2 = m.realtime_process(torch.from_numpy(mix2).cuda(), None, flag=True, train=False).cpu().numpy()
    assert np.abs(p2 - g["out_cont"]).max() < TOL_REL * max(1.0, np.abs(g["out_cont"]).max())
    # CPU tensors in, CPU tensors out (predict_fullsubnet.py uses .cuda(); the drop-in accepts both)
    p3 = m.realtime_process(torch.from_numpy(mix), None, flag=False, train=False)
    assert not p3.is_cuda and np.abs(p3.numpy() - pred).max() < 1e-5


def test_streams_independent_and_oracle_agrees():
    m = make(FSN_SMALL, 11)
    o = FSNOracle(synth.make_fsn_weights(seed=11, **FSN_SMALL), **FSN_SMALL)
    mix, _ = synth.make_mixture(4, 5000)
    x = torch.from_numpy(mix)
    y = m.realtime_process(x.cuda(), None, flag=False, train=False).cpu().numpy()
    with torch.no_grad():
        want, _ = o.realtime_process(x)
    assert np.abs(y - want.numpy()).max() < TOL_REL * max(1.0, float(want.abs().max()))
    yb = m.realtime_process(x[2:3].cuda(), None, flag=False, train=False).cpu().numpy()
    assert np.abs(yb[0] - y[2]).max() < 1e-4


def test_realtime_process_whole_utterance_train_true_matches_reference():
    """train=True (the signature's default, fullsubnet.py:921-927): all chunks concatenated into ONE forward, so both
    CumLayerNorms take a single step over the whole utterance instead of one per chunk.  Fixture: the unmodified reference
    with train=True, incl. the 4-tuple outputs and a flag=True continuation piece (second norm step, carried LSTM state)."""
    g = load("fsn_small_whole")
    m = make(FSN_SMALL, 11)
    B, L = int(g["meta"][1]), int(g["meta"][2])
    mix, src = synth.make_mixture(B, L)
    s3 = torch.from_numpy(np.repeat(src[:, None, :], 3, axis=1).copy())
    pred, crm, sf, xf = m.realtime_process(torch.from_numpy(mix).cuda(), s3.cuda(), flag=False, train=True)
    pred = pred.cpu().numpy()
    assert rel_err(crm.cpu().numpy(), g["crm"]) < TOL_REL
    assert rel_err(sf.cpu().numpy(), g["sf"]) < 1e-5 and rel_err(xf.cpu().numpy(), g["xf"]) < 1e-5
    assert np.abs(pred - g["out"]).max() < TOL_REL * max(1.0, np.abs(g["out"]).max())
    assert si_sdr_db(pred, g["out"]) > TOL_DB
    mix2, _ = synth.make_mixture(B, L // 2, first_stream=100)
    p2 = m.realtime_process(torch.from_numpy(mix2).cuda(), None, flag=True, train=True).cpu().numpy()
    assert np.abs(p2 - g["out_cont"]).max() < TOL_REL * max(1.0, np.abs(g["out_cont"]).max())
    # the chunk loop is a different function of the same weights (per-chunk running norms): it must NOT reproduce this
    p_loop = m.realtime_process(torch.from_numpy(mix).cuda(), None, flag=False, train=False).cpu().numpy()
    assert np.abs(p_loop - g["out"]).max() > 10 * np.abs(pred - g["out"]).max()


@pytest.mark.parametrize("precision", ["tf32", "fp16"])
def test_full_config_realtime_process_matches_reference(precision):
    """config.yaml:153-172 sizes (full-band 512, sub-band 384 hidden units) through the whole realtime_process in both
    precisions of the LSTM operands."""
    g = load("fsn_full")
    m = make(FSN_FULL, 5, precision=precision)
    seed, B, L = [int(v) for v in g["meta"]]
    mix, _ = synth.make_mixture(B, L)
    pred = m.realtime_process(torch.from_numpy(mix).cuda(), None, flag=False, train=False).cpu().numpy()
    assert pred.shape == g["out"].shape
    assert np.abs(pred - g["out"]).max() < TOL_REL * max(1.0, np.abs(g["out"]).max())
    assert si_sdr_db(pred, g["out"]) > TOL_DB


@pytest.mark.parametrize("precision,B,first,count,max_streams",
                         [("tf32", 4, 1, 2, None), ("fp16", 4, 1, 2, None),
                          ("tf32", 300, 100, 130, 512), ("fp16", 300, 100, 130, 512)],
                         ids=["tf32", "fp16", "tf32-B300-of-512", "fp16-B300-of-512"])
def test_partial_state_reset_touches_only_the_given_streams(precision, B, first, count, max_streams):
    """se_fsn_reset_state(first, count) (fullsubnet.py:826-832 for a sub-range of the streams): the LSTM cell states are
    stored unit-major ([H][capacity x bins], gemm_tc.cu EPI_LSTM), so a stream range is a strided block of every unit
    row.  Streams first .. first+count-1 are reset between two calls, the others continue: the reset streams must
    reproduce a run from a fully reset model bit for bit, the others the uninterrupted continuation.  300 streams on a
    context of 512: the pitch of the unit rows is the capacity, not the batch."""
    from speech_enhancement_mi_b200._native import check, lib
    mix1, _ = synth.make_mixture(B, 6400)
    mix2, _ = synth.make_mixture(B, 6400, first_stream=50)
    x1, x2 = torch.from_numpy(mix1).cuda(), torch.from_numpy(mix2).cuda()
    # fp16 operands need 64-unit tiles (the TMA / CTA-pair path of the LSTM steps): sb_hidden 64 there
    FSN_SMALL = dict(globals()["FSN_SMALL"], sb_hidden=64) if precision == "fp16" else globals()["FSN_SMALL"]

    def run(between):
        m = make(FSN_SMALL, 11, precision=precision, max_streams=max_streams)
        m.realtime_process(x1, None, flag=False, train=False)
        assert m._ctx_capacity == (max_streams or B)
        between(m)
        return m.realtime_process(x2, None, flag=True, train=False).cpu().numpy()

    y_cont = run(lambda m: None)
    y_fresh = run(lambda m: m.reset_state(B))
    y = run(lambda m: check(lib().se_fsn_reset_state(m._ctx, first, count, None), "se_fsn_reset_state"))
    sel = np.zeros(B, dtype=bool)
    sel[first:first + count] = True
    assert np.array_equal(y[~sel], y_cont[~sel])
    assert np.array_equal(y[sel], y_fresh[sel])
    # the carried state matters for every reset stream, or this test would prove nothing
    assert np.abs(y_cont[sel] - y_fresh[sel]).max(axis=1).min() > 1e-4
