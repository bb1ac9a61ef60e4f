"""GPU: d loss / d mixture of realtime_process (se_crn_train_backward_input) for the teacher (CRN_ELU.TemporalCRN) and
the distilled student (distillation_crn.TemporalCRN).

The reference differentiates the mixture through torch.stft -> features -> network -> iSTFT -> overlap-add with the
carried conv buffers and GRU state detached (CRN_ELU.py:185,243), so autograd through oracle/crn_oracle.py (pinned to
the unmodified reference by tests/golden) is the oracle for d mixture.

Stated tolerances, about 5x the error measured on one B200 (NVIDIA B200, 1000 W power limit; worst case in brackets):
against the oracle, fp32 and 3xtf32 relative L2 error 2.5e-3 [4.9e-4, student; teacher 1.5e-4, most of it inherited
from d loss / d pred, whose own error against the oracle test_train_gpu.py states] and cosine 0.999999 [0.99999988];
tf32 cosine 0.9997 [0.99994]; the directional derivative 4e-3 [7e-4: the central difference's own error, measured against the oracle's
autograd on the CPU];
one stream of four against the same stream alone 1e-5 [1.5e-6]."""
import contextlib
import functools
import io

import numpy as np
import pytest
import torch

from common import CONFIGS, make_model
from oracle import crn_oracle, synth

pytestmark = pytest.mark.gpu

K = 3200


def _oracle(tag):
    cfg, seed, student = CONFIGS[tag]
    w = synth.make_crn_weights(seed=seed, **cfg)
    return crn_oracle.CRNOracle({k: torch.from_numpy(v) for k, v in w.items()}, segment_length=K, student=student, **cfg)


def _pieces(B, lengths):
    """Consecutive pieces of B streams: the first fresh (flag=False), the rest flag=True continuations."""
    out = []
    for i, L in enumerate(lengths):
        mix, src = synth.make_mixture(B, L, first_stream=100 * i)
        out.append((mix, src, [L] * B, i > 0))
    return out


@functools.lru_cache(maxsize=None)
def _oracle_dmix(tag, B, lengths, silence=None):
    o = _oracle(tag)
    res = []
    for mix, src, lens, flag in _pieces(B, lengths):
        if silence is not None:
            mix[..., silence[0]:silence[1]] = 0.0
        x = torch.from_numpy(mix).requires_grad_(True)
        pred = o.realtime_process(x, flag)
        loss, _, _ = crn_oracle.compute_loss(torch.from_numpy(src), pred, torch.tensor(lens))
        loss.backward()
        res.append(x.grad.numpy().copy())
    return res


def _pred(out):
    return out[0] if isinstance(out, tuple) else out


def _native_dmix(model, mix, src, lens, flag, device="cuda"):
    x = torch.from_numpy(mix).to(device).requires_grad_(True)
    pred = _pred(model.realtime_process(x, flag))
    with contextlib.redirect_stdout(io.StringIO()):
        loss, _, _ = model.compute_loss(torch.from_numpy(src).cuda(), pred, torch.tensor(lens))
    loss.backward()
    return x.grad


def _cmp(a, b):
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    b = np.asarray(b, dtype=np.float64).reshape(-1)
    rel = float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))
    cos = float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30))
    return rel, cos


def _check(got, want, precision, what):
    rel, cos = _cmp(got, want)
    print(f"{what} [{precision}]: relative L2 {rel:.3e}, cosine {cos:.7f}")
    assert np.isfinite(got).all()
    if precision == "tf32":
        assert cos >= 0.9997, (rel, cos)
    else:
        assert rel <= 2.5e-3 and cos >= 0.999999, (rel, cos)


def _run_pieces(tag, precision, B, lengths, train=True, silence=None):
    model = make_model(tag, precision=precision).cuda()
    model.train(train)
    got = []
    for mix, src, lens, flag in _pieces(B, lengths):
        if silence is not None:
            mix[..., silence[0]:silence[1]] = 0.0
        got.append(_native_dmix(model, mix, src, lens, flag).cpu().numpy())
    return model, got


# ---- 1, 2: parity with the oracle's autograd, fresh piece and a flag=True continuation ----------------------------------
@pytest.mark.parametrize("precision", ["fp32", "3xtf32", "tf32"])
@pytest.mark.parametrize("tag,B,lengths", [("crn_small", 2, (8000, 4800)), ("crn_teacher", 1, (6400, 4800)),
                                           ("crn_student", 1, (6400, 4800))])
def test_dmixture_matches_oracle_autograd(tag, B, lengths, precision):
    want = _oracle_dmix(tag, B, lengths)
    _, got = _run_pieces(tag, precision, B, lengths)
    for i, (g, w) in enumerate(zip(got, want)):
        _check(g, w, precision, f"{tag} piece {i}")


# ---- 3: directional derivative of J = <pred, w> by central differences (fp32, not the oracle's autograd) ------------
@pytest.mark.parametrize("tag,eps", [("crn_small", 1e-2), ("crn_student", 1e-3)])
def test_dmixture_directional_derivative(tag, eps):
    """d mixture is the derivative of realtime_process with the state entering every chunk held fixed: the reference
    detaches the carried conv buffers and GRU state (CRN_ELU.py:185,243).  So the central difference is taken of that
    function -- the oracle's forward (no autograd) with each chunk's entering state frozen at its value for the
    unperturbed mixture.  The direction scales each microphone by its own random gain: it keeps every STFT phase, so J
    stays smooth along it (a direction that rotates phases carries some bin across the atan2 / arctan branch cut, where
    the phase feature jumps by 2 pi or pi).  The phase-difference adjoint is covered by the oracle tests above."""
    mix, _ = synth.make_mixture(2, 8000)
    x0 = torch.from_numpy(mix)
    gen = torch.Generator().manual_seed(5)
    w = torch.randn(2, 8000, generator=gen)
    v = torch.randn(2, 3, 1, generator=gen) * x0
    o = _oracle(tag)
    P = K // 2

    def j_frozen(x, states):
        B, M, L = x.shape
        o.reset()
        seg, gap = crn_oracle.segmentation(torch.cat([torch.zeros(B, M, P), x], dim=-1), K)
        N = seg.shape[0] // B
        spec = o.stft_trans(seg).reshape(B, N, M, o.num_freqs, -1, 2)
        outs = []
        for n in range(N):
            if states is None:
                seen.append((dict(o.buf), o.h))
            else:
                o.buf, o.h = dict(states[n][0]), states[n][1]
            outs.append(o.istft_trans(o.forward(spec[:, n])))
        y = crn_oracle.over_add(torch.stack(outs, dim=1), gap)[..., P:]
        return float((y.double() * w.double()).sum())

    seen = []
    with torch.no_grad():
        j_frozen(x0, None)
        numeric = (j_frozen(x0 + eps * v, seen) - j_frozen(x0 - eps * v, seen)) / (2 * eps)
    model = make_model(tag, precision="fp32").cuda().eval()
    for p in model.parameters():
        p.requires_grad_(False)
    x = x0.cuda().requires_grad_(True)
    (_pred(model.realtime_process(x, False)) * w.cuda()).sum().backward()
    analytic = float((x.grad.cpu().double() * v.double()).sum())
    print(f"{tag}: <d mixture, v> {analytic:.6e}, central difference {numeric:.6e}")
    assert abs(analytic - numeric) <= 4e-3 * abs(numeric)


# ---- 4: parameter gradients unchanged; d mixture of a frozen model equals the one with parameter gradients -----------
def test_parameter_gradients_unchanged_and_frozen_dmixture():
    mix, src = synth.make_mixture(2, 8000)
    lens = [8000, 6500]
    model = make_model("crn_small", precision="fp32").cuda().train()

    def step(input_grad):
        model.zero_grad()
        x = torch.from_numpy(mix).cuda().requires_grad_(input_grad)
        pred = model.realtime_process(x, False)
        with contextlib.redirect_stdout(io.StringIO()):
            loss, _, _ = model.compute_loss(torch.from_numpy(src).cuda(), pred, torch.tensor(lens))
        loss.backward()
        grads = torch.cat([p.grad.reshape(-1) for p in model.parameters()]).cpu().numpy()
        return grads, (x.grad.cpu().numpy() if input_grad else None)

    a, _ = step(False)
    b, _ = step(False)
    c, d1 = step(True)
    _, d2 = step(True)
    spread = float(np.abs(a - b).max())
    err = float(np.abs(c - a).max())
    print(f"parameter gradients: spread of two plain backwards {spread:.3e}, with d mixture {err:.3e}")
    assert err <= 3 * spread + 1e-7 * float(np.abs(a).max())
    for p in model.parameters():
        p.requires_grad_(False)
    model.zero_grad()
    x = torch.from_numpy(mix).cuda().requires_grad_(True)
    pred = model.realtime_process(x, False)
    with contextlib.redirect_stdout(io.StringIO()):
        loss, _, _ = model.compute_loss(torch.from_numpy(src).cuda(), pred, torch.tensor(lens))
    loss.backward()
    d0 = x.grad.cpu().numpy()
    dspread = float(np.abs(d1 - d2).max())
    derr = float(np.abs(d0 - d1).max())
    print(f"d mixture: spread of two backwards {dspread:.3e}, without parameter gradients {derr:.3e}")
    assert derr <= 3 * dspread + 1e-7 * float(np.abs(d1).max())


# ---- 5: streams are independent ------------------------------------------------------------------------------------
def test_streams_independent():
    model = make_model("crn_small", precision="fp32").cuda().eval()
    mix, _ = synth.make_mixture(4, 6400)
    w = torch.randn(6400, generator=torch.Generator().manual_seed(2)).cuda()

    def dmix(m):
        x = torch.from_numpy(m).cuda().requires_grad_(True)
        pred = model.realtime_process(x, False)
        (pred[-1 if m.shape[0] == 1 else 2] * w).sum().backward()
        return x.grad.cpu().numpy()

    g4 = dmix(mix)
    g1 = dmix(mix[2:3].copy())
    assert np.all(g4[[0, 1, 3]] == 0.0)
    rel, cos = _cmp(g4[2], g1[0])
    print(f"stream 2 of 4 vs alone: relative L2 {rel:.3e}")
    assert rel <= 1e-5


# ---- 6: grid edges (gap 1, K/2, K), the front pad, digital silence -------------------------------------------------
@pytest.mark.parametrize("L,gap", [(6399, 1), (4800, K // 2), (6400, K)])
def test_dmixture_grid_edges(L, gap):
    assert crn_oracle.chunk_grid(L + K // 2, K)[0] == gap
    want = _oracle_dmix("crn_small", 2, (L,))
    _, got = _run_pieces("crn_small", "fp32", 2, (L,))
    _check(got[0], want[0], "fp32", f"L={L} gap={gap}")
    # the first samples (front pad: their first chunk is the padded one) and the last (gap) carry gradient as well
    assert np.abs(got[0][..., :8]).max() > 0 and np.abs(got[0][..., -8:]).max() > 0


@pytest.mark.parametrize("tag", ["crn_small", "crn_teacher"])
def test_dmixture_digital_silence(tag):
    """An exactly silent stretch makes whole frames of the spectrum exactly 0: the magnitude and atan2 adjoints must give
    0 there, as torch's autograd does (no NaN from 0 / 0), and the rest must still match."""
    silence = (2400, 5600)
    want = _oracle_dmix(tag, 1, (8000,), silence)
    _, got = _run_pieces(tag, "fp32", 1, (8000,), silence=silence)
    _check(got[0], want[0], "fp32", f"{tag} with silence")


# ---- 7: through autograd -------------------------------------------------------------------------------------------
def test_eval_mode_frozen_autograd_grad():
    mix, src = synth.make_mixture(1, 6400)
    model = make_model("crn_small", precision="fp32").cuda().eval()
    for p in model.parameters():
        p.requires_grad_(False)
    x = torch.from_numpy(mix).cuda().requires_grad_(True)
    pred = model.realtime_process(x, False)
    assert pred.grad_fn is not None
    with contextlib.redirect_stdout(io.StringIO()):
        loss, _, _ = model.compute_loss(torch.from_numpy(src).cuda(), pred, torch.tensor([6400]))
    (g,) = torch.autograd.grad(loss, x)
    _check(g.cpu().numpy(), _oracle_dmix("crn_small", 1, (6400,))[0], "fp32", "eval, frozen")
    # no_grad and a mixture without requires_grad keep the inference path (no graph)
    with torch.no_grad():
        assert model.realtime_process(x, False).grad_fn is None
    assert model.realtime_process(x.detach(), False).grad_fn is None


def test_learned_gain_and_cpu_mixture():
    mix, src = synth.make_mixture(2, 6400)
    raw = torch.from_numpy(mix).cuda()
    lens = torch.tensor([6400, 6400])
    model = make_model("crn_small", precision="fp32").cuda().train()

    def run(x):
        model.zero_grad()
        pred = model.realtime_process(x, False)
        with contextlib.redirect_stdout(io.StringIO()):
            loss, _, _ = model.compute_loss(torch.from_numpy(src).cuda(), pred, lens)
        loss.backward()
        return {k: p.grad.clone() for k, p in model.named_parameters()}

    ref_grads = run(raw)
    ref2 = run(raw)  # the weight gradients accumulate in atomics: two plain backwards differ in the last bits
    spread = max(float((ref2[k] - g).abs().max()) for k, g in ref_grads.items())
    xr = raw.clone().requires_grad_(True)
    run(xr)
    gain = torch.nn.Parameter(torch.ones((), device="cuda"))
    grads = run(gain * raw)
    want = float((raw.double() * xr.grad.double()).sum())
    print(f"gain.grad {float(gain.grad):.6e}, sum raw * d mixture {want:.6e}")
    assert abs(float(gain.grad) - want) <= 1e-5 * abs(want) + 1e-7
    err = max(float((grads[k] - g).abs().max()) for k, g in ref_grads.items())
    print(f"parameter gradients with the gain: {err:.3e} from a run without it (spread of two runs {spread:.3e})")
    assert err <= 3 * spread + 1e-7 * max(float(g.abs().max()) for g in ref_grads.values())
    xc = torch.from_numpy(mix).requires_grad_(True)
    run(xc)
    assert xc.grad.device.type == "cpu" and xc.grad.dtype == torch.float32
    rel, _ = _cmp(xc.grad.numpy(), xr.grad.cpu().numpy())
    assert rel <= 1e-5
