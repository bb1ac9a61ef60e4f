"""Shared helpers for the parity tests (test infrastructure; may import oracle/)."""
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

from oracle import synth  # noqa: E402
from oracle.crn_oracle import CRNOracle, si_sdr_db  # noqa: E402

GOLDEN = os.path.join(REPO, "tests", "golden")

TEACHER = dict(num_channels=[16, 32, 64, 128], num_freqs=201, hidden=512, num_layers=2, num_inputs=3, kernel_size=3)
STUDENT = dict(num_channels=[16, 32, 64, 64], num_freqs=201, hidden=128, num_layers=2, num_inputs=3, kernel_size=3)
SMALL = dict(num_channels=[8, 8, 16, 16], num_freqs=201, hidden=32, num_layers=2, num_inputs=3, kernel_size=3)
CONFIGS = {"crn_small": (SMALL, 7, False), "crn_teacher": (TEACHER, 0, False), "crn_student": (STUDENT, 3, True)}

# Stated floating-point tolerances of the CUDA path against the reference (north_star: "max-abs error on the waveform
# plus an SI-SDR delta"), set at roughly 4-5x the error MEASURED on the three fixtures (B200, round 2; worst case in
# brackets) so that a regression of that size fails:
#   fp32  re-associates sums (tiled GEMM, four-step FFT) but keeps fp32 everywhere  [wave 3e-6 x peak, spectrum 2.2e-6, 114 dB]
#   tf32  tcgen05 kind::tf32 on fp32 storage (10-bit mantissa operands)              [wave 3.0e-3 x peak, spectrum 2.0e-3, 55.9 dB]
#   fp16  fp16 operand storage (11-bit significand), fp32 accumulate / statistics / state
#                                                                                    [wave 5.0e-3 x peak (student), spectrum 2.9e-3, 53.0 dB]
# wave_max_abs is relative to max(1, peak of the reference waveform); spec_rel to the peak of the reference spectrum.
TOL = {
    "fp32": dict(wave_max_abs=2e-5, spec_rel=2e-5, si_sdr_vs_ref_db=100.0),
    "tf32": dict(wave_max_abs=1.2e-2, spec_rel=1e-2, si_sdr_vs_ref_db=48.0),
    "fp16": dict(wave_max_abs=1.2e-2, spec_rel=1.2e-2, si_sdr_vs_ref_db=48.0),
}


FSN_SMALL = dict(num_freqs=201, num_mics=3, fb_hidden=64, sb_hidden=32, sb_num_neighbors=15, fb_num_neighbors=0,
                 num_layers=2)
FSN_FULL = dict(num_freqs=201, num_mics=3, fb_hidden=512, sb_hidden=384, sb_num_neighbors=15, fb_num_neighbors=0,
                num_layers=2)
# FullSubNet against the reference / oracle, tf32 and fp16: max-abs error on mask and waveform relative to the peak, and
# SI-SDR against the reference waveform
FSN_TOL_REL, FSN_TOL_DB = 2e-2, 40.0


def make_fsn(cfg, seed, **kw):
    """The product FullSubNet with the deterministic synthetic weights of (cfg, seed) loaded through load_state_dict."""
    from speech_enhancement_mi_b200 import fullsubnet
    m = fullsubnet.FullSubNet(
        num_freqs=cfg["num_freqs"], look_ahead=0, sequence_model="LSTM", fb_num_neighbors=cfg["fb_num_neighbors"],
        sb_num_neighbors=cfg["sb_num_neighbors"], fb_output_activate_function="ReLU", sb_output_activate_function=False,
        fb_model_hidden_size=cfg["fb_hidden"], sb_model_hidden_size=cfg["sb_hidden"], num_mics=cfg["num_mics"],
        num_layers=cfg["num_layers"], weight_init=False, sample_rate=16000, segment_length=3200, win_length=25,
        hop_length=10, n_fft=400, **kw)
    w = synth.make_fsn_weights(seed=seed, **cfg)
    missing, unexpected = m.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()}, strict=True)
    assert not missing and not unexpected
    return m.eval()


def load_golden(tag):
    z = np.load(os.path.join(GOLDEN, f"{tag}.npz"))
    return {k: z[k] for k in z.files}


def make_oracle(tag):
    cfg, seed, student = CONFIGS[tag]
    w = synth.make_crn_weights(seed=seed, **cfg)
    return CRNOracle({k: torch.from_numpy(v) for k, v in w.items()}, segment_length=3200, student=student, **cfg), w


def make_model(tag, precision="fp32", **kw):
    """The product model with the deterministic synthetic weights of `tag` loaded through load_state_dict."""
    from speech_enhancement_mi_b200 import CRN_ELU, distillation_crn
    cfg, seed, student = CONFIGS[tag]
    cls = distillation_crn.TemporalCRN if student else CRN_ELU.TemporalCRN
    model = cls(segment_length=3200, dropout=0.0, precision=precision, **cfg, **kw)
    w = synth.make_crn_weights(seed=seed, **cfg)
    sd = {k: torch.from_numpy(v) for k, v in synth.with_alias_keys(w).items()}
    missing, unexpected = model.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    return model.eval()


def oracle_stream_steps(oracle, chunks, model):
    """The oracle's streaming steps over `chunks` (each [D, 3, 3200], CPU) from a reset state: the concatenated outputs
    [D, 1600 * len(chunks)] and a bool mask [D] of the streams on the atan2 branch cut.

    The reference's phase feature is an UNWRAPPED atan2 (CRN_ELU.py:370-371): a bin on the negative real axis whose
    imaginary part is rounding noise (e.g. 1.8e-7 vs -8.5e-8 next to a spectrum peak of 48) gets +pi or -pi depending on
    the last bit of the FFT, and the feature jumps by 2 pi.  Both results are valid roundings of the same signal, but such
    a stream cannot be compared at the fp32 tolerance: streams whose two spectra (the oracle's and `model.stft_trans`,
    asserted within 1e-6 of the peak of each other) land on different sides of the cut are flagged, and callers hold
    them to the fp16 tolerance instead.  At most ONE of a handful of streams may sit on the cut (observed: one, depending
    on the FFT's last bit); more would mean the transform itself has drifted, not the cut."""
    D = chunks[0].shape[0]
    with torch.no_grad():
        oracle.reset()
        state = None
        want = []
        on_cut = torch.zeros(D, dtype=torch.bool)
        for c in chunks:
            xo = oracle.stft_trans(c)
            xc = model.stft_trans(c.cuda()).cpu()
            assert (xo - xc).abs().max() < 1e-6 * xo.abs().max()
            jump = (torch.atan2(xo[..., 1], xo[..., 0]) - torch.atan2(xc[..., 1], xc[..., 0])).abs() > 3.0
            on_cut |= jump.flatten(1).any(1)
            y, state = oracle.stream_step(c, state)
            want.append(y.numpy())
    print(f"streams on the atan2 branch cut (held to the fp16 tolerance in fp32): {np.flatnonzero(on_cut.numpy()).tolist()}")
    assert int(on_cut.sum()) <= 1
    return np.concatenate(want, axis=-1), on_cut.numpy()


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


DISTILL_TEACHER = dict(num_channels=[16, 32, 32, 48], num_freqs=201, hidden=64, num_layers=2, num_inputs=3, kernel_size=3)


def distill_weights():
    """Teacher (seed 21) and student (seed 22) weights of tests/golden/distill.npz after the reference's parameter
    aliasing (distillation_crn.py:527-529: parameters are zipped in registration order and a student parameter with the
    teacher's shape SHARES its storage; the fixture loads the teacher first, so both end up with the student's values)."""
    wt = synth.make_crn_weights(seed=21, **DISTILL_TEACHER)
    ws = synth.make_crn_weights(seed=22, **STUDENT)
    for kt, ks in zip(wt, ws):
        if wt[kt].shape == ws[ks].shape:
            wt[kt] = ws[ks].copy()
    return wt, ws


def distill_setup(g):
    """Oracle teacher / student, the connector parameters stored in the fixture and the first piece's data."""
    wt, ws = distill_weights()
    teacher = CRNOracle({k: torch.from_numpy(v) for k, v in wt.items()}, segment_length=3200, student=True,
                        **DISTILL_TEACHER)
    student = CRNOracle({k: torch.from_numpy(v) for k, v in ws.items()}, segment_length=3200, student=True, **STUDENT)
    connectors = [(torch.from_numpy(g[f"connector/{i}.0.weight"]), torch.from_numpy(g[f"connector/{i}.1.weight"]),
                   torch.from_numpy(g[f"connector/{i}.1.bias"])) for i in range(5)]
    mix, src = synth.make_mixture(2, 4000)
    return teacher, student, connectors, (mix, src, [4000, 3300])
