"""GPU: the gated skip path of the 32- and 64-channel decoder levels as one tcgen05 launch (skip_blend_tc.cu).

In fp16 inference, decoder levels 0 and 1 run their residual-mask / residual 1x1 pair, both GlobalLayerNorms and the
skip blend in `skip_blend_tc_kernel`, one stream per CTA at a time with the CTAs striding over the streams.  A launch
guard proves the fp16 step runs it (and neither the skip-pair kernels nor the blend kernel it replaces) while the tf32
step does not.  The block-level check recomputes each level in float64 with the oracle's transposed-conv block
(CRNOracle._tdeconv) from the tensors the step left in the context -- the level's input, its skip tensor -- and
compares the level's output, for batches of one stream, of one stream past a full round of CTAs and of three rounds."""
import ctypes as C

import numpy as np
import pytest
import torch

from common import make_model, make_oracle
from oracle import synth
from test_stream_counts_gpu import launches, profiled_step

pytestmark = pytest.mark.gpu

# The reference runs in float64 on the same fp16 inputs, so what remains is the fp16 rounding (2^-11 relative) of the
# weights, of the deconv output y and of the stored block output.  Measured worst case on one B200 (teacher and student,
# both levels, every checked stream): 7.4e-4 x peak; the tolerance leaves a factor of about 13 above that.
TOL = 1e-2  # x max(1, peak of the reference output)


def read(model, name, b):
    from speech_enhancement_mi_b200._native import check, lib
    buf = np.zeros(1 << 20, dtype=np.float32)
    dims = (C.c_int * 3)()
    check(lib().se_debug_read(model._ctx, name.encode(), b, buf.ctypes.data, buf.size, dims), "se_debug_read")
    return buf[: dims[0] * dims[1] * dims[2]].reshape(dims[0], dims[1], dims[2])  # [T][F][C]


def chunk(B):
    """One 3200-sample chunk per stream: 8 distinct mixtures, replicated with a per-stream gain so that no two streams
    of a CTA's rounds carry the same data."""
    mix, _ = synth.make_mixture(8, 3200)
    gain = (1.0 + 0.05 * np.arange(B, dtype=np.float32))[:, None, None]
    return torch.from_numpy(np.ascontiguousarray(mix[np.arange(B) % 8] * gain, dtype=np.float32))


@pytest.mark.parametrize("tag", ["crn_teacher", "crn_student"])
def test_fp16_step_runs_the_fused_skip_blend(tag):
    model = make_model(tag, "fp16")
    _, counts = profiled_step(model, chunk(4).cuda())
    assert launches(counts, "skip_blend_tc_kernel") == 2, counts
    assert sum(n for k, n in counts.items() if "norm_apply_h8_kernel<2>" in k) == 0, counts
    assert sum(n for k, n in counts.items() if "skip_small" in k) == 0, counts
    model = make_model(tag, "tf32")
    _, counts = profiled_step(model, chunk(4).cuda())
    assert launches(counts, "skip_blend_tc_kernel") == 0, counts


def level_ref(oracle, j, x, res):
    """Decoder level j in float64 from [T][F][C] input and skip tensors -> [T][F][C]."""
    xt = torch.from_numpy(x).double().permute(2, 1, 0)[None]    # [1, C, F, T]
    rt = torch.from_numpy(res).double().permute(2, 1, 0)[None]
    with torch.no_grad():
        y = oracle._tdeconv(f"deconvlist.{j}", xt, 2 ** j, rt)
    return y[0].permute(2, 1, 0).numpy()


@pytest.mark.parametrize("B", [1, 149, 297])
@pytest.mark.parametrize("tag", ["crn_teacher", "crn_student"])
def test_skip_blend_levels_match_float64_block(tag, B):
    oracle, _ = make_oracle(tag)
    oracle.w = {k: v.double() for k, v in oracle.w.items()}
    model = make_model(tag, "fp16")
    with torch.no_grad():
        model.process_chunk(chunk(B).cuda())
    torch.cuda.synchronize()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    streams = sorted({0, B - 1} | {b for b in (sms, 2 * sms, B - 1 - sms) if 0 <= b < B})
    worst = {}
    for j, (xin, skip, out) in enumerate([("dec_in0", "enc_in3", "dec_in1"), ("dec_in1", "enc_in2", "dec_in2")]):
        for b in streams:
            want = level_ref(oracle, j, read(model, xin, b), read(model, skip, b))
            got = read(model, out, b)
            assert got.shape == want.shape
            err = float(np.abs(got - want).max()) / max(1.0, float(np.abs(want).max()))
            worst[(j, b)] = err
    assert max(worst.values()) < TOL, f"{tag} B={B}: worst error x peak per (level, stream): {worst}"
    print(f"{tag} B={B}: worst {max(worst.values()):.2e}")
