"""GPU: export / import of per-stream streaming state (TemporalCRN / FullSubNet .export_state / .import_state behind
se_crn_state_export / _import and se_fsn_state_export / _import).

A record must hold everything the next step of a stream reads.  Every continuation below imports into DIRTY rows (rows
that just served other audio and were not reset), so a piece of state missing from the record shows up as a different
output instead of hiding behind a zero row; and states are taken after one chunk and mid-stream after several.

Bitwise checks: a CRN stream is bitwise reproducible under the same batch geometry (same rows, same B).  A FullSubNet
step accumulates its CumLayerNorm sums with double atomics in no fixed order, so its outputs are held to the replica
tolerance of test_fsn_stream_gpu.py even there (the records themselves are compared bit for bit).  Moved rows or another
B are held to the replica tolerances of test_stream_counts_gpu.py / test_fsn_stream_counts_gpu.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from common import FSN_FULL, FSN_SMALL, make_fsn, make_model

pytestmark = pytest.mark.gpu

K = 3200
REP_TOL = {"fp32": 2e-5, "tf32": 2e-3, "3xtf32": 2e-5, "fp16": 2e-3, "fsn": 1e-5}  # x max(1, peak)
FSN_CFGS = {"small": (FSN_SMALL, 11), "small64": (dict(FSN_SMALL, sb_hidden=64), 11), "full": (FSN_FULL, 5)}


def model_of(kind, tag, precision, max_streams):
    if kind == "crn":
        return make_model(tag, precision, max_streams=max_streams)
    cfg, seed = FSN_CFGS[tag]
    return make_fsn(cfg, seed, max_streams=max_streams, precision=precision)


def chunks(B, n, seed):
    """n chunks [B, 3, 3200] on cuda:0: noise plus a per-stream tone, so that streams differ."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(K * n, dtype=torch.float32) / 16000
    f0 = 200 + 1800 * torch.rand(B, 1, 1, generator=g)
    x = 0.3 * torch.sin(2 * np.pi * f0 * t) + 0.1 * torch.randn(B, 3, K * n, generator=g)
    return [x[:, :, i * K:(i + 1) * K].contiguous().cuda() for i in range(n)]


def run(model, cs):
    return np.concatenate([model.process_chunk(c).cpu().numpy() for c in cs], axis=-1)


def tol(kind, precision):
    return REP_TOL["fsn" if kind == "fsn" else precision]


def assert_same(got, want, kind, what=""):
    """bitwise for the CRN; the FullSubNet replica tolerance (see the module docstring)"""
    if kind == "crn":
        assert np.array_equal(got, want), f"{what}: max |diff| {np.abs(got - want).max():.3e}"
    else:
        peak = max(1.0, float(np.abs(want).max()))
        assert np.abs(got - want).max() < REP_TOL["fsn"] * peak, what


def assert_close(got, want, kind, precision, what=""):
    peak = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(got - want).max())
    assert err < tol(kind, precision) * peak, f"{what}: {err:.3e} vs peak {peak:.3f}"


def records(state):
    return state.data.cpu().numpy()


# ---- 1. record round trip -------------------------------------------------------------------------------------------
ROUND_TRIP = [("crn", t, p) for t in ("crn_small", "crn_teacher", "crn_student") for p in ("fp32", "tf32", "fp16", "3xtf32")]
ROUND_TRIP += [("fsn", "small", "tf32"), ("fsn", "small", "3xtf32"), ("fsn", "small64", "fp16"), ("fsn", "full", "tf32"),
               ("fsn", "full", "fp16")]


@pytest.mark.parametrize("kind,tag,precision", ROUND_TRIP, ids=["-".join(c) for c in ROUND_TRIP])
def test_record_round_trip_is_byte_identical(kind, tag, precision):
    B = 6
    a = model_of(kind, tag, precision, 8)
    run(a, chunks(B, 3, 1))
    rows = [4, 0, 5, 2, 1, 3]
    sa = a.export_state(rows)
    assert sa.data.dtype == torch.uint8 and tuple(sa.data.shape) == (B, sa.data.shape[1])
    assert sa.data.shape[1] % 16 == 0
    b = model_of(kind, tag, precision, 13)  # another capacity: other unit-major strides, same records
    run(b, chunks(B + 3, 2, 2))  # dirty rows
    dst = [7, 11, 0, 2, 9, 3]
    b.import_state(sa, dst)
    sb = b.export_state(dst)
    assert sb.layout == sa.layout
    assert np.array_equal(records(sb), records(sa))
    assert records(sa).any(axis=1).all(), "a stream that has run carries non-zero state"


@pytest.mark.parametrize("kind,tag", [("crn", "crn_small"), ("fsn", "small")])
def test_layout_separates_precisions(kind, tag):
    layouts = {}
    for p in ("tf32", "3xtf32") + (("fp32",) if kind == "crn" else ()):
        m = model_of(kind, tag, p, 4)
        run(m, chunks(2, 1, 3))
        layouts[p] = m.export_state([0]).layout
    assert len(set(layouts.values())) == len(layouts), layouts


# ---- 2. continuation, same geometry -----------------------------------------------------------------------------------
CONT = [("crn", "crn_teacher", "fp16", {}), ("crn", "crn_teacher", "tf32", {}), ("crn", "crn_small", "fp32", {}),
        ("crn", "crn_student", "fp16", {}), ("crn", "crn_small", "fp16", {"SE_B200_FRONT_MMA": "0"}),
        ("crn", "crn_small", "fp16", {"SE_B200_FRONT_MMA": "0", "SE_B200_PRECONV_TC": "0"}),
        ("fsn", "small", "tf32", {}), ("fsn", "small64", "fp16", {})]


@pytest.mark.parametrize("k", [1, 5])
@pytest.mark.parametrize("kind,tag,precision,env", CONT,
                         ids=["-".join([c[0], c[1], c[2]] + [f"{a}={v}" for a, v in c[3].items()]) for c in CONT])
def test_continuation_same_geometry(monkeypatch, kind, tag, precision, env, k):
    for name, v in env.items():
        monkeypatch.setenv(name, v)
    B = 12
    a = model_of(kind, tag, precision, 16)
    b = model_of(kind, tag, precision, 40)
    run(a, chunks(B, k, 10 + k))
    run(b, chunks(B, 3, 99))  # rows of b are dirty
    b.import_state(a.export_state(range(B)), torch.arange(B))
    nxt = chunks(B, 3, 20 + k)
    assert_same(run(b, nxt), run(a, nxt), kind, "continuation in another context")


# ---- 3. continuation, moved rows at another B --------------------------------------------------------------------------
@pytest.mark.parametrize("kind,tag,precision", [("crn", "crn_teacher", "fp16"), ("crn", "crn_teacher", "fp32"),
                                                ("fsn", "small", "tf32")])
def test_continuation_moved_rows_other_batch(kind, tag, precision):
    B, B2 = 300, 340  # more streams than one GRU wave / one 128-row tile; B2 another geometry
    a = model_of(kind, tag, precision, 512)
    b = model_of(kind, tag, precision, 512)
    run(a, chunks(B, 4, 30))
    run(b, chunks(B2, 2, 31))
    perm = torch.randperm(B2, generator=torch.Generator().manual_seed(5))[:B]
    b.import_state(a.export_state(range(B)), perm)
    nxt = chunks(B, 3, 32)
    want = run(a, nxt)
    other = chunks(B2, 3, 33)
    moved = []
    for c, o in zip(nxt, other):
        x = o.clone()
        x[perm.cuda()] = c
        moved.append(x)
    got = run(b, moved)[perm.numpy()]
    assert_close(got, want, kind, precision, "moved rows")


# ---- 4. compaction ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,tag,precision", [("crn", "crn_small", "fp32"), ("crn", "crn_student", "fp16"),
                                                ("fsn", "small", "tf32")])
def test_compaction_moves_tail_into_holes(kind, tag, precision):
    B = 300
    live = model_of(kind, tag, precision, 512)
    ref = model_of(kind, tag, precision, 512)
    first = chunks(B, 3, 40)
    run(live, first)
    run(ref, first)
    rng = np.random.default_rng(6)
    ended = np.sort(rng.choice(B, B // 3, replace=False))
    survivors = np.setdiff1d(np.arange(B), ended)
    n = len(survivors)
    holes = [int(r) for r in ended if r < n]
    tail = [int(r) for r in survivors if r >= n]
    assert len(holes) == len(tail) > 0
    keep = [int(r) for r in survivors if r < n]
    before = records(live.export_state(keep))
    live.import_state(live.export_state(tail), holes)
    assert np.array_equal(records(live.export_state(keep)), before), "rows that were not touched keep their state"
    slot = np.arange(B)  # stream -> row after compaction
    slot[tail] = holes
    nxt = chunks(B, 3, 41)
    want = run(ref, nxt)[survivors]
    order = np.argsort(slot[survivors])  # survivors by new row
    idx = torch.from_numpy(survivors[order]).cuda()
    got = np.empty_like(want)
    got[order] = run(live, [c[idx] for c in nxt])
    assert_close(got, want, kind, precision, "compacted streams")


# ---- 5. export is read-only -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,tag,precision", [("crn", "crn_teacher", "fp16"), ("fsn", "small64", "fp16")])
def test_export_is_read_only(kind, tag, precision):
    B = 10
    a = model_of(kind, tag, precision, 16)
    twin = model_of(kind, tag, precision, 16)
    cs = chunks(B, 3, 50)
    run(a, cs)
    run(twin, cs)
    s1 = a.export_state([3, 3, 0, 9, 3])  # repeats are allowed on export
    s2 = a.export_state(range(B))
    assert np.array_equal(records(s1)[0], records(s1)[1]) and np.array_equal(records(s1)[0], records(s2)[3])
    assert np.array_equal(records(a.export_state(range(B))), records(s2))
    nxt = chunks(B, 2, 51)
    assert_same(run(a, nxt), run(twin, nxt), kind, "source after export")


# ---- 6. host checkpoint -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,tag,precision", [("crn", "crn_teacher", "fp16"), ("fsn", "small", "tf32")])
def test_host_checkpoint_resumes(tmp_path, kind, tag, precision):
    B = 8
    a = model_of(kind, tag, precision, 8)
    run(a, chunks(B, 4, 60))
    st = a.export_state(range(B))
    np.save(tmp_path / "state.npy", st.data.cpu().numpy())
    (tmp_path / "layout.txt").write_text(str(st.layout))
    b = model_of(kind, tag, precision, 8)
    run(b, chunks(B, 1, 61))  # dirty
    state = type(st)(int((tmp_path / "layout.txt").read_text()), torch.from_numpy(np.load(tmp_path / "state.npy")))
    b.import_state(state, range(B))
    nxt = chunks(B, 3, 62)
    assert_same(run(b, nxt), run(a, nxt), kind, "resumed from a host checkpoint")


# ---- 7. growth --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,tag,precision", [("crn", "crn_student", "fp16"), ("crn", "crn_small", "tf32"),
                                                ("fsn", "small64", "fp16")])
def test_growth_into_a_larger_model(kind, tag, precision):
    B = 48
    small = model_of(kind, tag, precision, 64)
    run(small, chunks(B, 3, 70))
    st = small.export_state(range(B))
    big = model_of(kind, tag, precision, 256)
    big.import_state(st, range(B))  # creates the context
    assert big._ctx_capacity == 256
    nxt = chunks(B, 3, 71)
    assert_same(run(big, nxt), run(small, nxt), kind, "grown model")


def test_import_creates_a_context_large_enough():
    a = model_of("crn", "crn_small", "fp32", 4)
    run(a, chunks(4, 1, 72))
    m = model_of("crn", "crn_small", "fp32", 2)
    m.import_state(a.export_state([0, 1]), [5, 9])
    assert m._ctx_capacity == 10 and not m._fresh


# ---- 8. cross-GPU -----------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("kind,tag,precision", [("crn", "crn_teacher", "fp16"), ("fsn", "small", "tf32")])
def test_cross_gpu_migration(kind, tag, precision):
    B = 16
    a = model_of(kind, tag, precision, 16)
    run(a, chunks(B, 3, 80))
    st = a.export_state(range(B))
    moved = type(st)(st.layout, st.data.to("cuda:1"))
    b = model_of(kind, tag, precision, 32)
    b.import_state(moved, range(B))
    assert b._ctx_device == 1
    nxt = chunks(B, 3, 81)
    got = np.concatenate([b.process_chunk(c.to("cuda:1")).cpu().numpy() for c in nxt], axis=-1)
    assert_close(got, run(a, nxt), kind, precision, "stream moved to cuda:1")


# ---- 9. captured step graphs see imported state -----------------------------------------------------------------------
@pytest.mark.parametrize("kind,tag,precision", [("crn", "crn_teacher", "fp16"), ("fsn", "small", "tf32")])
def test_captured_graph_sees_imported_state(kind, tag, precision):
    B = 12
    a = model_of(kind, tag, precision, 16)
    src = model_of(kind, tag, precision, 16)
    run(a, chunks(B, 3, 90))  # graph for B captured and replayed
    run(src, chunks(B, 4, 91))
    a.import_state(src.export_state(range(B)), range(B))
    nxt = chunks(B, 2, 92)
    assert_same(run(a, nxt), run(src, nxt), kind, "replayed graph after import")


# ---- 10. errors -------------------------------------------------------------------------------------------------------
def test_layout_mismatch_is_rejected():
    from speech_enhancement_mi_b200._native import lib
    pairs = [(("crn", "crn_teacher", "tf32"), ("crn", "crn_teacher", "fp16")),
             (("crn", "crn_teacher", "fp16"), ("crn", "crn_student", "fp16")),
             (("crn", "crn_small", "tf32"), ("fsn", "small", "tf32"))]
    for src_cfg, dst_cfg in pairs:
        src = model_of(*src_cfg, 4)
        run(src, chunks(2, 1, 100))
        st = src.export_state([0, 1])
        dst = model_of(*dst_cfg, 4)
        run(dst, chunks(2, 1, 101))
        with pytest.raises(ValueError, match="layout"):
            dst.import_state(st, [0, 1])
        # the native check, for C-ABI callers
        fn = lib().se_crn_state_import if dst_cfg[0] == "crn" else lib().se_fsn_state_import
        rows = (C.c_int32 * 2)(0, 1)
        assert fn(dst._ctx, rows, 2, C.c_void_p(st.data.data_ptr()), C.c_uint64(st.layout), None) != 0
        assert b"layout mismatch" in lib().se_last_error()


@pytest.mark.parametrize("kind,tag,precision", [("crn", "crn_small", "fp32"), ("fsn", "small", "tf32")])
def test_bad_rows_and_sizes_are_rejected(kind, tag, precision):
    m = model_of(kind, tag, precision, 4)
    run(m, chunks(2, 1, 110))
    with pytest.raises(RuntimeError, match="outside"):
        m.export_state([0, 4])
    st = m.export_state([1, 0])
    with pytest.raises(RuntimeError, match="outside"):
        m.import_state(st, [-1, 0])
    with pytest.raises(RuntimeError, match="appears twice"):
        m.import_state(st, [2, 2])
    with pytest.raises(ValueError, match="record size"):
        m.import_state(type(st)(st.layout, st.data[:, :-16]), [0, 1])
    with pytest.raises(ValueError, match="records for"):
        m.import_state(st, [0])


def test_training_context_is_rejected():
    from speech_enhancement_mi_b200._native import lib
    m = model_of("crn", "crn_small", "fp32", 4)
    cfg = m._config(4, training=True)
    ctx = C.c_void_p()
    assert lib().se_ctx_create(C.byref(ctx), 0, C.byref(cfg)) == 0
    try:
        buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda:0")
        rows = (C.c_int32 * 1)(0)
        assert lib().se_crn_state_export(ctx, rows, 1, C.c_void_p(buf.data_ptr()), None) != 0
        assert b"training" in lib().se_last_error()
        assert lib().se_crn_state_import(ctx, rows, 1, C.c_void_p(buf.data_ptr()), C.c_uint64(0), None) != 0
        assert b"training" in lib().se_last_error()
    finally:
        lib().se_ctx_destroy(ctx)


def test_chunk_batch_state_owner_cannot_export():
    m = model_of("crn", "crn_small", "fp32", 4)
    g = torch.Generator().manual_seed(120)
    with torch.no_grad():
        m.realtime_process(0.1 * torch.randn(1, 3, 16000, generator=g).cuda())
    assert m._state_owner == "chunk-batch"
    with pytest.raises(RuntimeError, match="chunk-batch"):
        m.export_state([0])
