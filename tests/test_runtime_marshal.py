"""What the numpy wrappers of runtime.py hand to the C ABI, checked without a GPU: ``runtime._call`` (their one way to the
library) is replaced by a recorder.  Batches arrive in CSR form (one concatenated array + int32 offsets), a one-item
batch is passed without a copy, selection masks arrive as 0 / 1 bytes whatever their dtype, and malformed arguments
raise ValueError before the library is reached."""
import numpy as np
import pytest

THR2 = (1.5 / 3217.0) ** 2


@pytest.fixture
def rt(rg):
    return rg.runtime


@pytest.fixture
def calls(rg, rt, monkeypatch):
    """The (name, device, args) of every library call the wrappers make; outputs are left as allocated.  Each argument
    list is checked against the entry point's ctypes prototype (count and types, context handle first)."""
    cabi = rg._cabi
    cabi.load_library()
    seen = []

    def record(name, device, *args):
        fn, conv = cabi._calls[name]
        assert len(args) + 1 == len(fn.argtypes), name
        for argtype, c, a in zip(fn.argtypes, conv, (0,) + args):
            argtype.from_param(c(a))
        seen.append((name, device, args))
    monkeypatch.setattr(rt, "_call", record)
    return seen


@pytest.fixture
def no_calls(rt, monkeypatch):
    def fail(name, *_):
        raise AssertionError(f"{name} reached the library")
    monkeypatch.setattr(rt, "_call", fail)


def _rows(rng, n, w):
    return rng.standard_normal((n, w))


def _idx(rng, h, k, n):
    return rng.integers(0, n, (h, k)).astype(np.int32)


def _csr(arrays, tail, dtype):
    off = np.concatenate([[0], np.cumsum([len(a) for a in arrays])]).astype(np.int32)
    flat = np.concatenate(arrays).astype(dtype) if arrays else np.zeros((0,) + tail, dtype)
    return flat, off


def _same(got, want):
    assert got.dtype == want.dtype and got.shape == want.shape and np.array_equal(got, want, equal_nan=True)


# per batched wrapper: its call and, per packed input, (argument position, input list, offset table position, tail, dtype)
def _wrappers(rt, rng, sizes):
    pts = [_rows(rng, n, 4) for n in sizes]
    X = [_rows(rng, n, 3) for n in sizes]
    y = [_rows(rng, n, 2) for n in sizes]
    idx8 = [_idx(rng, 5 + k, 8, max(n, 1)) for k, n in enumerate(sizes)]
    idx6 = [_idx(rng, 7 + k, 6, max(n, 1)) for k, n in enumerate(sizes)]
    P = len(sizes)
    R, t = np.tile(np.eye(3), (P, 1, 1)), np.zeros((P, 3))
    C = np.tile(np.hstack([np.eye(3), np.zeros((3, 1))]), (P, 1, 1))
    F = np.tile(np.eye(3), (P, 1, 1))
    return {
        "f_ransac_batched": (lambda: rt.f_ransac_batched(pts, idx8),
                             [(2, pts, 3, (4,), np.float64), (4, idx8, 5, (8,), np.int32)]),
        "pnp_ransac_batched": (lambda: rt.pnp_ransac_batched(X, y, idx6, THR2),
                               [(2, X, 4, (3,), np.float64), (3, y, 4, (2,), np.float64), (6, idx6, 7, (6,), np.int32)]),
        "triangulate": (lambda: rt.triangulate(C, C, y, y), [(5, y, 4, (2,), np.float64), (6, y, 4, (2,), np.float64)]),
        "two_view_init": (lambda: rt.two_view_init(pts, F, np.eye(3)), [(2, pts, 3, (4,), np.float64)]),
        "gold_standard": (lambda: rt.gold_standard(pts, F), [(2, pts, 3, (4,), np.float64)]),
        "pnp_refine_batched": (lambda: rt.pnp_refine_batched(X, y, R, t),
                               [(2, X, 4, (3,), np.float64), (3, y, 4, (2,), np.float64)]),
    }


@pytest.mark.parametrize("sizes", [[30, 0, 17], [40], []], ids=["multi", "single", "empty"])
@pytest.mark.parametrize("name", ["f_ransac_batched", "pnp_ransac_batched", "triangulate", "two_view_init",
                                  "gold_standard", "pnp_refine_batched"])
def test_batches_are_passed_in_csr_form(rt, calls, name, sizes):
    run, packed = _wrappers(rt, np.random.default_rng(len(sizes)), sizes)[name]
    run()
    (_, _, args), = calls
    for pos, arrays, off_pos, tail, dtype in packed:
        flat, off = _csr(arrays, tail, dtype)
        _same(args[off_pos], off)
        _same(args[pos], flat)
        if len(arrays) == 1:                                   # one item: the caller's own memory, no copy
            assert args[pos].ctypes.data == arrays[0].ctypes.data


def test_device_drawn_samples_pass_offsets_only(rt, calls):
    pts = [np.zeros((n, 4)) for n in (20, 9)]
    rt.f_ransac_batched(pts, None, n_hyp=[100, 3], sample_seed=5, first_pair=2)
    (name, _, args), = calls
    assert name == "rg_f_ransac_host2" and args[4] is None
    _same(args[5], np.array([0, 100, 103], np.int32))
    assert args[11:13] == (5, 2)


def test_consecutive_blocks_of_one_buffer_are_not_copied(rg, rt, calls):
    blocks = rg.sampling.fast_batch([30, 20], 50, 8, seed=1)
    rt.f_ransac_batched([np.zeros((30, 4)), np.zeros((20, 4))], blocks)
    assert calls[0][2][4].ctypes.data == blocks[0].ctypes.data


@pytest.mark.parametrize("dtype", [np.int64, np.float64, bool])
def test_masks_select_every_nonzero_value(rt, calls, dtype):
    values = {np.int64: [0, 2, 256, 1, 0], np.float64: [0.0, 0.5, 256.0, -1.0, 0.0], bool: [0, 1, 1, 1, 0]}[dtype]
    m = np.array(values, dtype=dtype)
    pts = [np.zeros((5, 4)), np.zeros((5, 4))]
    X, y = [np.zeros((5, 3))] * 2, [np.zeros((5, 2))] * 2
    R, t = np.tile(np.eye(3), (2, 1, 1)), np.zeros((2, 3))
    rt.two_view_init(pts, np.tile(np.eye(3), (2, 1, 1)), np.eye(3), masks=[m, m[::-1]])
    rt.gold_standard(pts, np.tile(np.eye(3), (2, 1, 1)), masks=[m, m[::-1]])
    rt.pnp_refine_batched(X, y, R, t, masks=[m, m[::-1]])
    want = np.array([0, 1, 1, 1, 0] * 2, np.uint8)
    for (_, _, args), pos in zip(calls, (6, 5, 6)):
        _same(args[pos], want)


def test_pnp_ransac_is_one_view_of_the_batched_call(rt, calls):
    """pnp_ransac is built on pnp_ransac_batched, so the call comparison mainly pins n_vote = [n_sel or N], the no-copy
    inputs and the unwrapped result types.  That this one-view call computes what rg_pnp_ransac_host did rests on the C
    side: rg_pnp_ransac_host (csrc/pnp_api.cu) is a shim that calls rg_pnp_ransac_batched_host with view_off {0, N},
    n_vote {N_sel} and its other arguments unchanged."""
    rng = np.random.default_rng(3)
    X, y, idx = _rows(rng, 60, 3), _rows(rng, 60, 2), _idx(rng, 9, 6, 40)
    for n_sel, vote in ((None, 60), (40, 40)):
        calls.clear()
        one = rt.pnp_ransac(X, y, idx, THR2, n_sel=n_sel, want_counts=True, want_poses=True, want_flags=True, device=1)
        rt.pnp_ransac_batched([X], [y], [idx], THR2, n_vote=[vote], want_counts=True, want_poses=True, want_flags=True,
                              device=1)
        (n1, d1, a1), (n2, d2, a2) = calls
        assert n1 == n2 == "rg_pnp_ransac_batched_host" and d1 == d2 == 1 and len(a1) == len(a2)
        for a, b in zip(a1, a2):
            if isinstance(a, np.ndarray):
                _same(a, b)
            else:
                assert a == b
        assert a1[2].ctypes.data == X.ctypes.data and a1[3].ctypes.data == y.ctypes.data
        assert a1[6].ctypes.data == idx.ctypes.data
        assert isinstance(one["best_idx"], int) and isinstance(one["best_count"], int)
        assert one["R"].shape == (3, 3) and one["t"].shape == (3,) and one["mask"].shape == (60,)
        assert one["counts"].shape == (9,) and one["poses"].shape == (9, 12) and one["flags"].shape == (9,)


z = np.zeros
PTS, IDX8, X3, Y2, IDX6 = z((20, 4)), z((5, 8), np.int32), z((20, 3)), z((20, 2)), z((5, 6), np.int32)
R1, T1, CAM = np.eye(3)[None], z((1, 3)), z((1, 3, 4))
F1 = np.eye(3)[None]
MALFORMED = {
    "f_ransac_batched: points (N, 3)": lambda rt: rt.f_ransac_batched([z((20, 3))], [IDX8]),
    "f_ransac_batched: samples (H, 7)": lambda rt: rt.f_ransac_batched([PTS], [z((5, 7), np.int32)]),
    "f_ransac_batched: list lengths": lambda rt: rt.f_ransac_batched([PTS, PTS], [IDX8]),
    "f_ransac_batched: n_hyp length": lambda rt: rt.f_ransac_batched([PTS], None, n_hyp=[3, 4]),
    "f8pt_solve: index range": lambda rt: rt.f8pt_solve(PTS, IDX8 + 20),
    "pnp_ransac: X / y rows": lambda rt: rt.pnp_ransac(X3, Y2[:10], IDX6, THR2),
    "pnp_ransac: 1-D samples": lambda rt: rt.pnp_ransac(X3, Y2, IDX6.ravel(), THR2),
    "pnp_ransac_batched: sample widths":
        lambda rt: rt.pnp_ransac_batched([X3, X3], [Y2, Y2], [IDX6, z((5, 7), np.int32)], THR2),
    "pnp_ransac_batched: list lengths": lambda rt: rt.pnp_ransac_batched([X3], [Y2, Y2], [IDX6], THR2),
    "pnp_refine_batched: X / y rows": lambda rt: rt.pnp_refine_batched([X3], [Y2[:3]], R1, T1),
    "pnp_refine_batched: poses": lambda rt: rt.pnp_refine_batched([X3], [Y2], np.concatenate([R1, R1]), T1),
    "pnp_refine_batched: mask length": lambda rt: rt.pnp_refine_batched([X3], [Y2], R1, T1, masks=[z(19)]),
    "pnp_refine: K": lambda rt: rt.pnp_refine(X3, Y2, R1[0], T1[0], K=np.eye(4)),
    "pnp_refine: rounds without thr2": lambda rt: rt.pnp_refine(X3, Y2, R1[0], T1[0], rounds=2),
    "triangulate: x1 / x2 rows": lambda rt: rt.triangulate(CAM, CAM, [z((3, 2))], [z((4, 2))]),
    "triangulate: cameras": lambda rt: rt.triangulate(CAM, z((2, 3, 4)), [Y2], [Y2]),
    "triangulate: points (N, 3)": lambda rt: rt.triangulate(CAM, CAM, [X3], [X3]),
    "fmatrix_from_cameras: cameras": lambda rt: rt.fmatrix_from_cameras(CAM, z((2, 3, 4))),
    "relative_pose: points": lambda rt: rt.relative_pose(F1, z((2, 2)), z((1, 2))),
    "relative_pose: K": lambda rt: rt.relative_pose(F1, z((1, 2)), z((1, 2)), K=np.eye(4)),
    "two_view_init: F": lambda rt: rt.two_view_init([PTS], z((2, 3, 3)), np.eye(3)),
    "two_view_init: mask length": lambda rt: rt.two_view_init([PTS], F1, np.eye(3), masks=[z(19)]),
    "two_view_init: mask count": lambda rt: rt.two_view_init([PTS], F1, np.eye(3), masks=[z(20), z(20)]),
    "gold_standard: F0": lambda rt: rt.gold_standard([PTS], z((2, 3, 3))),
    "gold_standard: mask length": lambda rt: rt.gold_standard([PTS], F1, masks=[z(21)]),
    "bundle_adjust: observations": lambda rt: rt.bundle_adjust(z((1, 3, 4)), z((2, 3)), z((4, 2)), z(4), z(3)),
    "ba_residuals: parameters": lambda rt: rt.ba_residuals(z(10), z(2), z(2), z(2), z(2), 1, 0),
    "match_first_within: queries": lambda rt: rt.match_first_within(z((3, 2)), z(5)),
}


@pytest.mark.parametrize("case", MALFORMED)
def test_malformed_arguments_raise_before_the_library(rt, no_calls, case):
    with pytest.raises(ValueError):
        MALFORMED[case](rt)


def test_offsets_refuse_int32_overflow(rg):
    assert rg.device.offsets is rg.runtime.offsets
    _same(rg.runtime.offsets([3, 0, 4]), np.array([0, 3, 3, 7], np.int32))
    with pytest.raises(ValueError):
        rg.runtime.offsets([2 ** 30, 2 ** 30])
