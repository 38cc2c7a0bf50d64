"""Device-resident entry points (the ``_dev`` half of the C ABI) for callers that keep their batches in HBM.

torch is used ONLY as a carrier of device memory and streams (``data_ptr()`` / ``current_stream()``); every kernel that
runs is in librg_b200.so.  All calls are asynchronous on torch's current stream.  ``parallel.py`` builds the multi-GPU
decompositions on top of these, ``bench.py`` times them.
"""
from __future__ import annotations

import contextlib

import numpy as np

from . import _cabi as cabi
from ._cabi import FLAG_BOUNDED, FLAG_REUSE_POINTS, MODE_EPI_MAX, SCORE_FP32_GUARDED, SOLVER_QR, TIE_FIRST
from .runtime import offsets, pnp_k_table  # noqa: F401  (offsets: part of this module's interface)


def _torch():
    import torch
    return torch


def _stream():
    return _torch().cuda.current_stream().cuda_stream


def _dev_index(t) -> int:
    return int(t.device.index if t.device.index is not None else _torch().cuda.current_device())


def _cuda_device(device=None):
    """torch.device of CUDA device ``device`` (default: the current one)."""
    torch = _torch()
    return torch.device("cuda", torch.cuda.current_device() if device is None else int(device))


def _call(name, device: int, *args) -> None:
    """Entry point ``name`` with the context of CUDA device ``device`` and torch's current stream as its first two
    arguments."""
    cabi.call(name, cabi.context(device), _stream(), *args)


def synth_two_view(P: int, N: int, first_pair: int = 0, seed_base: int = 1000, cams=None, bbox=None, outlier_frac: float = 0.3,
                   sigma_px: float = 0.5, image_size=(640.0, 480.0), device=None, out=None):
    """(P, N, 4) float64 CUDA tensor: the synthetic pairs ``first_pair .. first_pair + P`` of BASELINE config 5, generated
    on the device (rg_synth_two_view_dev); ``philox.synth_two_view`` replays any of them on the host.  Also returns the
    (P, 2) int32 tensor of the camera pairs drawn."""
    torch = _torch()
    from . import synth
    dev = _cuda_device(device)
    cams = np.ascontiguousarray(synth.dino()["Ps"] if cams is None else cams, dtype=np.float64).reshape(-1, 12)
    bbox = np.ascontiguousarray(synth.DINO_BBOX if bbox is None else bbox, dtype=np.float64).reshape(6)
    pts = out if out is not None else torch.empty((P, N, 4), dtype=torch.float64, device=dev)
    cam_pair = torch.empty((P, 2), dtype=torch.int32, device=dev)
    done = 0
    while done < P:                                       # grid.y is limited to 65535 pairs per launch
        n = min(P - done, 32768)
        _call("rg_synth_two_view_dev", dev.index, n, first_pair + done, N, cams, cams.shape[0], bbox, seed_base,
              outlier_frac, sigma_px, image_size[0], image_size[1], pts[done:], cam_pair[done:])
        done += n
    return pts, cam_pair


def sample_indices(n_points_list, n_hyp, k: int = 8, seed: int = 0, first_pair: int = 0, hyp_first: int = 0, device=None):
    """(sum H, k) int32 CUDA tensor of the index sets a seeded call draws (rg_sample_indices_dev)."""
    torch = _torch()
    dev = _cuda_device(device)
    n_pts = np.ascontiguousarray(n_points_list, dtype=np.int32).ravel()
    P = n_pts.size
    hyp_off = offsets(np.full(P, n_hyp) if np.isscalar(n_hyp) else n_hyp)
    out = torch.empty((int(hyp_off[-1]), k), dtype=torch.int32, device=dev)
    _call("rg_sample_indices_dev", dev.index, P, n_pts, hyp_off, k, seed, first_pair, hyp_first, out)
    return out


class FOutputs:
    """Device output buffers of a batched F-RANSAC call over P pairs (allocated once, reused across calls)."""

    def __init__(self, P: int, n_total: int = 0, device=None, want_mask: bool = False, want_key: bool = False):
        torch = _torch()
        dev = _cuda_device(device)
        # one contiguous block per pair: [best_idx i32][best_count i32][F 9 x f64] is what the pair-sharded gather ships
        self.best_idx = torch.empty(max(P, 1), dtype=torch.int32, device=dev)
        self.best_count = torch.empty(max(P, 1), dtype=torch.int32, device=dev)
        self.F = torch.empty((max(P, 1), 9), dtype=torch.float64, device=dev)
        self.mask = torch.empty(max(n_total, 1), dtype=torch.uint8, device=dev) if want_mask else None
        self.key = torch.empty(max(P, 1), dtype=torch.int64, device=dev) if want_key else None
        self.P = P


def f_ransac(d_pts, pair_off, d_idx, hyp_off, out: FOutputs, thr=1.5, mode=MODE_EPI_MAX, tie_mode=TIE_FIRST, solver=SOLVER_QR,
             score_path=SCORE_FP32_GUARDED, flags=FLAG_BOUNDED, seed=0, first_pair=0, hyp_first=0):
    """rg_f_ransac_dev2 on CUDA tensors.  d_idx None = samples drawn on the device from ``seed``.  The default flags ask for
    the bounded sweep (option 12 decides whether it runs): the results are those of the full sweep, only the per-hypothesis
    counts behind ``rg_f_last_hypotheses_dev`` are not kept."""
    _call("rg_f_ransac_dev2", _dev_index(d_pts), len(pair_off) - 1, d_pts, pair_off, d_idx, hyp_off, thr, mode, tie_mode,
          solver, score_path, flags, seed, first_pair, hyp_first, out.best_idx, out.best_count, out.F, out.mask, out.key)
    return out


def f_inlier_mask(d_pts, pair_off, d_F, thr=1.5, mode=MODE_EPI_MAX, out=None):
    """uint8 inlier mask of one F per pair (reference criterion), all on the device."""
    torch = _torch()
    if out is None:
        out = torch.empty(max(int(pair_off[-1]), 1), dtype=torch.uint8, device=d_pts.device)
    _call("rg_f_inlier_mask_dev", _dev_index(d_pts), len(pair_off) - 1, d_pts, pair_off, d_F, thr, mode, out)
    return out


class PnpOutputs:
    def __init__(self, V: int, n_total: int = 0, device=None, want_mask: bool = False, want_key: bool = False):
        torch = _torch()
        dev = _cuda_device(device)
        self.best_idx = torch.empty(max(V, 1), dtype=torch.int32, device=dev)
        self.best_count = torch.empty(max(V, 1), dtype=torch.int32, device=dev)
        self.Rt = torch.empty((max(V, 1), 12), dtype=torch.float64, device=dev)
        self.mask = torch.empty(max(n_total, 1), dtype=torch.uint8, device=dev) if want_mask else None
        self.key = torch.empty(max(V, 1), dtype=torch.int64, device=dev) if want_key else None


def pnp_ransac(d_X, d_y, view_off, d_idx, hyp_off, out: PnpOutputs, thr2, n=6, n_vote=None, score_path=SCORE_FP32_GUARDED,
               hyp_first=0):
    """rg_pnp_ransac_batched_dev2 on CUDA tensors."""
    vote = None if n_vote is None else np.ascontiguousarray(n_vote, dtype=np.int32)
    _call("rg_pnp_ransac_batched_dev2", _dev_index(d_X), len(view_off) - 1, d_X, d_y, view_off, vote, d_idx, hyp_off, n,
          thr2, score_path, hyp_first, out.best_idx, out.best_count, out.Rt, out.mask, out.key)
    return out


def _check_dense(t, name, dtype, tail=(), rows=None):
    """The kernels index raw device pointers: a tensor must be a contiguous CUDA tensor of the expected dtype and shape
    (a strided view, e.g. torch.from_numpy of a Fortran-ordered array, would be read in the wrong order)."""
    torch = _torch()
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.is_contiguous()):
        raise ValueError(f"{name} must be a contiguous CUDA tensor of dtype {dtype}")
    if tuple(t.shape[1:]) != tuple(tail) or (rows is not None and t.shape[0] < rows):
        raise ValueError(f"{name} must have shape (>= {rows}, {', '.join(map(str, tail))})" if tail else
                         f"{name} must have at least {rows} elements")


class PnpRefineOutputs:
    """Device outputs of pnp_refine: per view cost (float64), iters and status (int32)."""

    def __init__(self, V: int, device=None):
        torch = _torch()
        dev = _cuda_device(device)
        self.cost = torch.empty(max(V, 1), dtype=torch.float64, device=dev)
        self.iters = torch.empty(max(V, 1), dtype=torch.int32, device=dev)
        self.status = torch.empty(max(V, 1), dtype=torch.int32, device=dev)


def pnp_refine(d_X, d_y, view_off, out: PnpOutputs, d_mask=None, K=None, max_iter=50, ftol=1e-12, rounds=1, thr2=None,
               mask_out=None, res: PnpRefineOutputs | None = None):
    """rg_pnp_refine_dev: refines ``out.Rt`` IN PLACE on the current stream (Levenberg-Marquardt on the reprojection
    error, see runtime.pnp_refine_batched).  ``pnp_ransac(...)`` then ``pnp_refine(..., d_mask=out.mask)`` is the chained
    form: no host synchronisation between the two.  K: HOST (3, 3) or (V, 3, 3) array (validated before anything is
    enqueued).  mask_out (uint8 CUDA tensor, may be out.mask) receives the last consensus (needs thr2).  Returns ``res``
    (allocated when None)."""
    V = len(view_off) - 1
    if int(rounds) > 1 and thr2 is None:
        raise ValueError("rounds > 1 needs thr2 (the consensus threshold)")
    if mask_out is not None and thr2 is None:
        raise ValueError("mask_out needs thr2 (the consensus threshold)")
    torch = _torch()
    n = int(view_off[-1]) if V else 0
    _check_dense(d_X, "d_X", torch.float64, (3,), n)
    _check_dense(d_y, "d_y", torch.float64, (2,), n)
    _check_dense(out.Rt, "out.Rt", torch.float64, (12,), V)
    if d_mask is not None:
        _check_dense(d_mask.reshape(-1), "d_mask", torch.uint8, (), n)
    if mask_out is not None:
        _check_dense(mask_out.reshape(-1), "mask_out", torch.uint8, (), n)
    Kt = pnp_k_table(K, V)
    if res is None:
        res = PnpRefineOutputs(V, device=_dev_index(d_X))
    _call("rg_pnp_refine_dev", _dev_index(d_X), V, d_X, d_y, view_off, Kt, d_mask, out.Rt, max_iter, ftol, rounds,
          0.0 if thr2 is None else thr2, mask_out, res.cost, res.iters, res.status)
    return res


class P2PExchange:
    """The cross-GPU argmax of the hypothesis-split mode as ONE kernel over NVLink peer memory (csrc/p2p_api.cu) instead of
    NCCL collectives.  Collective constructor: every rank of ``group`` builds it at the same point; the 64-byte CUDA IPC
    handles are all-gathered through torch.distributed (any backend)."""

    def __init__(self, group=None, device=None):
        torch = _torch()
        import torch.distributed as dist
        self.dev = _cuda_device(device)
        self.ctx = cabi.context(self.dev.index)
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        # every step below is followed by a collective that ALL ranks reach even when a local CUDA call failed, so that a
        # rank whose IPC mapping is refused (containers without shared IPC namespaces) makes everybody raise, not hang
        h = np.zeros(64, dtype=np.uint8)
        err = None
        try:
            cabi.call("rg_p2p_create", self.ctx, self.rank, self.world, h)
        except Exception as e:           # noqa: BLE001 - reported to every rank below
            err = repr(e)
        mine = (err, h.tobytes())
        got = [mine]
        if self.world > 1:
            got = [None] * self.world
            dist.all_gather_object(got, mine, group=group)
        if err is None and all(g[0] is None for g in got):
            try:
                cabi.call("rg_p2p_connect", self.ctx, np.frombuffer(b"".join(g[1] for g in got), dtype=np.uint8))
            except Exception as e:       # noqa: BLE001
                err = repr(e)
        errs = [err]
        if self.world > 1:
            errs = [None] * self.world
            dist.all_gather_object(errs, err, group=group)          # also the barrier: every peer mapped every buffer
        bad = [(r, e) for r, e in enumerate(errs) if e is not None] + [(r, g[0]) for r, g in enumerate(got) if g[0] is not None]
        if bad:
            self.close()
            raise cabi.RGError(f"peer-memory exchange unavailable (rank {bad[0][0]}: {bad[0][1]})")
        self.status = torch.zeros(1, dtype=torch.int32, device=self.dev)

    def argmax(self, key, payload, best_idx, best_count, payload_out):
        """key (P,) int64, payload (P, npay) float64 -> winner's global index / count / payload on every rank (async)."""
        P = key.numel()
        npay = payload.shape[1] if payload is not None else 0
        cabi.call("rg_p2p_argmax_exchange", self.ctx, _stream(), P, key, payload if npay else None, npay, best_idx,
                  best_count, payload_out if npay else None, self.status)

    def check(self):
        s = int(self.status.item())
        if s:
            raise cabi.RGError(f"p2p argmax exchange: rank {s - 1} did not arrive (timeout)")

    def close(self):
        """Unmaps the peers' buffers.  Best effort (a failure is not raised): it also runs on the constructor's error
        path, where the error to report is the one that made the exchange unavailable."""
        with contextlib.suppress(cabi.RGError, ValueError):
            cabi.call("rg_p2p_destroy", self.ctx)
