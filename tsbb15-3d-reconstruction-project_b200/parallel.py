"""Multi-GPU sharding of the RANSAC path: one process per GPU, ``torch.distributed`` (NCCL over NVLink) as plumbing.

Two decompositions (SURVEY.md section 8e):

* by image pair (``f_ransac_pairs_sharded``): pairs are independent, rank g takes a contiguous block of pairs, there is
  NO collective on the data path; the tiny per-pair results (best index, count, F) are gathered afterwards.
* by hypothesis block inside one pair (``f_ransac_split_hypotheses``): every rank holds all N correspondences, scores
  its slice of the hypotheses, and ONE 8-byte max-all-reduce on the key ``(count << 32) | (0xFFFFFFFF - index)`` picks
  the global winner with the lowest index among equal counts (= first-maximum rule of fun.py:320); the owner of the
  winner broadcasts F and the inlier mask.

``compute`` can be injected so the distributed logic is testable on CPU with the gloo backend (tests/ use the oracle
there); by default it is the CUDA library.
"""
from __future__ import annotations

import numpy as np

from . import _cabi as cabi
from . import runtime as _rt


def shard_range(n_units: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block partition: the first ``n_units % world`` ranks get one extra unit."""
    base, extra = divmod(n_units, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_owner(n_units: int, index: int, world: int) -> int:
    """The rank whose ``shard_range`` block holds unit ``index``; -1 when none does."""
    for r in range(world):
        lo, hi = shard_range(n_units, r, world)
        if lo <= index < hi:
            return r
    return -1


def argmax_key(count: int, index: int) -> int:
    """Monotone key: larger count wins, then the LOWER hypothesis index."""
    return (int(count) << 32) | (0xFFFFFFFF - int(index))


def key_decode(key: int) -> tuple[int, int]:
    return int(key) >> 32, 0xFFFFFFFF - (int(key) & 0xFFFFFFFF)


def _dist():
    import torch.distributed as dist
    return dist


def _world(group=None):
    dist = _dist()
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def _device_for_collectives(group=None):
    import torch
    dist = _dist()
    if dist.is_initialized() and dist.get_backend(group) == "nccl":
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


class NcclComm:
    """A raw ``ncclComm_t`` for the C-ABI reduction ``rg_argmax_allreduce`` (include/rg_b200.h) — what a host that does
    not use torch would create itself.  The unique id is made on rank 0 and handed to the other ranks through
    ``exchange`` (default: ``torch.distributed.broadcast_object_list`` on whatever backend is initialised)."""

    def __init__(self, rank: int, world: int, exchange=None, lib_name: str | None = None):
        import ctypes as C
        import os
        self._C = C
        self.lib = C.CDLL(lib_name or os.environ.get("RG_NCCL_LIB") or "libnccl.so.2", mode=C.RTLD_GLOBAL)

        class UniqueId(C.Structure):
            _fields_ = [("internal", C.c_char * 128)]

        self.lib.ncclGetUniqueId.argtypes = [C.POINTER(UniqueId)]
        self.lib.ncclCommInitRank.argtypes = [C.POINTER(C.c_void_p), C.c_int, UniqueId, C.c_int]
        self.lib.ncclCommDestroy.argtypes = [C.c_void_p]
        uid = UniqueId()
        if rank == 0 and self.lib.ncclGetUniqueId(C.byref(uid)) != 0:
            raise RuntimeError("ncclGetUniqueId failed")
        raw = bytes(C.string_at(C.byref(uid), 128))
        if exchange is None:
            def exchange(b):
                box = [b]
                _dist().broadcast_object_list(box, src=0)
                return box[0]
        raw = exchange(raw)
        C.memmove(C.byref(uid), raw, 128)
        self.handle = C.c_void_p()
        rc = self.lib.ncclCommInitRank(C.byref(self.handle), int(world), uid, int(rank))
        if rc != 0:
            raise RuntimeError(f"ncclCommInitRank failed ({rc})")
        self.rank, self.world = rank, world

    def close(self):
        if self.handle:
            self.lib.ncclCommDestroy(self.handle)
            self.handle = None


def argmax_allreduce_c(best_idx, best_count, index_offset, comm: NcclComm, stream=0):
    """(best_idx, best_count) of this rank's hypothesis block -> global winner, entirely through the C ABI on the device:
    rg_argmax_pack_dev -> rg_argmax_allreduce (ONE ncclAllReduce(max) of 8 bytes per pair) -> rg_argmax_unpack_dev."""
    import torch
    bi = torch.as_tensor(np.atleast_1d(np.asarray(best_idx, dtype=np.int32))).cuda()
    bc = torch.as_tensor(np.atleast_1d(np.asarray(best_count, dtype=np.int32))).cuda()
    P = bi.numel()
    key = torch.empty(P, dtype=torch.int64, device=bi.device)
    st = stream or torch.cuda.current_stream().cuda_stream
    cabi.call("rg_argmax_pack_dev", st, P, bi, bc, index_offset, key)
    cabi.call("rg_argmax_allreduce", comm.handle, st, key, P)
    cabi.call("rg_argmax_unpack_dev", st, P, key, bi, bc)
    torch.cuda.current_stream().synchronize()
    return bi.cpu().numpy(), bc.cpu().numpy()


def _gather_blocks(block: np.ndarray, sizes, group=None) -> np.ndarray:
    """Rank r passes its block of ``sizes[r]`` rows; every rank receives the blocks of all ranks, concatenated in rank
    order.  One all_gather of fixed-size buffers, padded to the largest block."""
    import torch
    rank, world = _world(group)
    block = torch.from_numpy(np.ascontiguousarray(block))
    buf = torch.zeros((max(1, int(max(sizes))),) + tuple(block.shape[1:]), dtype=block.dtype)
    buf[:block.shape[0]] = block
    buf = buf.to(_device_for_collectives(group))
    gathered = [torch.empty_like(buf) for _ in range(world)]
    _dist().all_gather(gathered, buf, group=group)
    return np.concatenate([g[:n].cpu().numpy() for g, n in zip(gathered, sizes)])


def f_ransac_pairs_sharded(pts_list, idx_list, thr=1.5, group=None, gather=True, gather_mask=False, compute=None,
                           **kw) -> dict:
    """Pair-sharded batched F-RANSAC.  Every rank passes the SAME full lists (or at least its own shard filled in);
    returns, on every rank, arrays over all pairs when ``gather`` is True, else only the local shard's results.
    gather_mask: also gather the winners' inlier masks (one uint8 all-gather, padded to the largest shard)."""
    rank, world = _world(group)
    P = len(pts_list)
    lo, hi = shard_range(P, rank, world)
    compute = compute or _rt.f_ransac_batched
    if gather_mask:
        kw = dict(kw, want_mask=True)
    if hi > lo:
        local = compute(pts_list[lo:hi], idx_list[lo:hi], thr=thr, **kw)
    else:
        local = {"best_idx": np.zeros(0, np.int32), "best_count": np.zeros(0, np.int32), "F": np.zeros((0, 3, 3)), "mask": []}
    out_local = {"range": (lo, hi), "best_idx": np.asarray(local["best_idx"]), "best_count": np.asarray(local["best_count"]),
                 "F": np.asarray(local["F"])}
    if "mask" in local:
        out_local["mask"] = list(local["mask"])
    if not gather or world == 1:
        return out_local
    starts = [shard_range(P, r, world)[0] for r in range(world)] + [P]          # the ranks' first pairs
    # one float64 row per pair: [best_idx, best_count, F(9)]
    rows = _gather_blocks(np.column_stack([out_local["best_idx"], out_local["best_count"],
                                           out_local["F"].reshape(hi - lo, 9)]), np.diff(starts), group)
    out = {"range": (lo, hi), "best_idx": rows[:, 0].astype(np.int32), "best_count": rows[:, 1].astype(np.int32),
           "F": rows[:, 2:].reshape(P, 3, 3)}
    if gather_mask:
        off = _rt.offsets([np.asarray(p).reshape(-1, 4).shape[0] for p in pts_list])     # of the pairs' masks
        mine = np.concatenate([np.zeros(0, np.uint8)] + [np.asarray(m, dtype=np.uint8) for m in out_local["mask"]])
        out["mask"] = _rt._split(_gather_blocks(mine, np.diff(off[starts]), group), off)
    return out


def _split_winner(best_idx: int, best_count: int, lo: int, payload: np.ndarray, mask, H: int, group=None,
                  reduced_key: int | None = None):
    """The winner of ONE RANSAC whose H hypotheses are split over the ranks: this rank's winner is hypothesis ``lo +
    best_idx`` (-1: none); one max-all-reduce of the ranks' ``argmax_key``, unless ``reduced_key`` already holds its
    result, picks the global winner, and its owner broadcasts its float64 ``payload`` (the model) and its inlier
    ``mask`` (as bytes).  Returns (best_idx, best_count, payload, mask, owner); (-1, 0, NaN, zeros, -1) when no rank
    has a winner."""
    rank, world = _world(group)
    key = argmax_key(best_count, lo + best_idx) if best_idx >= 0 else 0
    if world == 1:
        cnt, gi = key_decode(key) if key else (0, -1)
        return gi, cnt, payload, mask, 0
    import torch
    dist = _dist()
    dev = _device_for_collectives(group)
    if reduced_key is None:
        k = torch.tensor([key], dtype=torch.int64, device=dev)
        dist.all_reduce(k, op=dist.ReduceOp.MAX, group=group)
        reduced_key = int(k.item())
    if reduced_key == 0:
        return -1, 0, np.full(payload.size, np.nan), np.zeros(len(mask), np.uint8), -1
    cnt, gi = key_decode(reduced_key)
    owner = shard_owner(H, gi, world)
    src = dist.get_global_rank(group, owner) if group is not None else owner
    pw = torch.zeros(payload.size, dtype=torch.float64)
    mw = torch.zeros(len(mask), dtype=torch.uint8)
    if rank == owner:
        pw = torch.from_numpy(np.ascontiguousarray(payload, dtype=np.float64))
        mw = torch.from_numpy(np.ascontiguousarray(np.asarray(mask, dtype=np.uint8)))
    pw, mw = pw.to(dev), mw.to(dev)
    dist.broadcast(pw, src=src, group=group)
    dist.broadcast(mw, src=src, group=group)
    return gi, cnt, pw.cpu().numpy(), mw.cpu().numpy(), owner


def f_ransac_split_hypotheses(pts, idx, thr=1.5, group=None, compute=None, nccl_comm: NcclComm | None = None, **kw) -> dict:
    """One pair, hypotheses split across ranks, one max-all-reduce of an int64 key (first-maximum selection).
    nccl_comm: reduce through the library's own C entry point ``rg_argmax_allreduce`` on that communicator instead of
    ``torch.distributed.all_reduce`` (same key, same result)."""
    rank, world = _world(group)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    H = idx.shape[0]
    lo, hi = shard_range(H, rank, world)
    compute = compute or _rt.f_ransac_batched
    kw = dict(kw)
    kw["want_mask"] = True
    if world > 1 and kw.get("tie_mode", _rt.TIE_FIRST) != _rt.TIE_FIRST:
        # the cross-rank key implements the first maximum; the reference's tie rule (fun.py:324-328) is a sequential replay
        # over ALL maximal hypotheses and cannot be merged from per-rank winners
        raise ValueError("f_ransac_split_hypotheses supports tie_mode=TIE_FIRST only when the hypotheses are split")
    n = np.asarray(pts).reshape(-1, 4).shape[0]
    if hi > lo:
        local = compute([pts], [idx[lo:hi]], thr=thr, **kw)
    else:                                            # H < world: this rank holds no hypothesis
        local = {"best_idx": np.array([-1], np.int32), "best_count": np.array([0], np.int32),
                 "F": np.full((1, 3, 3), np.nan), "mask": [np.zeros(n, np.uint8)]}
    reduced = None
    if nccl_comm is not None and world > 1:
        gi_a, cnt_a = argmax_allreduce_c(local["best_idx"][:1], local["best_count"][:1], lo, nccl_comm)
        reduced = argmax_key(int(cnt_a[0]), int(gi_a[0])) if gi_a[0] >= 0 else 0
    gi, cnt, F, mask, owner = _split_winner(int(local["best_idx"][0]), int(local["best_count"][0]), lo,
                                            np.asarray(local["F"][0], dtype=np.float64).reshape(9), local["mask"][0], H,
                                            group, reduced)
    return {"best_idx": gi, "best_count": cnt, "F": F.reshape(3, 3), "mask": mask, "owner": owner}


def pnp_ransac_split_hypotheses(X, y, idx, thr2, group=None, compute=None, **kw) -> dict:
    """PnP-RANSAC of ONE view (BASELINE config 4 at G > 1) with the pose hypotheses split across ranks: every rank holds
    all N correspondences and scores its slice of the (H, n) samples; the same 8-byte max-all-reduce on
    ``(count << 32) | ~index`` as the F path picks the winner (first maximum, ransac.py:108); its owner broadcasts
    R, t and the consensus mask."""
    rank, world = _world(group)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    H = idx.shape[0]
    lo, hi = shard_range(H, rank, world)
    compute = compute or _rt.pnp_ransac
    kw = dict(kw)
    kw["want_mask"] = True
    n = np.asarray(X).reshape(-1, 3).shape[0]
    if hi > lo:
        local = compute(X, y, idx[lo:hi], thr2, **kw)
    else:
        local = {"best_idx": -1, "best_count": 0, "R": np.full((3, 3), np.nan), "t": np.full(3, np.nan),
                 "mask": np.zeros(n, np.uint8)}
    Rt = np.concatenate([np.ravel(local["R"]), np.ravel(local["t"])]).astype(np.float64)
    gi, cnt, Rt, mask, owner = _split_winner(int(local["best_idx"]), int(local["best_count"]), lo, Rt, local["mask"], H,
                                             group)
    return {"best_idx": gi, "best_count": cnt, "R": Rt[:9].reshape(3, 3), "t": Rt[9:].copy(), "mask": mask, "owner": owner}


def pnp_ransac_views_sharded(X_list, y_list, idx_list, thr2, group=None, compute=None, **kw) -> dict:
    """View-sharded batched PnP-RANSAC (BASELINE config 2 at G > 1): views are independent, rank g takes a contiguous
    block, no data-path collective; (best index, count, R, t) of all views are gathered on every rank."""
    rank, world = _world(group)
    V = len(X_list)
    lo, hi = shard_range(V, rank, world)
    compute = compute or _rt.pnp_ransac_batched
    if hi > lo:
        local = compute(X_list[lo:hi], y_list[lo:hi], idx_list[lo:hi], thr2, **kw)
    else:
        local = {"best_idx": np.zeros(0, np.int32), "best_count": np.zeros(0, np.int32), "R": np.zeros((0, 3, 3)),
                 "t": np.zeros((0, 3))}
    out = {"range": (lo, hi), "best_idx": np.asarray(local["best_idx"]), "best_count": np.asarray(local["best_count"]),
           "R": np.asarray(local["R"]), "t": np.asarray(local["t"])}
    if world == 1:
        return out
    starts = [shard_range(V, r, world)[0] for r in range(world)] + [V]          # the ranks' first views
    # one float64 row per view: [best_idx, best_count, R(9), t(3)]
    rows = _gather_blocks(np.column_stack([out["best_idx"], out["best_count"], out["R"].reshape(hi - lo, 9),
                                           out["t"].reshape(hi - lo, 3)]), np.diff(starts), group)
    return {"range": (lo, hi), "best_idx": rows[:, 0].astype(np.int32), "best_count": rows[:, 1].astype(np.int32),
            "R": rows[:, 2:11].reshape(V, 3, 3), "t": rows[:, 11:].copy()}


# ---------------------------------------------------------------------------------------------------------------
# device-resident decompositions (what bench.py times; torch tensors only carry device memory)
# ---------------------------------------------------------------------------------------------------------------
class PairShardedRansac:
    """BASELINE config 5 (SURVEY.md section 8d/8e item 1): ``P_total`` image pairs of ``N`` correspondences x ``H``
    hypotheses, a FIXED total split over the ranks of ``group`` in contiguous blocks (strong scaling); pairs are independent,
    so there is no collective on the data path — only the results (index, count, F per pair = 80 bytes, optionally the
    inlier masks) are all-gathered.  Reference loop being multiplied: fun.py:303-328 per pair, main.py:93-126 over pairs.

    Inputs are either generated on the device from ``seed_base + pair`` (``generate``; host-replayable, philox.py) or supplied
    by the caller (``load``); sample index sets are drawn on the device from ``sample_seed`` (or supplied)."""

    def __init__(self, P_total: int, N: int, H: int, group=None, device=None, want_mask: bool = True):
        import torch
        from . import device as dv
        self.dv = dv
        self.group = group
        self.rank, self.world = _world(group)
        self.P_total, self.N, self.H = int(P_total), int(N), int(H)
        self.lo, self.hi = shard_range(self.P_total, self.rank, self.world)
        self.P = self.hi - self.lo
        self.per = (self.P_total + self.world - 1) // self.world          # padded shard size of the gathers
        self.dev = dv._cuda_device(device)
        self.pair_off = dv.offsets(np.full(self.P, self.N))
        self.hyp_off = dv.offsets(np.full(self.P, self.H))
        # results of the local shard as ONE block [F: per x 72 B][idx: per x 4 B][count: per x 4 B] -> one all-gather
        self.block = torch.zeros(self.per * 80, dtype=torch.uint8, device=self.dev)
        self.out = dv.FOutputs.__new__(dv.FOutputs)
        self.out.F = self.block[: self.per * 72].view(torch.float64).view(self.per, 9)
        self.out.best_idx = self.block[self.per * 72: self.per * 76].view(torch.int32)
        self.out.best_count = self.block[self.per * 76:].view(torch.int32)
        self.out.mask = torch.zeros(max(self.per * self.N, 1), dtype=torch.uint8, device=self.dev) if want_mask else None
        self.out.key = None
        self.out.P = self.P
        self.all_block = torch.empty(self.world * self.per * 80, dtype=torch.uint8, device=self.dev) if self.world > 1 else None
        self.all_mask = (torch.empty(self.world * self.per * self.N, dtype=torch.uint8, device=self.dev)
                         if (self.world > 1 and want_mask) else None)
        self.d_pts = None
        self.d_idx = None

    # ---- inputs
    def generate(self, seed_base: int = 1000, **kw):
        self.d_pts, self.cam_pair = self.dv.synth_two_view(self.P, self.N, first_pair=self.lo, seed_base=seed_base,
                                                           device=self.dev.index, **kw)
        return self.d_pts

    def load(self, d_pts, d_idx=None):
        self.d_pts, self.d_idx = d_pts, d_idx

    # ---- compute (asynchronous on the current stream)
    def run(self, thr=1.5, sample_seed: int = 0, **kw):
        if self.P:
            self.dv.f_ransac(self.d_pts, self.pair_off, self.d_idx, self.hyp_off, self.out, thr=thr, seed=sample_seed,
                             first_pair=self.lo, **kw)
        return self.out

    # ---- the same through the HOST-buffer entry point (end-to-end: uploads and result downloads inside the call)
    def alloc_host(self, want_mask: bool = True):
        """Page-locked host buffers for the local shard: inputs (P, N, 4) f64 and the per-pair results."""
        import torch
        self.h_pts = torch.empty((max(self.P, 1), self.N, 4), dtype=torch.float64, pin_memory=True)
        self.h_block = torch.zeros(self.per * 80, dtype=torch.uint8, pin_memory=True)
        self.h_F = self.h_block[: self.per * 72].view(torch.float64).view(self.per, 9)
        self.h_best_idx = self.h_block[self.per * 72: self.per * 76].view(torch.int32)
        self.h_best_count = self.h_block[self.per * 76:].view(torch.int32)
        self.h_mask = torch.empty(max(self.P * self.N, 1), dtype=torch.uint8, pin_memory=True) if want_mask else None
        self.h_all_block = torch.empty(self.world * self.per * 80, dtype=torch.uint8, pin_memory=True) if self.world > 1 else None
        return self.h_pts

    def run_host(self, thr=1.5, sample_seed: int = 0, mode=0, tie_mode=0, solver=0, score_path=0, h_idx=None):
        """rg_f_ransac_host2 on the local shard (synchronous: returns when the shard's results are in host memory), then the
        all-gather of the 80-byte results of all ranks (H2D of the local block, NCCL, D2H of everything)."""
        if self.P:
            self.dv._call("rg_f_ransac_host2", self.dev.index, self.P, self.h_pts, self.pair_off, h_idx, self.hyp_off, thr,
                          mode, tie_mode, solver, score_path, sample_seed, self.lo, self.h_best_idx, self.h_best_count,
                          self.h_F, self.h_mask, None, None, None)
        if self.world == 1:
            return self.h_block
        self.block.copy_(self.h_block, non_blocking=True)
        _dist().all_gather_into_tensor(self.all_block, self.block, group=self.group)
        self.h_all_block.copy_(self.all_block, non_blocking=True)
        import torch
        torch.cuda.current_stream().synchronize()
        return self.h_all_block

    def gather(self, masks: bool = True) -> dict:
        """All ranks receive the results of all pairs (device tensors; one NCCL all-gather of 80 B per pair, one of N bytes
        per pair for the masks)."""
        import torch
        if self.world == 1:
            blk, msk = self.block, self.out.mask
        else:
            dist = _dist()
            dist.all_gather_into_tensor(self.all_block, self.block, group=self.group)
            blk = self.all_block
            msk = None
            if masks and self.all_mask is not None:
                dist.all_gather_into_tensor(self.all_mask, self.out.mask, group=self.group)
                msk = self.all_mask
        return {"block": blk, "mask": msk}

    def unpack(self, gathered: dict) -> dict:
        """Host view of ``gather``'s result: arrays over all P_total pairs (synchronises)."""
        blk = gathered["block"].cpu().numpy()
        best_idx = np.empty(self.P_total, np.int32)
        best_count = np.empty(self.P_total, np.int32)
        F = np.empty((self.P_total, 3, 3))
        msk = gathered["mask"].cpu().numpy() if gathered["mask"] is not None else None
        masks = [] if msk is not None else None
        for r in range(self.world):
            a, b = shard_range(self.P_total, r, self.world)
            seg = blk[r * self.per * 80:(r + 1) * self.per * 80]
            F[a:b] = seg[: self.per * 72].view(np.float64).reshape(self.per, 3, 3)[: b - a]
            best_idx[a:b] = seg[self.per * 72: self.per * 76].view(np.int32)[: b - a]
            best_count[a:b] = seg[self.per * 76:].view(np.int32)[: b - a]
            if msk is not None:
                m = msk[r * self.per * self.N:(r + 1) * self.per * self.N].reshape(self.per, self.N)
                masks.extend(m[k] for k in range(b - a))
        return {"best_idx": best_idx, "best_count": best_count, "F": F, "mask": masks}


class SplitHypothesesF:
    """One image pair whose hypotheses are split over the ranks (BASELINE config 3 at G > 1, SURVEY.md section 8e item 2):
    every rank holds all N correspondences, prepares them ONCE (RG_FLAG_REUSE_POINTS afterwards), scores hypotheses
    [lo, hi), and the winner — key (count << 32 | ~global index) together with its F — is found by ONE peer-memory exchange
    kernel (P2PExchange) or, ``exchange="nccl"``, by the C-ABI ncclAllReduce(max) + a broadcast of F.  Every rank then
    computes the winner's inlier mask locally.  First-maximum selection only (fun.py:320-323)."""

    def __init__(self, d_pts, H: int, group=None, exchange: str = "p2p", nccl_comm: "NcclComm | None" = None, idx=None,
                 sample_seed: int = 0):
        import torch
        from . import device as dv
        self.dv = dv
        self.group = group
        self.rank, self.world = _world(group)
        self.d_pts = d_pts
        self.N = int(d_pts.shape[0])
        self.H = int(H)
        self.lo, self.hi = shard_range(self.H, self.rank, self.world)
        self.pair_off = np.array([0, self.N], dtype=np.int32)
        self.hyp_off = np.array([0, self.hi - self.lo], dtype=np.int32)
        dev = d_pts.device
        self.d_idx = None
        if idx is not None:
            self.d_idx = torch.from_numpy(np.ascontiguousarray(np.asarray(idx, dtype=np.int32)[self.lo:self.hi])).to(dev)
        self.sample_seed = int(sample_seed)
        self.out = dv.FOutputs(1, self.N, device=dev.index, want_mask=False, want_key=True)
        self.g_idx = torch.empty(1, dtype=torch.int32, device=dev)
        self.g_cnt = torch.empty(1, dtype=torch.int32, device=dev)
        self.g_F = torch.empty((1, 9), dtype=torch.float64, device=dev)
        self.mask = torch.empty(self.N, dtype=torch.uint8, device=dev)
        self.exchange = exchange if self.world > 1 else "none"
        self.p2p = dv.P2PExchange(group, device=dev.index) if self.exchange == "p2p" else None
        self.nccl_comm = nccl_comm
        self.prepared = False
        self.prepared_thr = None

    def run(self, thr=1.5, mode=0, want_mask: bool = True, **kw):
        """Asynchronous on the current stream; results in g_idx / g_cnt / g_F / mask (device)."""
        import torch
        dv = self.dv
        flags = dv.FLAG_REUSE_POINTS if (self.prepared and self.prepared_thr == thr) else 0
        if self.hi > self.lo:
            dv.f_ransac(self.d_pts, self.pair_off, self.d_idx, self.hyp_off, self.out, thr=thr, mode=mode, flags=flags,
                        seed=self.sample_seed, first_pair=0, hyp_first=self.lo, **kw)
            self.prepared, self.prepared_thr = True, thr
        else:
            self.out.key.zero_()
            self.out.F.fill_(float("nan"))
        if self.exchange == "none":
            cabi.call("rg_argmax_unpack_dev", dv._stream(), 1, self.out.key, self.g_idx, self.g_cnt)
            self.g_F.copy_(self.out.F)
        elif self.exchange == "p2p":
            self.p2p.argmax(self.out.key, self.out.F, self.g_idx, self.g_cnt, self.g_F)
        else:
            dist = _dist()
            if self.nccl_comm is not None:
                gkey = self.out.key.clone()
                cabi.call("rg_argmax_allreduce", self.nccl_comm.handle, dv._stream(), gkey, 1)
            else:
                gkey = self.out.key.clone()
                dist.all_reduce(gkey, op=dist.ReduceOp.MAX, group=self.group)
            # payload: the owner is the rank whose block holds the winning global index; everybody else contributes zeros
            # to a 72-byte sum
            cabi.call("rg_argmax_unpack_dev", dv._stream(), 1, gkey, self.g_idx, self.g_cnt)
            own = ((self.g_idx >= self.lo) & (self.g_idx < self.hi)).to(torch.float64)
            self.g_F.copy_(torch.nan_to_num(self.out.F) * own)
            dist.all_reduce(self.g_F, op=dist.ReduceOp.SUM, group=self.group)
        if want_mask:
            dv.f_inlier_mask(self.d_pts, self.pair_off, self.g_F, thr=thr, mode=mode, out=self.mask)
        return self

    def capture(self, thr=1.5, mode=0, want_mask: bool = True, **kw):
        """Capture run()'s launch chain in a CUDA graph.  Once the points are prepared and the plan is cached the chain is
        memset -> solve -> score -> fix-up -> argmax -> exchange kernel -> mask kernel with no host synchronisation, so it
        can be replayed with one launch (``replay``).  Collective: every rank captures and replays the same number of times.
        Not available with exchange="nccl" (the NCCL collectives are issued by torch)."""
        import torch
        if self.exchange not in ("none", "p2p"):
            raise ValueError("graph capture needs exchange='p2p' (or a single rank)")
        for _ in range(2):                                   # prepared points, cached plan, workspaces at their final size
            self.run(thr=thr, mode=mode, want_mask=want_mask, **kw)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.run(thr=thr, mode=mode, want_mask=want_mask, **kw)
        self.graph = g
        return g

    def replay(self):
        self.graph.replay()
        return self

    def result(self) -> dict:
        if self.p2p is not None:
            self.p2p.check()
        gi, gc = int(self.g_idx.item()), int(self.g_cnt.item())
        owner = shard_owner(self.H, gi, self.world)
        return {"best_idx": gi, "best_count": gc, "F": self.g_F.cpu().numpy().reshape(3, 3), "mask": self.mask.cpu().numpy(),
                "owner": owner}


class SplitHypothesesPnp:
    """BASELINE config 4 at G > 1: ONE view's pose hypotheses split over the ranks; same exchange as SplitHypothesesF with the
    12-double payload (R | t); the consensus mask is computed by the owner's call only when the view is not split, so here
    every rank re-scores the winner with a one-hypothesis call (ransac.py:96-105)."""

    def __init__(self, d_X, d_y, idx, n: int = 6, group=None, exchange: str = "p2p"):
        import torch
        from . import device as dv
        self.dv = dv
        self.group = group
        self.rank, self.world = _world(group)
        self.d_X, self.d_y = d_X, d_y
        self.N = int(d_X.shape[0])
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        self.H, self.n = int(idx.shape[0]), int(n)
        self.lo, self.hi = shard_range(self.H, self.rank, self.world)
        dev = d_X.device
        self.d_idx = torch.from_numpy(np.ascontiguousarray(idx[self.lo:self.hi])).to(dev)
        self.view_off = np.array([0, self.N], dtype=np.int32)
        self.hyp_off = np.array([0, self.hi - self.lo], dtype=np.int32)
        self.out = dv.PnpOutputs(1, self.N, device=dev.index, want_mask=False, want_key=True)
        self.g_idx = torch.empty(1, dtype=torch.int32, device=dev)
        self.g_cnt = torch.empty(1, dtype=torch.int32, device=dev)
        self.g_Rt = torch.empty((1, 12), dtype=torch.float64, device=dev)
        self.exchange = exchange if self.world > 1 else "none"
        self.p2p = dv.P2PExchange(group, device=dev.index) if self.exchange == "p2p" else None

    def run(self, thr2):
        import torch
        dv = self.dv
        if self.hi > self.lo:
            dv.pnp_ransac(self.d_X, self.d_y, self.view_off, self.d_idx, self.hyp_off, self.out, thr2, n=self.n,
                          hyp_first=self.lo)
        else:
            self.out.key.zero_()
            self.out.Rt.fill_(float("nan"))
        if self.exchange == "p2p":
            self.p2p.argmax(self.out.key, self.out.Rt, self.g_idx, self.g_cnt, self.g_Rt)
        else:
            gkey = self.out.key
            if self.exchange == "nccl":
                dist = _dist()
                gkey = self.out.key.clone()
                dist.all_reduce(gkey, op=dist.ReduceOp.MAX, group=self.group)
            cabi.call("rg_argmax_unpack_dev", dv._stream(), 1, gkey, self.g_idx, self.g_cnt)
            if self.exchange == "nccl":
                own = ((self.g_idx >= self.lo) & (self.g_idx < self.hi)).to(torch.float64)
                self.g_Rt.copy_(torch.nan_to_num(self.out.Rt) * own)
                dist.all_reduce(self.g_Rt, op=dist.ReduceOp.SUM, group=self.group)
            else:
                self.g_Rt.copy_(self.out.Rt)
        return self

    def result(self) -> dict:
        if self.p2p is not None:
            self.p2p.check()
        Rt = self.g_Rt.cpu().numpy().reshape(12)
        return {"best_idx": int(self.g_idx.item()), "best_count": int(self.g_cnt.item()), "R": Rt[:9].reshape(3, 3),
                "t": Rt[9:].copy()}
