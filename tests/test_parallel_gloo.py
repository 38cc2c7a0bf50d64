"""world_size-2 gloo tests (CPU) of the multi-GPU host logic in parallel.py; the compute kernel is replaced by the
oracle so that only sharding, key packing and the collectives are exercised here."""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle_compute(pts_list, idx_list, thr=1.5, **kw):
    from oracle import f_path as orc
    P = len(pts_list)
    out = {"best_idx": np.full(P, -1, np.int32), "best_count": np.zeros(P, np.int32), "F": np.full((P, 3, 3), np.nan),
           "mask": []}
    for p in range(P):
        pts = np.asarray(pts_list[p])
        r = orc.f_ransac(pts[:, :2].T.copy(), pts[:, 2:].T.copy(), idx_list[p], thr, tie="first")
        out["best_idx"][p], out["best_count"][p] = r["best"], r["counts"].max() if r["best"] >= 0 else 0
        if r["best"] >= 0:
            out["F"][p] = r["F"]
        out["mask"].append(r["mask"])
    return out


def _oracle_pnp(X, y, idx, thr2, **kw):
    from oracle import pnp_path as opnp
    X = np.asarray(X, dtype=np.float64)
    yh = np.hstack([np.asarray(y, dtype=np.float64), np.ones((len(X), 1))])
    r = opnp.pnp_ransac(X, yh, np.asarray(idx), thr2)
    return {"best_idx": r["best"], "best_count": int(r["counts"].max()) if r["best"] >= 0 else 0,
            "R": r["R"] if r["best"] >= 0 else np.full((3, 3), np.nan), "t": r["t"] if r["best"] >= 0 else np.full(3, np.nan),
            "mask": r["mask"]}


def _oracle_pnp_batched(X_list, y_list, idx_list, thr2, **kw):
    rs = [_oracle_pnp(X, y, i, thr2) for X, y, i in zip(X_list, y_list, idx_list)]
    return {"best_idx": np.array([r["best_idx"] for r in rs], np.int32), "best_count": np.array([r["best_count"] for r in rs], np.int32),
            "R": np.stack([r["R"] for r in rs]), "t": np.stack([r["t"] for r in rs])}


def _pnp_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from tsbb15_b200 import parallel, sampling, synth
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        thr2 = (1.5 / 3217.0) ** 2
        X, y, _ = synth.pnp_scene(200, seed=3, sigma_px=0.02, outlier_frac=0.2)
        idx = sampling.fast(200, 25, 6, seed=1)
        one = parallel.pnp_ransac_split_hypotheses(X, y, idx, thr2, compute=_oracle_pnp)
        views = [synth.pnp_scene(80 + 10 * v, seed=v, sigma_px=0.02, outlier_frac=0.1)[:2] for v in range(3)]
        vidx = [sampling.fast(len(v[0]), 80, 6, seed=v_) for v_, v in enumerate(views)]
        sh = parallel.pnp_ransac_views_sharded([v[0] for v in views], [v[1] for v in views], vidx, thr2,
                                               compute=_oracle_pnp_batched)
        q.put((rank, one["best_idx"], one["best_count"], one["R"].tolist(), one["t"].tolist(), one["mask"].tolist(),
               one["owner"], sh["range"], sh["best_idx"].tolist(), sh["best_count"].tolist(), sh["R"].tolist()))
    finally:
        dist.destroy_process_group()


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    import tsbb15_b200 as rg
    from tsbb15_b200 import parallel, sampling, synth
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        pairs = synth.multi_pair(5, 300)
        idxs = [sampling.fast(300, 40, 8, seed=p) for p in range(5)]
        res = parallel.f_ransac_pairs_sharded(pairs, idxs, thr=1.5, compute=_oracle_compute)
        split = parallel.f_ransac_split_hypotheses(pairs[0], idxs[0], thr=1.5, compute=_oracle_compute)
        # the cross-rank key is the first maximum: the reference's sequential tie rule cannot be merged from per-rank winners
        try:
            parallel.f_ransac_split_hypotheses(pairs[0], idxs[0], thr=1.5, compute=_oracle_compute, tie_mode=rg.TIE_REFERENCE)
            raise AssertionError("tie_mode=TIE_REFERENCE must be refused when the hypotheses are split")
        except ValueError:
            pass
        # fewer hypotheses than ranks: the rank without work contributes a zero key instead of calling compute on nothing
        tiny = parallel.f_ransac_split_hypotheses(pairs[0], idxs[0][:1], thr=1.5, compute=_oracle_compute)
        assert tiny["best_idx"] in (0, -1) and tiny["mask"].shape == (300,)
        masks = parallel.f_ransac_pairs_sharded(pairs, idxs, thr=1.5, compute=_oracle_compute, gather_mask=True)["mask"]
        assert len(masks) == 5 and all(m.shape == (300,) for m in masks)
        q.put((rank, res["range"], res["best_idx"].tolist(), res["best_count"].tolist(), res["F"].tolist(),
               split["best_idx"], split["best_count"], split["F"].tolist(), split["mask"].tolist(), split["owner"]))
    finally:
        dist.destroy_process_group()


def test_shard_range_and_keys(rg):
    par = rg.parallel
    for n in (0, 1, 5, 8, 4096):
        for w in (1, 2, 3, 8):
            rs = [par.shard_range(n, r, w) for r in range(w)]
            assert rs[0][0] == 0 and rs[-1][1] == n
            assert all(rs[i][1] == rs[i + 1][0] for i in range(w - 1))
            assert max(b - a for a, b in rs) - min(b - a for a, b in rs) <= 1
            assert [par.shard_owner(n, i, w) for i in range(n)] == [r for r, (a, b) in enumerate(rs) for _ in range(a, b)]
            assert par.shard_owner(n, n, w) == par.shard_owner(n, -1, w) == -1
    assert par.argmax_key(10, 5) > par.argmax_key(10, 6) > par.argmax_key(9, 0)
    assert par.key_decode(par.argmax_key(123, 4567)) == (123, 4567)


def test_world_size_2_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted(q.get(timeout=240) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    sys.path.insert(0, ROOT)
    from tsbb15_b200 import sampling, synth
    pairs = synth.multi_pair(5, 300)
    idxs = [sampling.fast(300, 40, 8, seed=p) for p in range(5)]
    ref = _oracle_compute(pairs, idxs, 1.5)
    assert outs[0][1] == (0, 3) and outs[1][1] == (3, 5)
    for o in outs:                                        # both ranks hold the full, identical, correct result
        assert o[2] == ref["best_idx"].tolist() and o[3] == ref["best_count"].tolist()
        assert np.allclose(np.array(o[4]), ref["F"])
        assert o[5] == int(ref["best_idx"][0]) and o[6] == int(ref["best_count"][0])
        assert np.allclose(np.array(o[7]), ref["F"][0])
        assert o[8] == ref["mask"][0].tolist()
    assert outs[0][9] == outs[1][9] in (0, 1)


def test_world_size_2_gloo_pnp():
    """PnP: hypotheses of one view split over two ranks (one 8-byte max-all-reduce) and views sharded over ranks."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_pnp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted(q.get(timeout=240) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    sys.path.insert(0, ROOT)
    from tsbb15_b200 import sampling, synth
    thr2 = (1.5 / 3217.0) ** 2
    X, y, _ = synth.pnp_scene(200, seed=3, sigma_px=0.02, outlier_frac=0.2)
    ref = _oracle_pnp(X, y, sampling.fast(200, 25, 6, seed=1), thr2)
    views = [synth.pnp_scene(80 + 10 * v, seed=v, sigma_px=0.02, outlier_frac=0.1)[:2] for v in range(3)]
    vidx = [sampling.fast(len(v[0]), 80, 6, seed=v_) for v_, v in enumerate(views)]
    refb = _oracle_pnp_batched([v[0] for v in views], [v[1] for v in views], vidx, thr2)
    assert outs[0][7] == (0, 2) and outs[1][7] == (2, 3)
    for o in outs:
        assert o[1] == ref["best_idx"] >= 0 and o[2] == ref["best_count"]
        assert np.allclose(np.array(o[3]), ref["R"]) and np.allclose(np.array(o[4]), ref["t"])
        assert o[5] == ref["mask"].tolist()
        assert o[8] == refb["best_idx"].tolist() and o[9] == refb["best_count"].tolist()
        assert np.allclose(np.array(o[10]), refb["R"], equal_nan=True)
    assert (refb["best_idx"] >= 0).any()
    assert outs[0][6] == outs[1][6] in (0, 1)
