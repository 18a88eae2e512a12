"""gloo test (CPU, world 2 and 3) of ShardedIndex.range_search: the counts exchange, the padded payload exchange, the
merge rule of wb_range_merge_dev and the failure protocol.  The CUDA calls are replaced by doubles: the local range
search is tests/range_oracle.py over the rank's rows, and the merge is a numpy version of range_merge_parts_kernel's
rule.  The GPU version of the same property is tests/test_range_sharded_gpu.py."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import oracle as O
from range_oracle import ivf_range_search, range_search
from wise_b200.sharded import ShardedIndex

N, DIM, NLIST = 3000, 32, 16


def _canon(lims, D, I):
    """Order every query's hits by (float32 score desc, id asc): the single-index order, as ids grow with position."""
    D, I = D.copy(), I.copy()
    for q in range(lims.size - 1):
        a, b = int(lims[q]), int(lims[q + 1])
        o = np.lexsort((I[a:b], -D[a:b].astype(np.float64)))
        D[a:b], I[a:b] = D[a:b][o], I[a:b][o]
    return lims.astype(np.uint64), D, I


def _reference(xb, ids, xq, thresh, keep=None, ivf=None):
    """Range search of one index over rows xb (keep: the rows a selector keeps; ivf: (assign, centroids, nprobe))."""
    rows = np.arange(xb.shape[0]) if keep is None else np.nonzero(keep)[0]
    if ivf is None:
        return _canon(*range_search(xb[rows], xq, thresh, ids[rows]))
    assign, cent, nprobe = ivf
    return _canon(*ivf_range_search(xb[rows], ids[rows], assign[rows], cent, xq, thresh, nprobe))


class _Params:
    """Stands for faiss SearchParameters(sel=IDSelectorRange(lo, hi)) (+ nprobe for IVF)."""

    def __init__(self, lo, hi, nprobe=None):
        self.lo, self.hi, self.nprobe = lo, hi, nprobe


class _Shard:
    """Test double with what ShardedIndex reads from a faiss_compat index; `ivf` = (assign, centroids) or None."""

    def __init__(self, xb, ids, ivf=None, nprobe=1):
        self.xb, self.ids, self.d, self.ivf, self.nprobe = xb, ids, xb.shape[1], ivf, nprobe

    @property
    def ntotal(self):
        return self.xb.shape[0]

    def _search_params(self, p):
        return (p.nprobe or self.nprobe), (self.ids >= p.lo) & (self.ids < p.hi)


def _local_range_search(index, q, thresh, nprobe, keep=None):
    ivf = None if index.ivf is None else (index.ivf[0], index.ivf[1], nprobe)
    lims, D, I = _reference(index.xb, index.ids, q.numpy(), thresh, keep, ivf)
    return torch.from_numpy(lims.astype(np.int64)), torch.from_numpy(D), torch.from_numpy(I)


def _failing_local_range_search(index, q, thresh, nprobe, keep=None):
    if dist.get_rank() == 1:
        raise RuntimeError("range_search: query 0 has too many results")
    return _local_range_search(index, q, thresh, nprobe, keep)


def _order_bits(d):
    u = (d + np.float32(0)).view(np.uint32).astype(np.uint64)  # -0 -> +0, as order_f32
    return np.where(u >> 31, ~u & 0xFFFFFFFF, u | 0x80000000)


def _numpy_range_merge(lims_parts, Dp, Ip, lims):
    """range_merge_parts_kernel's rule: entry i of part p goes to lims[q] + (i - lp[q]) + the entries of every other
    part o that come first (larger order bits if o > p, larger or equal if o < p)."""
    lp, Dp, Ip, lims = lims_parts.numpy(), Dp.numpy(), Ip.numpy(), lims.numpy()
    parts, nq = lp.shape[0], lp.shape[1] - 1
    D = np.full(int(lims[-1]), np.nan, np.float32)
    I = np.full(int(lims[-1]), -7, np.int64)
    for q in range(nq):
        runs = [_order_bits(Dp[o, lp[o, q]:lp[o, q + 1]])[::-1] for o in range(parts)]  # ascending
        for p in range(parts):
            a, b = lp[p, q], lp[p, q + 1]
            key = _order_bits(Dp[p, a:b])
            out = lims[q] + np.arange(b - a)
            for o in range(parts):
                if o != p:
                    out = out + runs[o].size - np.searchsorted(runs[o], key, "left" if o < p else "right")
            D[out], I[out] = Dp[p, a:b], Ip[p, a:b]
    assert not np.any(I == -7), "the merge is not a permutation"
    return torch.from_numpy(D), torch.from_numpy(I)


def _data():
    xb = O.unit_gaussian(N, DIM, 41)
    xb[N - 40:] = xb[:40]  # duplicates on the last rank of rows on the first rank
    xb[1400:1500] = 0.0  # rows that never score above a positive threshold
    ids = np.arange(N, dtype=np.int64) * 3 + 7
    xq = np.concatenate([O.unit_gaussian(5, DIM, 42), xb[3:4], np.zeros((1, DIM), np.float32)])  # a tie; no hits
    cent = O.unit_gaussian(NLIST, DIM, 43)
    return xb, ids, xq, cent, O.ivf_assign(xb, cent)


def _bounds(world):
    """Contiguous row ranges in rank order: with world 2, rank 0 holds no rows; with world 3, rank 1 holds only
    all-zero rows (no hits above a positive threshold) and the duplicates of rank 0's rows live on rank 2."""
    if world == 3:
        return [(0, 1400), (1400, 1500), (1500, N)]
    return [(0, 0), (0, N)]


CASES = [(kind, t, sel) for kind in ("flat", "ivf") for t in (0.3, 0.6, -2.0) for sel in (False, True)]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        xb, ids, xq, cent, assign = _data()
        lo, hi = _bounds(world)[rank]
        res = {}
        for kind, t, sel in CASES:
            ivf = (assign[lo:hi], cent) if kind == "ivf" else None
            sh = ShardedIndex(_Shard(xb[lo:hi], ids[lo:hi], ivf, nprobe=3), local_range_search=_local_range_search,
                              range_merge=_numpy_range_merge)
            params = _Params(ids[200], ids[2900], nprobe=5 if kind == "ivf" else None) if sel else None
            lims, D, I = sh.range_search(xq, t, params=params)
            assert lims.dtype == np.uint64 and D.dtype == np.float32 and I.dtype == np.int64
            res[f"{kind}_{t}_{sel}"] = np.concatenate([lims.view(np.int64), D.view(np.int32).astype(np.int64), I])
            l0, D0, I0 = sh.range_search(xq[:0], t, params=params)
            assert l0.tolist() == [0] and l0.dtype == np.uint64 and D0.size == 0 and I0.size == 0
        # a failure on rank 1 raises on every rank, and the index stays usable
        sh = ShardedIndex(_Shard(xb[lo:hi], ids[lo:hi]), local_range_search=_failing_local_range_search,
                          range_merge=_numpy_range_merge)
        with pytest.raises(RuntimeError, match=r"failed on rank\(s\) \[1\]"):
            sh.range_search(xq, 0.3)
        sh._local_range_search = _local_range_search
        lims, D, I = sh.range_search(xq, 0.3)
        res["after_failure"] = np.concatenate([lims.view(np.int64), I])
        np.savez(os.path.join(out, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_range_equals_single_index(tmp_path, world):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    xb, ids, xq, cent, assign = _data()
    got = [np.load(tmp_path / f"r{r}.npz") for r in range(world)]
    for kind, t, sel in CASES:
        key = f"{kind}_{t}_{sel}"
        for g in got[1:]:
            assert np.array_equal(g[key], got[0][key]), key  # identical on every rank
        keep = (ids >= ids[200]) & (ids < ids[2900]) if sel else None
        ivf = (assign, cent, 5 if sel else 3) if kind == "ivf" else None
        lims, D, I = _reference(xb, ids, xq, t, keep, ivf)
        want = np.concatenate([lims.view(np.int64), D.view(np.int32).astype(np.int64), I])
        assert np.array_equal(got[0][key], want), key  # bit for bit the single-index result
        if t > 0:
            assert lims[-2] == lims[-1]  # the zero query has no hits
        if t > 0 and not sel:  # the duplicate of row 3 (last rank) follows row 3 (first rank)
            a = int(lims[5])
            assert I[a] == ids[3] and I[a + 1] == ids[N - 40 + 3] and D[a] == D[a + 1]
    lims, _, I = _reference(xb, ids, xq, 0.3)
    assert np.array_equal(got[0]["after_failure"], np.concatenate([lims.view(np.int64), I]))
