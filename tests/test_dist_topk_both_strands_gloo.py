"""CPU, world_size 2, gloo: all_pairs_step(..., identity=(model, t, True), top_k=K) -- each query's K best hits over both
strands, the query blocks sharded over ranks -- equals the same step in one process, strands included.  The engine is a
stand-in built on the oracle: each rank reverse-complements the gathered histograms itself, a pair's identity is the
better of its two strands (ties go to forward), and a query's hits are ordered by identity descending then database row
ascending.  Also: an engine without topk_both_strands still refuses a both-strand top_k."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as tdist
import torch.multiprocessing as mp

from conftest import weights_text
from meshclust2_b200 import dist as mdist
from meshclust2_b200 import synth
from oracle import port

T = 0.45
K = 8


def _rc_perm(k):
    j = np.arange(4 ** k, dtype=np.int64)
    r = np.zeros_like(j)
    for p in range(k):
        r = r * 4 + (3 - ((j >> (2 * p)) & 3))
    return r


class OneStrandEngine:
    """K1 through the oracle; no top-K search of its own"""

    def __init__(self, seqs, per):
        self.seqs, self.per = seqs, per
        self.device = torch.device("cpu")

    def count(self):
        pts = [port.get_point(s, 5, 1) for s in self.seqs]
        self.H = np.stack([p["hist"] for p in pts]) if pts else np.zeros((0, 1024), dtype=np.uint8)
        self.ln = np.array([p["len"] for p in pts], dtype=np.int64)
        self.mag = np.array([p["mag"] for p in pts], dtype=np.int64)

    def use_local_as_full(self):
        self.full = (self.H, self.ln, self.mag)

    def export_local(self):
        bins = torch.ones((self.per, 1024), dtype=torch.uint8)
        ln = torch.zeros((self.per,), dtype=torch.int64)
        mag = torch.zeros((self.per,), dtype=torch.int64)
        n = len(self.seqs)
        bins[:n] = torch.from_numpy(self.H)
        ln[:n] = torch.from_numpy(self.ln)
        mag[:n] = torch.from_numpy(self.mag)
        return bins, ln, mag

    def install_full(self, bins, length, mag, n_total):
        assert bins.shape[0] == n_total
        self.full = (bins.numpy(), length.numpy(), mag.numpy())


class BothStrandTopkEngine(OneStrandEngine):
    """the both-strand top-K identity search through the oracle"""

    def topk_both_strands(self, q0, q1, upper_only, cutoff, identity, top_k):
        model, t = identity
        H, ln, mag = self.full
        R = np.empty_like(H)
        R[:, _rc_perm(5)] = H                   # the other strand of every gathered row, built on this rank
        nq = q1 - q0
        d = np.full((nq, top_k), np.iinfo(np.uint64).max, dtype=np.uint64)
        ident = np.full((nq, top_k), -1.0)
        strand = np.full((nq, top_k), -1, dtype=np.int8)
        count = np.zeros(nq, dtype=np.uint32)
        n_hits = np.zeros(nq, dtype=np.uint64)
        n_scored = 0
        for r in range(q0, q1):
            lo, hi = int(float(ln[r]) * cutoff), int(float(ln[r]) / cutoff)
            hits = []
            for c in range(r + 1 if upper_only else 0, H.shape[0]):
                if lo <= ln[c] <= hi:
                    n_scored += 1
                    f = port.predict_pair(model, H[c], H[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                    v = port.predict_pair(model, H[c], R[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                    if max(f, v) >= t:
                        hits.append((-max(f, v), c, 1 if v > f else 0))
            hits.sort()
            top = hits[:top_k]
            n_hits[r - q0], count[r - q0] = len(hits), len(top)
            for j, (v, c, st) in enumerate(top):
                d[r - q0, j], ident[r - q0, j], strand[r - q0, j] = c, -v, st
        return int(n_hits.sum()), n_scored, dict(d=d, identity=ident, strand=strand, count=count, n_hits=n_hits)


def _model():
    m = port.Model.from_text(weights_text("weights_cfg1_id90"))
    m.weights[0] = 0.0          # without the intercept the sums of this set spread over about [0.1, 3]
    return m


def _rows(res):
    """{query row: (d, identity, strand, count, n_hits)} from a step's tables"""
    out = {}
    for q0, q1, tb in res["topk"]:
        for i in range(q1 - q0):
            out[q0 + i] = (tb["d"][i].tolist(), tb["identity"][i].tolist(), tb["strand"][i].tolist(), int(tb["count"][i]),
                           int(tb["n_hits"][i]))
    return out


def _worker(rank, world, port_no, n_total, upper, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_no)
    tdist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        per, bounds = mdist.shard_bounds(n_total, world)
        lo, hi = bounds[rank]
        seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31, lo=lo, hi=hi)
        eng = BothStrandTopkEngine(seqs, per)
        res = mdist.all_pairs_step(eng, mdist.Comm(tdist), torch, n_total, 0.9, upper_only=upper, blocks_per_rank=2,
                                   identity=(_model(), T, True), top_k=K)
        gathered = [None] * world
        tdist.all_gather_object(gathered, _rows(res))
        if rank == 0:
            merged = {}
            for g in gathered:
                assert not set(g) & set(merged)            # a query lives on exactly one rank
                merged.update(g)
            out.put((res["n_scored"], res["n_close"], merged))
    finally:
        tdist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.timeout(300)
@pytest.mark.parametrize("upper", [True, False], ids=["upper", "square"])
def test_two_ranks_both_strand_topk_step_equals_one_rank(upper):
    n_total = 61      # odd: the tail shard is padded for the all-gather
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    pno = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, pno, n_total, upper, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31)
    eng = BothStrandTopkEngine(seqs, n_total)
    res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n_total, 0.9, upper_only=upper, blocks_per_rank=2,
                               identity=(_model(), T, True), top_k=K)
    want = (res["n_scored"], res["n_close"], _rows(res))
    assert got == want
    rows = want[2]
    assert sorted(rows) == list(range(n_total))
    assert 0 < want[1] < want[0]
    assert any(c == K and h > K for _, _, _, c, h in rows.values())      # some queries have more hits than K
    assert any(c < K for _, _, _, c, h in rows.values())                 # and some fewer, padded
    strands = {s for _, _, st, c, _ in rows.values() for s in st[:c]}
    assert strands == {0, 1}                                              # hits on both strands made the tables
    for _, _, st, c, _ in rows.values():
        assert all(s == -1 for s in st[c:])
    assert len(res["survivors"]) == 0


def test_both_strand_top_k_needs_an_engine_that_ranks_both_strands():
    for identity in (None, (_model(), T, True)):
        with pytest.raises(ValueError):
            mdist.all_pairs_step(OneStrandEngine([], 0), mdist.Comm(None), torch, 0, 0.9, identity=identity, top_k=K)
    with pytest.raises(ValueError):         # a both-strand engine still needs an identity search for top_k
        mdist.all_pairs_step(BothStrandTopkEngine([], 0), mdist.Comm(None), torch, 0, 0.9, identity=None, top_k=K)
