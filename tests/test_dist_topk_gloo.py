"""CPU, world_size 2, gloo: all_pairs_step(..., identity=(model, t), top_k=K) -- each query's K best identity hits, the
query blocks sharded over ranks -- equals the same step in one process.  The engine is a stand-in built on the oracle: a
query's hits are its in-window pairs with identity >= t, ordered by identity descending then database row ascending."""
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


class TopkEngine:
    """K1 and the top-K identity search through the oracle"""

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

    def topk(self, q0, q1, upper_only, cutoff, identity, top_k):
        model, t = identity
        H, ln, mag = self.full
        nq = q1 - q0
        d = np.full((nq, top_k), np.iinfo(np.uint64).max, dtype=np.uint64)
        ident = np.full((nq, top_k), -1.0)
        count = np.zeros(nq, dtype=np.uint32)
        n_hits = np.zeros(nq, dtype=np.uint64)
        n_scored = 0
        for r in range(q0, q1):
            lo, hi = int(float(ln[r]) * cutoff), int(float(ln[r]) / cutoff)
            hits = []
            for c in range(r + 1 if upper_only else 0, H.shape[0]):
                if lo <= ln[c] <= hi:
                    n_scored += 1
                    v = port.predict_pair(model, H[c], H[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                    if v >= t:
                        hits.append((-v, c))
            hits.sort()
            top = hits[:top_k]
            n_hits[r - q0], count[r - q0] = len(hits), len(top)
            for j, (v, c) in enumerate(top):
                d[r - q0, j], ident[r - q0, j] = c, -v
        return int(n_hits.sum()), n_scored, dict(d=d, identity=ident, count=count, n_hits=n_hits)


def _model():
    m = port.Model.from_text(weights_text("weights_cfg1_id90"))
    m.weights[0] = 0.0          # without the intercept the sums of this set spread over about [0.1, 3]
    return m


def _rows(res):
    """{query row: (d, identity, count, n_hits)} from a step's tables"""
    out = {}
    for q0, q1, tb in res["topk"]:
        for i in range(q1 - q0):
            out[q0 + i] = (tb["d"][i].tolist(), tb["identity"][i].tolist(), int(tb["count"][i]), int(tb["n_hits"][i]))
    return out


def _worker(rank, world, port_no, n_total, upper, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_no)
    tdist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        per, bounds = mdist.shard_bounds(n_total, world)
        lo, hi = bounds[rank]
        seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31, lo=lo, hi=hi)
        eng = TopkEngine(seqs, per)
        res = mdist.all_pairs_step(eng, mdist.Comm(tdist), torch, n_total, 0.9, upper_only=upper, blocks_per_rank=2,
                                   identity=(_model(), T), top_k=K)
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
def test_two_ranks_topk_step_equals_one_rank(upper):
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
    eng = TopkEngine(seqs, n_total)
    res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n_total, 0.9, upper_only=upper, blocks_per_rank=2,
                               identity=(_model(), T), top_k=K)
    want = (res["n_scored"], res["n_close"], _rows(res))
    assert got == want
    rows = want[2]
    assert sorted(rows) == list(range(n_total))
    assert 0 < want[1] < want[0]
    assert any(c == K and h > K for _, _, c, h in rows.values())      # some queries have more hits than K
    assert any(c < K for _, _, c, h in rows.values())                 # and some fewer, padded
    assert len(res["survivors"]) == 0


def test_top_k_needs_one_strand_identity():
    eng = TopkEngine([], 0)
    for identity in (None, (_model(), T, True)):
        with pytest.raises(ValueError):
            mdist.all_pairs_step(eng, mdist.Comm(None), torch, 0, 0.9, identity=identity, top_k=K)
