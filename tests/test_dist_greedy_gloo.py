"""CPU, world_size 2, gloo: all_pairs_step(..., identity=(model, t[, True]), greedy=True) -- greedy representative
clustering with every query-row block shared over the ranks, the part slots all-gathered and the block added on every
rank -- equals the same step in one process and one sequential greedy pass over all edges, on one and on both strands.
The engine is a stand-in built on the oracle: an edge is an upper-triangle pair whose identity (the better strand's with
both strands, strand 1 when the reverse one is larger) is >= t; its slots are numpy arrays and add_block is a host
greedy update.  Also: a capacity at which only one rank overflows, the ValueError cases of `greedy`, and block_shares."""
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
from test_dist_topk_both_strands_gloo import OneStrandEngine, _rc_perm

T = 0.6
CUTOFF = 0.9


def _model():
    m = port.Model.from_text(weights_text("weights_cfg1_id90"))
    m.weights[0] = 0.0          # without the intercept the sums of this set spread over about [0.1, 3]
    return m


def _edges(H, ln, mag, model, t, both, q0, q1):
    """the edges (r, c, identity, strand) of query rows [q0, q1) and the forward in-window pair count"""
    R = np.empty_like(H)
    R[:, _rc_perm(5)] = H
    n = H.shape[0]
    out, n_scored = [], 0
    for r in range(q0, q1):
        lo, hi = int(float(ln[r]) * CUTOFF), int(float(ln[r]) / CUTOFF)
        for c in range(r + 1, n):
            if lo <= ln[c] <= hi:
                n_scored += 1
                v = port.predict_pair(model, H[c], H[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                s = 0
                if both:
                    w = port.predict_pair(model, H[c], R[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                    if w > v:
                        v, s = w, 1
                if v >= t:
                    out.append((r, c, v, s))
    return out, n_scored


def _sequential(n, edges):
    """one greedy pass over all edges: a row is a representative unless an earlier one has an edge to it; a member takes
    its heaviest edge from an earlier representative, the smallest such row on a tie"""
    into = [[] for _ in range(n)]
    for r, c, v, s in edges:
        into[c].append((r, v, s))
    rep = np.arange(n, dtype=np.uint64)
    ident = np.full(n, -1.0)
    strand = np.full(n, -1, dtype=np.int8)
    is_rep = np.zeros(n, dtype=bool)
    for c in range(n):
        best = None
        for r, v, s in into[c]:
            if is_rep[r] and (best is None or v > best[1] or (v == best[1] and r < best[0])):
                best = (r, v, s)
        if best is None:
            is_rep[c] = True
        else:
            rep[c], ident[c], strand[c] = best
    return dict(rep=rep, identity=ident, strand=strand, n_clusters=int(is_rep.sum()))


class GreedyEngine(OneStrandEngine):
    """the staged greedy clustering through the oracle; `cap` edges per part slot"""

    def __init__(self, seqs, per, cap=None):
        super().__init__(seqs, per)
        self.cap = cap

    def greedy_begin(self, cutoff, identity, n_parts):
        assert cutoff == CUTOFF
        self.model, self.t = identity[:2]
        self.both = len(identity) > 2 and bool(identity[2])
        H = self.full[0]
        n = self.n = H.shape[0]
        self.slots = [np.zeros((0, 4)) for _ in range(n_parts)]
        self.status = np.zeros(n, dtype=np.int8)             # 0 undecided, 1 representative, 2 member
        self.best = [None] * n                               # (r, identity, strand) of the best in-edge from a representative
        self.next = 0
        return self.cap or n

    def greedy_sweep_part(self, part, q0, q1):
        assert self.next <= q0 <= q1 <= self.n
        H, ln, mag = self.full
        e, ns = _edges(H, ln, mag, self.model, self.t, self.both, q0, q1)
        if len(e) <= (self.cap or self.n):
            self.slots[part] = np.array(e, dtype=np.float64).reshape(-1, 4)
        return len(e), ns

    def greedy_gather(self, comm, most):
        if comm.dist is None:
            return
        mine = torch.zeros((most, 4), dtype=torch.float64)
        own = self.slots[comm.rank]
        mine[:len(own)] = torch.from_numpy(own)
        out = [torch.empty_like(mine) for _ in range(comm.world)]
        comm.dist.all_gather(out, mine)
        self.slots = [o.numpy() for o in out]

    def greedy_add_block(self, qb, qe, shares, counts):
        assert qb == self.next and shares[0][0] == qb and shares[-1][1] == qe
        edges = []
        for (q0, q1), m, slot in zip(shares, counts, self.slots):
            for r, c, v, s in slot[:m]:
                assert q0 <= r < q1 and r < c < self.n
                edges.append((int(r), int(c), float(v), int(s)))
        into = {}
        for r, c, v, s in edges:
            into.setdefault(c, []).append(r)
        for c in range(qb, qe):
            if self.best[c] is None and not any(self.status[r] == 1 for r in into.get(c, [])):
                self.status[c] = 1
            else:
                self.status[c] = 2
        for r, c, v, s in edges:
            b = self.best[c]
            if self.status[r] == 1 and (b is None or v > b[1] or (v == b[1] and r < b[0])):
                self.best[c] = (r, v, s)
        self.next = qe

    def greedy_end(self):
        assert self.next == self.n
        rep = np.arange(self.n, dtype=np.uint64)
        ident = np.full(self.n, -1.0)
        strand = np.full(self.n, -1, dtype=np.int8)
        for c in range(self.n):
            if self.status[c] == 2:
                rep[c], ident[c], strand[c] = self.best[c]
        return dict(rep=rep, identity=ident, strand=strand, n_clusters=int((self.status == 1).sum()))


def _summary(res):
    g = res["greedy"]
    return (res["n_scored"], res["n_close"], g["rep"].tolist(), g["identity"].tolist(), g["strand"].tolist(), g["n_clusters"])


def _worker(rank, world, port_no, n_total, both, cap, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_no)
    tdist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        per, bounds = mdist.shard_bounds(n_total, world)
        lo, hi = bounds[rank]
        seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31, lo=lo, hi=hi)
        eng = GreedyEngine(seqs, per, cap)
        res = mdist.all_pairs_step(eng, mdist.Comm(tdist), torch, n_total, CUTOFF, identity=(_model(), T, both), greedy=True)
        gathered = [None] * world
        tdist.all_gather_object(gathered, (_summary(res), res["blocks"]))
        if rank == 0:
            assert all(g == gathered[0] for g in gathered)      # every rank holds the same result
            out.put(gathered[0])
    finally:
        tdist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _two_ranks(n_total, both, cap=None):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    pno = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, pno, n_total, both, cap, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return got


def _one_rank(n_total, both, cap=None):
    seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31)
    eng = GreedyEngine(seqs, n_total, cap)
    res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n_total, CUTOFF, identity=(_model(), T, both), greedy=True)
    return res, eng


@pytest.mark.timeout(300)
@pytest.mark.parametrize("both", [False, True], ids=["one_strand", "both_strands"])
def test_two_ranks_greedy_step_equals_one_rank(both):
    n_total = 61      # odd: the tail shard is padded for the all-gather
    got, blocks2 = _two_ranks(n_total, both)
    res, eng = _one_rank(n_total, both)
    assert got == _summary(res)
    for blocks in (blocks2, res["blocks"]):                     # the slots hold n_total edges: several blocks
        assert len(blocks) > 1 and blocks[0][0] == 0 and blocks[-1][1] == n_total
        assert all(blocks[i][1] == blocks[i + 1][0] for i in range(len(blocks) - 1))
    H, ln, mag = eng.full
    edges, ns = _edges(H, ln, mag, _model(), T, both, 0, n_total)
    want = _sequential(n_total, edges)
    g = res["greedy"]
    assert g["rep"].tolist() == want["rep"].tolist() and g["n_clusters"] == want["n_clusters"]
    assert g["identity"].tolist() == want["identity"].tolist() and g["strand"].tolist() == want["strand"].tolist()
    assert res["n_scored"] == ns and res["n_close"] == len(edges) > 0
    assert 1 < g["n_clusters"] < n_total and len(res["survivors"]) == 0


@pytest.mark.timeout(300)
def test_one_rank_overflows_both_split():
    """a capacity between the two ranks' edge counts of the first block: only one rank overflows, both split the block the
    same way, and the result is still the one-rank, one-pass result"""
    n_total = 61
    seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31)
    eng = GreedyEngine(seqs, n_total)
    eng.count()
    H, ln, mag = eng.H, eng.ln, eng.mag
    counts = [len(_edges(H, ln, mag, _model(), T, False, q0, q1)[0]) for q0, q1 in mdist.block_shares(0, n_total, n_total, 2)]
    cap = (min(counts) + max(counts)) // 2
    assert min(counts) <= cap < max(counts) and cap >= n_total
    got, blocks = _two_ranks(n_total, False, cap)
    assert len(blocks) > 1
    edges, _ = _edges(H, ln, mag, _model(), T, False, 0, n_total)
    want = _sequential(n_total, edges)
    assert got[2] == want["rep"].tolist() and got[3] == want["identity"].tolist() and got[5] == want["n_clusters"]
    res, _ = _one_rank(n_total, False)
    assert got == _summary(res)


def test_greedy_value_errors():
    eng = GreedyEngine([], 0)
    ident = (_model(), T)
    for kw in (dict(identity=None), dict(identity=ident, upper_only=False), dict(identity=ident, top_k=4),
               dict(identity=ident, components=True)):
        with pytest.raises(ValueError):
            mdist.all_pairs_step(eng, mdist.Comm(None), torch, 0, CUTOFF, greedy=True, **kw)
    with pytest.raises(ValueError):         # an engine without greedy_begin
        mdist.all_pairs_step(OneStrandEngine([], 0), mdist.Comm(None), torch, 0, CUTOFF, identity=ident, greedy=True)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_block_shares(world):
    for n in (0, 1, 2, 7, 61, 1000):
        for qb, qe in ((0, n), (n // 3, n), (n // 2, n // 2 + 3), (0, n // 4)):
            qe = min(qe, n)
            shares = mdist.block_shares(qb, qe, n, world)
            assert len(shares) == world and shares[0][0] == qb and shares[-1][1] == qe
            assert all(a <= b for a, b in shares) and all(shares[p][1] == shares[p + 1][0] for p in range(world - 1))
            cost = [sum(n - 1 - r + 160 for r in range(a, b)) for a, b in shares]
            row = n - 1 - qb + 160                  # the dearest row of the block
            total = sum(cost)
            assert all(abs(c - total / world) <= row for c in cost)
        if n:
            assert [s for s in mdist.block_shares(0, n, n, world) if s[1] > s[0]] == \
                [b for r in range(world) for b in mdist.triangle_row_blocks(n, world, r)]
