"""CPU, world_size 2, gloo: all_pairs_step(..., identity=(model, t[, True]), components=True) -- the single-linkage clusters
of the identity graph, the query blocks sharded over ranks and the per-rank labels all-gathered and joined -- equals the
same step in one process, on one and on both strands.  The engine is a stand-in built on the oracle: an edge is an
upper-triangle pair whose identity (the better strand's with both strands) is >= t, and the components come from a numpy
union-find labelled by their smallest row.  Also: the ValueError cases of `components`."""
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


def _union_find(n, a, b):
    """labels (smallest row of each component) of the graph on rows 0..n-1 with edges (a[i], b[i])"""
    parent = np.arange(n)

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    for u, v in zip(a, b):
        ru, rv = find(int(u)), find(int(v))
        if ru != rv:
            parent[max(ru, rv)] = min(ru, rv)
    return np.array([find(i) for i in range(n)], dtype=np.uint64)


class ComponentsEngine(OneStrandEngine):
    """identity clustering through the oracle"""

    def components(self, q0, q1, cutoff, identity):
        model, t = identity[:2]
        both = len(identity) > 2 and bool(identity[2])
        H, ln, mag = self.full
        R = np.empty_like(H)
        R[:, _rc_perm(5)] = H                   # the other strand of every gathered row, built on this rank
        n = H.shape[0]
        a, b, n_scored = [], [], 0
        for r in range(q0, q1):
            lo, hi = int(float(ln[r]) * cutoff), int(float(ln[r]) / cutoff)
            for c in range(r + 1, n):
                if lo <= ln[c] <= hi:
                    n_scored += 1
                    v = port.predict_pair(model, H[c], H[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                    if both:
                        v = max(v, port.predict_pair(model, H[c], R[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r])))
                    if v >= t:
                        a.append(r)
                        b.append(c)
        label = _union_find(n, a, b)
        return dict(label=label, n_components=len(np.unique(label)), n_scored=n_scored)

    def merge_components(self, labels):
        labels = np.asarray(labels, dtype=np.int64)
        n = labels.shape[1]
        label = _union_find(n, np.tile(np.arange(n), labels.shape[0]), labels.reshape(-1))
        return dict(label=label, n_components=len(np.unique(label)))


def _model():
    m = port.Model.from_text(weights_text("weights_cfg1_id90"))
    m.weights[0] = 0.0          # without the intercept the sums of this set spread over about [0.1, 3]
    return m


def _worker(rank, world, port_no, n_total, both, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_no)
    tdist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        per, bounds = mdist.shard_bounds(n_total, world)
        lo, hi = bounds[rank]
        seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31, lo=lo, hi=hi)
        eng = ComponentsEngine(seqs, per)
        res = mdist.all_pairs_step(eng, mdist.Comm(tdist), torch, n_total, 0.9, upper_only=True, blocks_per_rank=2,
                                   identity=(_model(), T, both), components=True)
        gathered = [None] * world
        comp = res["components"]
        tdist.all_gather_object(gathered, (comp["label"].tolist(), comp["n_components"]))
        if rank == 0:
            assert all(g == gathered[0] for g in gathered)      # every rank holds the same labels
            out.put((res["n_scored"], res["n_close"], gathered[0]))
    finally:
        tdist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.timeout(300)
@pytest.mark.parametrize("both", [False, True], ids=["one_strand", "both_strands"])
def test_two_ranks_components_step_equals_one_rank(both):
    n_total = 61      # odd: the tail shard is padded for the all-gather
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    pno = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, pno, n_total, both, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31)
    eng = ComponentsEngine(seqs, n_total)
    res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n_total, 0.9, upper_only=True, blocks_per_rank=2,
                               identity=(_model(), T, both), components=True)
    comp = res["components"]
    assert len(res["blocks"]) == 2
    want = (res["n_scored"], res["n_close"], (comp["label"].tolist(), comp["n_components"]))
    assert got == want
    # the labels are those of one call over the whole triangle
    eng.count()
    eng.use_local_as_full()
    whole = eng.components(0, n_total, 0.9, (_model(), T, both))
    assert comp["label"].tolist() == whole["label"].tolist() and comp["n_components"] == whole["n_components"]
    assert 1 < comp["n_components"] < n_total                  # neither every row apart nor one component
    assert res["n_scored"] == whole["n_scored"] > 0 and len(res["survivors"]) == 0


def test_both_strands_join_more():
    """the same step on both strands gives a partition at least as coarse, and here strictly coarser"""
    n_total = 40
    seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31)
    labels = {}
    for both in (False, True):
        eng = ComponentsEngine(seqs, n_total)
        res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n_total, 0.9, identity=(_model(), T, both), components=True)
        labels[both] = res["components"]["label"]
    one, two = labels[False], labels[True]
    assert all(two[i] == two[j] for i in range(n_total) for j in range(n_total) if one[i] == one[j])
    assert len(np.unique(two)) < len(np.unique(one))


def test_components_value_errors():
    eng = ComponentsEngine([], 0)
    ident = (_model(), T)
    for kw in (dict(identity=None), dict(identity=ident, upper_only=False), dict(identity=ident, top_k=4)):
        with pytest.raises(ValueError):
            mdist.all_pairs_step(eng, mdist.Comm(None), torch, 0, 0.9, components=True, **kw)
    with pytest.raises(ValueError):         # an engine without components
        mdist.all_pairs_step(OneStrandEngine([], 0), mdist.Comm(None), torch, 0, 0.9, identity=ident, components=True)
