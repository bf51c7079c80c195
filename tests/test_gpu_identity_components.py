"""GPU: identity clustering (mc2_identity_components, mc2_components_merge).  The reference is the flat search's edges
(mc2_identity_pairs over the upper triangle, or mc2_identity_pairs_both_strands, with room for every survivor) turned into
components by scipy's connected_components and labelled by the smallest row of each; labels, n_components and n_scored are
compared exactly.  Also against the oracle's predict_pair, on the coarse, full and row-streaming forms, with the block
split forced on either strand, over row and query sub-ranges joined by mc2_components_merge, and through the multi-GPU
driver's product engine."""
import ctypes as C

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from conftest import weights_path, weights_text
from helpers import all_singles_model, to_desc
from oracle import port
from test_gpu_both_strands import _big, _rc_rows, _strand_data
from test_gpu_identity_pairs import FLAGS5, TINY, _legacy, _oracle_identity, _regression, _spread, _window

pytestmark = pytest.mark.gpu

SCRATCH = 1 << 24           # survivors one block's sweep of one strand holds


def _canonical(n, a, b, begin=0):
    """labels (absolute smallest row of each component) of the graph on rows begin .. begin + n - 1, edges (a[i], b[i])"""
    a = np.asarray(a, dtype=np.int64) - begin
    b = np.asarray(b, dtype=np.int64) - begin
    g = coo_matrix((np.ones(len(a), dtype=np.int8), (a, b)), shape=(n, n))
    nc, lab = connected_components(g, directed=False)
    mins = np.full(nc, n, dtype=np.int64)
    np.minimum.at(mins, lab, np.arange(n))
    return (mins[lab] + begin).astype(np.uint64), nc


def _flat(ctx, gm, hs, t, both, q_range, rng_, cutoff=0.9, max_out=None):
    b0, b1 = rng_
    q0, q1 = q_range
    cap = max_out or max(1, (q1 - q0) * (b1 - b0))
    call = ctx.identity_pairs_both_strands if both else ctx.identity_pairs
    return call(gm, hs, hs, t, cutoff, q_range=q_range, d_range=rng_, upper_only=True, max_out=cap)


def _reference(ctx, gm, hs, t, both=False, q_range=None, range=None, cutoff=0.9, max_out=None):
    rng_ = range or (0, len(hs))
    q_range = q_range or rng_
    r = _flat(ctx, gm, hs, t, both, q_range, rng_, cutoff, max_out)
    assert len(r["q"]) == r["n_out"]                    # room for every edge
    label, nc = _canonical(rng_[1] - rng_[0], r["q"], r["d"], rng_[0])
    return dict(label=label, n_components=nc, n_scored=r["n_scored"], n_out=r["n_out"], q=r["q"], d=r["d"])


def _comp(ctx, gm, hs, t, both=False, q_range=None, range=None, cutoff=0.9):
    return ctx.identity_components(gm, hs, t, cutoff, both_strands=both, q_range=q_range, range=range)


def _check(ctx, gm, hs, t, both=False, max_out=None, **kw):
    want = _reference(ctx, gm, hs, t, both, max_out=max_out, **kw)
    got = _comp(ctx, gm, hs, t, both, **kw)
    assert got["label"].dtype == np.uint64
    assert np.array_equal(got["label"], want["label"])
    assert got["n_components"] == want["n_components"] and got["n_scored"] == want["n_scored"]
    return got, want


def _edge_t(ctx, gm, hs, per_row=0.5):
    """a threshold that keeps about per_row edges per row of the upper triangle (the highest identities): on sets of related
    groups of rows it mostly keeps pairs inside a group, so the graph has several components of several rows"""
    n = len(hs)
    every = ctx.identity_pairs(gm, hs, hs, -np.inf, 0.9, upper_only=True, max_out=n * n)
    return float(np.sort(every["identity"])[::-1][int(per_row * n)])


def _model(H, mag, ln, rng):
    """a regression model whose identities rarely clamp to 1 (a clamped tie at 1 would join a large share of all pairs)"""
    return _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng, lo=-1.0, hi=0.6)


def _nontrivial(r):
    return 1 < r["n_components"] < len(r["label"])


def _coarser(a, b, begin=0):
    """partition a (labels) is at least as coarse as b: rows b puts together, a puts together"""
    a, b = np.asarray(a, dtype=np.int64), np.asarray(b, dtype=np.int64)
    return bool(np.array_equal(a, a[b - begin]))


@pytest.mark.parametrize("case", ["coarse", "full", "legacy", "u16_big", "k8_u16"])
def test_components_vs_reference(built_lib, ctx, case):
    """coarse form (t = 0.9, 0.5), full form (t = 0 and the smallest positive double), row-streaming form
    (MC2_SWEEP_LEGACY=1), u16 counts above 255, k = 8 u16 wide rows; the whole set and a row range with begin > 0 and a
    query sub-range, on one and on both strands"""
    capi = built_lib
    rng = np.random.default_rng(47 if case == "k8_u16" else ["coarse", "full", "legacy", "u16_big"].index(case) + 20)
    k, eb, D, Q = _strand_data(rng, case)
    H = np.concatenate([D[0], Q[0]])            # a set in which about a quarter of the rows are other rows' reverse complements
    mag, ln = np.concatenate([D[1], Q[1]]), np.concatenate([D[2], Q[2]])
    n = len(H)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, k, mag=mag, length=ln)
    ts = {"full": (0.0, TINY), "coarse": (0.9, 0.5)}.get(case, (0.5,))
    if case != "full":
        ts += (_edge_t(ctx, gm, hs),)
    runs = [dict(), dict(range=(5, n - 3), q_range=(8, n - 10))]
    seen = []

    def go():
        for t in ts:
            for kw in runs:
                for both in (False, True):
                    _flat(ctx, gm, hs, t, both, kw.get("q_range", kw.get("range", (0, n))), kw.get("range", (0, n)), max_out=1)
                    sweep = ctx.last_sweep()
                    got, want = _check(ctx, gm, hs, t, both, **kw)
                    # one block: the sweeps of the flat call, on each strand
                    assert ctx.last_sweep()["n_exact"] == sweep["n_exact"]
                    assert ctx.last_sweep()["coarse"] == sweep["coarse"]
                    if case == "coarse":
                        assert ctx.last_sweep()["coarse"]
                    seen.append(_nontrivial(got))
    _legacy(go) if case == "legacy" else go()
    assert case == "full" or any(seen)


def test_both_strands_bridge_groups(built_lib, ctx):
    """on a set in which reverse complements of rows stand for their originals, the both-strand partition equals the
    reference of identity_pairs_both_strands' edges and is strictly coarser than the forward one"""
    capi = built_lib
    rng = np.random.default_rng(20)
    k, eb, D, Q = _strand_data(rng, "coarse")
    H = np.concatenate([D[0], Q[0]])
    mag, ln = np.concatenate([D[1], Q[1]]), np.concatenate([D[2], Q[2]])
    om = _model(H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, k, mag=mag, length=ln)
    for t in (0.9, 0.5, _edge_t(ctx, gm, hs)):
        one, _ = _check(ctx, gm, hs, t, False)
        two, _ = _check(ctx, gm, hs, t, True)
        assert _coarser(two["label"], one["label"])
    assert two["n_components"] < one["n_components"] and _nontrivial(two)


def test_components_vs_oracle(built_lib, ctx):
    """at least as coarse as the components of the oracle's edges with identity >= t + 1e-9, at least as fine as those of
    its edges with identity >= t - 1e-9, on one and on both strands"""
    capi = built_lib
    rng = np.random.default_rng(20)
    k, eb, D, Q = _strand_data(rng, "coarse")
    H = np.concatenate([D[0], Q[0]])
    mag, ln = np.concatenate([D[1], Q[1]]), np.concatenate([D[2], Q[2]])
    n = len(H)
    S = (H, mag, ln)
    om = _model(H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, k, mag=mag, length=ln)
    qs, ds = _window(ln, ln, 0.9, (0, n), (0, n), True)
    fwd = _oracle_identity(om, S, S, qs, ds)
    rev = _oracle_identity(om, (_rc_rows(H, k), mag, ln), S, qs, ds)
    for both, ident in ((False, fwd), (True, np.maximum(fwd, rev))):
        for t in (0.9, 0.5, _edge_t(ctx, gm, hs)):
            got = _comp(ctx, gm, hs, t, both)
            strict, _ = _canonical(n, qs[ident >= t + 1e-9], ds[ident >= t + 1e-9])
            loose, _ = _canonical(n, qs[ident >= t - 1e-9], ds[ident >= t - 1e-9])
            assert _coarser(got["label"], strict) and _coarser(loose, got["label"])
        assert _nontrivial(got)


def test_components_are_transitive(built_lib, ctx):
    """a mutation walk: single linkage puts two rows without an edge between them into one component"""
    capi = built_lib
    from meshclust2_b200 import synth
    rng = np.random.default_rng(5)
    walk = [synth.random_template(rng, 1000)]
    for _ in range(39):
        walk.append(synth.mutate(rng, walk[-1], 0.02))
    hs = ctx.count_kmers(ctx.seqs_from_text([bytes(x) for x in walk]), 5, 1)
    F = hs.download()
    om = _spread(all_singles_model(FLAGS5, F["hist"], F["mag"], F["len"], rng, n_combos=4), F["hist"], F["mag"], F["len"], rng)
    gm = _regression(ctx, capi, om)
    n = len(walk)
    every = ctx.identity_pairs(gm, hs, hs, -np.inf, 0.5, upper_only=True, max_out=n * n)
    assert every["n_out"] == n * (n - 1) // 2
    found = False
    for t in np.quantile(every["identity"], np.linspace(0.05, 0.95, 19)):
        got, want = _check(ctx, gm, hs, t, cutoff=0.5)
        edges = {(int(q), int(d)) for q, d in zip(want["q"], want["d"])}
        lab = got["label"]
        found = any(lab[i] == lab[j] and (i, j) not in edges for i in range(n) for j in range(i + 1, n))
        if found:
            break
    assert found


def _big_case(ctx, capi, seed, n, dense=False):
    """dense: the default spread of the identities, under which most in-window pairs have identity > 0"""
    rng = np.random.default_rng(seed)
    H, mag, ln = _big(rng, n)
    om = (_spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng) if dense else
          _model(H, mag, ln, rng))
    gm = _regression(ctx, capi, om)
    return gm, ctx.hset_from_host(H, 5, mag=mag, length=ln)


def test_block_split_on_each_strand(built_lib, ctx):
    """8 000 rows at the smallest positive t: more forward survivors than one block's scratch holds, and more reverse ones,
    so the block loop splits on each strand; the labels still equal the reference"""
    n = 8000
    gm, hs = _big_case(ctx, built_lib, 97, n, dense=True)
    fwd = ctx.identity_pairs(gm, hs, hs, TINY, 0.9, upper_only=True, max_out=1)
    rev = ctx.identity_pairs(gm, hs.reverse_complement(), hs, TINY, 0.9, upper_only=True, max_out=1)
    assert fwd["n_out"] > SCRATCH and rev["n_out"] > SCRATCH
    for both in (False, True):
        cap = fwd["n_out"] + (rev["n_out"] if both else 0)
        _check(ctx, gm, hs, TINY, both, max_out=cap)


def test_ranges_and_merge(built_lib, ctx):
    """begin > 0; a query range split over three calls and joined by components_merge equals one call; an empty query range
    gives every row its own label; the same call twice gives the same labels"""
    n = 1500
    gm, hs = _big_case(ctx, built_lib, 61, n)
    b0, b1 = 37, n - 11
    t = _edge_t(ctx, gm, hs)
    for both in (False, True):
        whole, _ = _check(ctx, gm, hs, t, both, range=(b0, b1))
        assert _nontrivial(whole)
        cuts = (b0, 400, 401, 1100, b1)
        parts = [_comp(ctx, gm, hs, t, both, q_range=(cuts[i], cuts[i + 1]), range=(b0, b1)) for i in range(4)]
        for p, (q0, q1) in zip(parts, zip(cuts[:-1], cuts[1:])):
            want = _reference(ctx, gm, hs, t, both, q_range=(q0, q1), range=(b0, b1))
            assert np.array_equal(p["label"], want["label"]) and p["n_components"] == want["n_components"]
        assert sum(p["n_scored"] for p in parts) == whole["n_scored"]
        m = ctx.components_merge(np.stack([p["label"] for p in parts]), b0)
        assert np.array_equal(m["label"], whole["label"]) and m["n_components"] == whole["n_components"]
        assert all(p["n_components"] > whole["n_components"] for p in parts)    # each part alone joins less
        again = _comp(ctx, gm, hs, t, both, range=(b0, b1))
        assert np.array_equal(again["label"], whole["label"])
        empty = _comp(ctx, gm, hs, 0.5, both, q_range=(200, 200), range=(b0, b1))
        assert np.array_equal(empty["label"], np.arange(b0, b1, dtype=np.uint64))
        assert empty["n_components"] == b1 - b0 and empty["n_scored"] == 0
    # merging a partition with itself, or with the identity partition, changes nothing
    ident = np.arange(b0, b1, dtype=np.uint64)
    m = ctx.components_merge(np.stack([whole["label"], ident, whole["label"]]), b0)
    assert np.array_equal(m["label"], whole["label"])
    got = _comp(ctx, gm, hs, 0.5, range=(300, 300))
    assert len(got["label"]) == 0 and got["n_components"] == 0


def test_errors(built_lib, ctx, golden):
    capi = built_lib
    L = capi.lib()
    H, ln = golden["hist_k5_eb1"][:4], golden["len_k5_eb1"][:4].copy()
    om = port.Model.from_text(weights_text("weights_cfg1_id90"))       # uses length_difference
    gm = ctx.model(to_desc(capi, om, regression=1))
    hs = ctx.hset_from_host(H, 5, length=ln)
    for model, t in ((ctx.model_from_file(weights_path("weights_cfg1_id90")), 0.5), (gm, float("nan"))):
        with pytest.raises(capi.Mc2Error) as e:
            _comp(ctx, model, hs, t)
        assert e.value.status == -1
    for kw in (dict(range=(0, 5)), dict(range=(1, 3), q_range=(0, 2)), dict(range=(1, 3), q_range=(2, 4)),
               dict(q_range=(3, 2)), dict(range=(3, 2)), dict(cutoff=0.0)):
        with pytest.raises(capi.Mc2Error) as e:
            _comp(ctx, gm, hs, 0.5, **kw)
        assert e.value.status == -1
    out = np.zeros(4, dtype=np.uint64)
    nc = C.c_uint64()
    for args in ((None, out.ctypes.data, C.byref(nc)), (hs.h, None, C.byref(nc)), (hs.h, out.ctypes.data, None)):
        assert L.mc2_identity_components(ctx.h, gm.h, 0.5, 0, args[0], 0, 4, 0, 4, 0.9, args[1], args[2], None) == -1
    ln0 = ln.copy()
    ln0[1] = ln0[2] = 0                                               # (1, 2): an upper-triangle pair in the window
    h0 = ctx.hset_from_host(H, 5, length=ln0)
    for both in (False, True):
        with pytest.raises(capi.Mc2Error) as e:                      # Feature::length_difference throws 123
            _comp(ctx, gm, h0, 0.5, both, q_range=(1, 2), range=(0, 4))
        assert e.value.status == -4
    # merge: no part, a label outside [begin, end), a range of 2^32 rows
    with pytest.raises(capi.Mc2Error) as e:
        ctx.components_merge(np.zeros((0, 4), dtype=np.uint64), 0)
    assert e.value.status == -1
    for bad in (np.array([[10, 10, 12, 14]]), np.array([[10, 10, 9, 11]])):
        with pytest.raises(capi.Mc2Error) as e:
            ctx.components_merge(bad, 10)
        assert e.value.status == -1
    lab = np.zeros(1, dtype=np.uint64)
    assert L.mc2_components_merge(ctx.h, 0, 1 << 32, 1, lab.ctypes.data, out.ctypes.data, C.byref(nc)) == -1


def test_all_pairs_step_components_equals_context_call(built_lib, ctx):
    """multi-GPU driver at world 1 through GpuEngine == Context.identity_components, on one and on both strands"""
    import torch
    from meshclust2_b200 import dist as mdist
    from meshclust2_b200 import synth
    capi = built_lib
    seqs, _ = synth.make_set(500, 1000, 30, 0.08, seed=6)
    enc = capi.encode_batch(seqs)
    n = len(seqs)
    cls = ctx.model_from_file(weights_path("weights_cfg1_id90"))
    eng = mdist.GpuEngine(capi, ctx, torch, cls, 5, 1, 0)
    eng.set_local_sequences(ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"]), n, n)
    pts = [port.get_point(s, 5, 1) for s in seqs]
    H = np.stack([p["hist"] for p in pts])
    mag = np.array([p["mag"] for p in pts], dtype=np.uint64)
    ln = np.array([p["len"] for p in pts], dtype=np.uint64)
    gm = _regression(ctx, capi, _model(H, mag, ln, np.random.default_rng(3)))
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    t = _edge_t(ctx, gm, hs)
    for both in (False, True):
        res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n, 0.9, upper_only=True, blocks_per_rank=3,
                                   identity=(gm, t, both), components=True)
        want = _comp(ctx, gm, hs, t, both)
        assert len(res["blocks"]) == 3
        assert np.array_equal(res["components"]["label"], want["label"])
        assert res["components"]["n_components"] == want["n_components"]
        assert res["n_scored"] == want["n_scored"] and len(res["survivors"]) == 0
        assert _nontrivial(want)
