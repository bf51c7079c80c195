"""GPU: greedy representative clustering (mc2_identity_greedy_clusters).  The reference is a plain sequential greedy pass on
the host over the flat search's edges (mc2_identity_pairs over the upper triangle, or mc2_identity_pairs_both_strands, with
room for every survivor); rep, the bits of identity, strand, n_clusters and n_scored are compared exactly.  Also its
structure (an independent set of representatives, members tied to an earlier representative by an edge, clusters inside
single-linkage components), the oracle's predict_pair, deep dependency chains, ties, both strands and the block split."""
import ctypes as C

import numpy as np
import pytest

from conftest import weights_path, weights_text
from helpers import all_singles_model, to_desc
from oracle import port
from test_gpu_both_strands import _rc_rows, _strand_data
from test_gpu_identity_components import SCRATCH, _big_case, _comp, _edge_t, _model
from test_gpu_identity_pairs import FLAGS5, TINY, _legacy, _oracle_identity, _regression, _spread, _window

pytestmark = pytest.mark.gpu


def _greedy(n, begin, q, d, ident, strand=None):
    """the sequential pass: rows in order, a row is a representative unless an earlier one has an edge to it; a member
    takes its heaviest edge from an earlier representative, the smallest such row on a numeric tie"""
    r = np.asarray(q, dtype=np.int64) - begin
    c = np.asarray(d, dtype=np.int64) - begin
    ident = np.asarray(ident, dtype=np.float64)
    st = np.zeros(len(r), dtype=np.int8) if strand is None else np.asarray(strand, dtype=np.int8)
    o = np.lexsort((r, -ident, c))              # per c: identity descending (-0.0 equal to +0.0), then r ascending
    r, c, ident, st = r[o], c[o], ident[o], st[o]
    starts = np.searchsorted(c, np.arange(n + 1))
    is_rep = np.zeros(n, dtype=bool)
    rep = np.arange(begin, begin + n, dtype=np.uint64)
    out_id = np.full(n, -1.0)
    out_str = np.full(n, -1, dtype=np.int8)
    for i in range(n):
        a, b = starts[i], starts[i + 1]
        hit = np.flatnonzero(is_rep[r[a:b]])
        if len(hit) == 0:
            is_rep[i] = True
        else:
            k = a + hit[0]
            rep[i] = begin + r[k]
            out_id[i] = ident[k]
            out_str[i] = st[k]
    return dict(rep=rep, identity=out_id, strand=out_str, n_clusters=int(is_rep.sum()))


def _flat(ctx, gm, hs, t, both, rng_, cutoff, max_out=None):
    b0, b1 = rng_
    call = ctx.identity_pairs_both_strands if both else ctx.identity_pairs
    r = call(gm, hs, hs, t, cutoff, q_range=rng_, d_range=rng_, upper_only=True, max_out=max_out or max(1, (b1 - b0) ** 2))
    assert len(r["q"]) == r["n_out"]                    # room for every edge
    return r


def _greedy_call(ctx, gm, hs, t, both=False, range=None, cutoff=0.9):
    return ctx.identity_greedy_clusters(gm, hs, t, cutoff, both_strands=both, range=range)


def _check(ctx, gm, hs, t, both=False, range=None, cutoff=0.9, max_out=None, structure=True):
    rng_ = range or (0, len(hs))
    b0, b1 = rng_
    flat = _flat(ctx, gm, hs, t, both, rng_, cutoff, max_out)
    want = _greedy(b1 - b0, b0, flat["q"], flat["d"], flat["identity"], flat["strand"] if both else None)
    got = _greedy_call(ctx, gm, hs, t, both, range, cutoff)
    assert got["rep"].dtype == np.uint64
    assert np.array_equal(got["rep"], want["rep"])
    assert np.array_equal(got["identity"].view(np.uint64), want["identity"].view(np.uint64))
    assert np.array_equal(got["strand"], want["strand"])
    assert got["n_clusters"] == want["n_clusters"] and got["n_scored"] == flat["n_scored"]
    if structure:
        _check_structure(ctx, gm, hs, t, both, rng_, cutoff, got, flat)
    return got, flat


def _check_structure(ctx, gm, hs, t, both, rng_, cutoff, got, flat):
    b0, b1 = rng_
    rows = np.arange(b0, b1, dtype=np.uint64)
    w = {(int(q), int(d)): (v, s) for q, d, v, s in zip(flat["q"], flat["d"], flat["identity"],
                                                        flat["strand"] if both else np.zeros(len(flat["q"]), np.int8))}
    is_rep = got["rep"] == rows
    assert got["n_clusters"] == int(is_rep.sum())
    assert (got["identity"][is_rep] == -1.0).all() and (got["strand"][is_rep] == -1).all()
    reps = set(rows[is_rep].tolist())
    assert not any(q in reps and d in reps for q, d in w)                  # an independent set
    for i in np.flatnonzero(~is_rep):
        r, c = int(got["rep"][i]), int(rows[i])
        assert r < c and r in reps and (r, c) in w                          # an earlier representative, by an edge
        v, s = w[(r, c)]
        assert got["identity"][i] == v and got["strand"][i] == s
    comp = _comp(ctx, gm, hs, t, both, range=rng_, cutoff=cutoff)
    lab = comp["label"]
    assert np.array_equal(lab[got["rep"].astype(np.int64) - b0], lab)       # a cluster lies inside one component
    assert got["n_clusters"] >= comp["n_components"]


@pytest.mark.parametrize("case", ["coarse", "full", "legacy", "u16_big", "k8_u16"])
def test_greedy_vs_reference(built_lib, ctx, case):
    """coarse form (t = 0.9, 0.5), full form (t = 0 and the smallest positive double), row-streaming form
    (MC2_SWEEP_LEGACY=1), u16 counts above 255, k = 8 u16 wide rows; the whole set and a row range with begin > 0, on one
    and on both strands; the sweeps are those of the flat call"""
    capi = built_lib
    rng = np.random.default_rng(47 if case == "k8_u16" else ["coarse", "full", "legacy", "u16_big"].index(case) + 20)
    k, eb, D, Q = _strand_data(rng, case)
    H = np.concatenate([D[0], Q[0]])            # a set in which about a quarter of the rows are other rows' reverse complements
    mag, ln = np.concatenate([D[1], Q[1]]), np.concatenate([D[2], Q[2]])
    n = len(H)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, k, mag=mag, length=ln)
    ts = (0.0, TINY) if case == "full" else (0.9, 0.5, _edge_t(ctx, gm, hs))
    seen = []

    def go():
        for t in ts:
            for rng_ in ((0, n), (5, n - 3)):
                for both in (False, True):
                    call = ctx.identity_pairs_both_strands if both else ctx.identity_pairs
                    call(gm, hs, hs, t, 0.9, q_range=rng_, d_range=rng_, upper_only=True, max_out=1)
                    sweep = ctx.last_sweep()
                    got = _greedy_call(ctx, gm, hs, t, both, rng_)
                    # one block: the sweeps of the flat call, on each strand
                    assert ctx.last_sweep()["n_exact"] == sweep["n_exact"]
                    assert ctx.last_sweep()["coarse"] == sweep["coarse"]
                    if case == "coarse":
                        assert ctx.last_sweep()["coarse"]
                    got, _ = _check(ctx, gm, hs, t, both, rng_)
                    seen.append(1 < got["n_clusters"] < rng_[1] - rng_[0])
    _legacy(go) if case == "legacy" else go()
    assert case == "full" or any(seen)


def test_greedy_vs_oracle(built_lib, ctx):
    """each member's identity to its representative is the oracle's within 1e-9 (on the reported strand) and >= t - 1e-9;
    every in-window pair of representatives scores < t + 1e-9 on both strands' better one"""
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
    fwd = np.full((n, n), -np.inf)
    rev = np.full((n, n), -np.inf)
    fwd[qs, ds] = _oracle_identity(om, S, S, qs, ds)
    rev[qs, ds] = _oracle_identity(om, (_rc_rows(H, k), mag, ln), S, qs, ds)
    seen = []
    for both in (False, True):
        best = np.maximum(fwd, rev) if both else fwd
        for t in (0.9, 0.5, _edge_t(ctx, gm, hs)):
            got = _greedy_call(ctx, gm, hs, t, both)
            rep = got["rep"].astype(np.int64)
            mem = np.flatnonzero(rep != np.arange(n))
            want = np.where(got["strand"][mem] == 1, rev[rep[mem], mem], fwd[rep[mem], mem])
            assert np.abs(got["identity"][mem] - want).max(initial=0) <= 1e-9
            assert (got["identity"][mem] >= t - 1e-9).all()
            reps = np.flatnonzero(rep == np.arange(n))
            assert (best[np.ix_(reps, reps)] < t + 1e-9).all()
            seen.append(1 < got["n_clusters"] < n)
    assert any(seen)


def _walk(ctx, capi, seed, n, rate):
    from meshclust2_b200 import synth
    rng = np.random.default_rng(seed)
    walk = [synth.random_template(rng, 1000)]
    for _ in range(n - 1):
        walk.append(synth.mutate(rng, walk[-1], rate))
    hs = ctx.count_kmers(ctx.seqs_from_text([bytes(x) for x in walk]), 5, 1)
    F = hs.download()
    om = _spread(all_singles_model(FLAGS5, F["hist"], F["mag"], F["len"], rng, n_combos=4), F["hist"], F["mag"], F["len"], rng)
    return _regression(ctx, capi, om), hs


def test_mutation_walk(built_lib, ctx):
    """a 40-row mutation walk at several t: exact, and at some t the representatives alternate along the walk (a member
    between two representatives that share no edge), which single linkage would have put in one cluster"""
    n = 40
    gm, hs = _walk(ctx, built_lib, 5, n, 0.02)
    every = ctx.identity_pairs(gm, hs, hs, -np.inf, 0.5, upper_only=True, max_out=n * n)
    assert every["n_out"] == n * (n - 1) // 2
    alternating = False
    for t in np.quantile(every["identity"], np.linspace(0.05, 0.95, 19)):
        got, _ = _check(ctx, gm, hs, t, cutoff=0.5)
        reps = np.flatnonzero(got["rep"] == np.arange(n))
        comp = _comp(ctx, gm, hs, t, cutoff=0.5)
        alternating |= any(b - a > 1 and comp["label"][a] == comp["label"][b] for a, b in zip(reps[:-1], reps[1:]))
    assert alternating


def test_deep_chain_in_one_block(built_lib, ctx):
    """a path of 3 000 rows in one block: identity = the length-difference similarity 1 - |len_r - len_c| / 64 and lengths
    1000 + 20 i, so at t = 0.5 the only edges are (i, i + 1) (0.6875; two rows apart 0.375).  Row i is undecided until row
    i - 1 is decided, a dependency chain through the whole block and its resolve rounds; the representatives are the even
    rows and each odd row goes to the row before it, on one and on both strands"""
    capi = built_lib
    from test_gpu_both_strands import _big
    rng = np.random.default_rng(9)
    n = 3000
    H, mag, _ = _big(rng, n)
    ln = (1000 + 20 * np.arange(n)).astype(np.uint64)
    flag = port.FEAT["length_difference"]
    gm = ctx.model(to_desc(capi, port.Model([(flag, 0.0, 64.0)], [(0, flag)], [0.0, 1.0]), regression=1))
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    rows = np.arange(n)
    for both in (False, True):
        got, flat = _check(ctx, gm, hs, 0.5, both, cutoff=0.5, structure=False)
        assert np.array_equal(np.sort(flat["q"].astype(np.int64)), rows[:-1])
        assert np.array_equal(flat["d"].astype(np.int64) - flat["q"].astype(np.int64), np.ones(n - 1, dtype=np.int64))
        assert np.array_equal(got["rep"].astype(np.int64), rows - rows % 2)
        assert got["n_clusters"] == n // 2 and (got["identity"][1::2] == 0.6875).all()


def test_ties_go_to_the_smaller_representative(built_lib, ctx):
    """groups of three rows: r1 (h, length 1000), r2 (h, length 1300) and m (h mutated, length 1120), cutoff 0.8: r1 and r2
    are outside each other's length window, so both can be representatives, and m is inside both; the features ignore
    length, so w(r1, m) and w(r2, m) are the same bits and m must go to r1"""
    capi = built_lib
    from test_gpu_both_strands import _big
    rng = np.random.default_rng(33)
    G = 30
    base, _, _ = _big(rng, G)
    rows, lens = [], []
    for g in range(G):
        h2 = base[g].copy()
        idx = rng.integers(0, h2.shape[0], 12)
        h2[idx] = h2[idx] + 1
        rows += [base[g], base[g], h2]
        lens += [1000, 1300, 1120]
    H = np.stack(rows)
    mag, ln = H.sum(axis=1, dtype=np.uint64), np.array(lens, dtype=np.uint64)
    flags = [port.FEAT[x] for x in ("euclidean", "emd", "manhattan", "pearson")]
    om = _spread(all_singles_model(flags, H, mag, ln, rng, n_combos=4), H, mag, ln, rng, lo=-1.0, hi=0.6)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    every = ctx.identity_pairs(gm, hs, hs, -np.inf, 0.8, upper_only=True, max_out=len(H) ** 2)
    w = {(int(a), int(b)): x for a, b, x in zip(every["q"], every["d"], every["identity"])}
    t = min(w[(3 * g, 3 * g + 2)] for g in range(G))
    assert all(w[(3 * g, 3 * g + 2)] == w[(3 * g + 1, 3 * g + 2)] for g in range(G))
    ties = 0
    for both in (False, True):
        got, _ = _check(ctx, gm, hs, t, both, cutoff=0.8)
        for g in range(G):
            r1, r2, m = 3 * g, 3 * g + 1, 3 * g + 2
            if got["rep"][r1] == r1 and got["rep"][r2] == r2:
                assert got["rep"][m] == r1
                ties += 1
    assert ties > 0


def test_negative_and_positive_zero_tie(built_lib, ctx):
    """identity = clamp(-0.0 - f): -0.0 or +0.0 on every pair, so at t = 0 every in-window pair is an edge of weight zero and
    every member goes to the smallest representative that reaches it, whichever zero it carries"""
    capi = built_lib
    from test_gpu_both_strands import _big
    rng = np.random.default_rng(71)
    n = 200
    H, mag, _ = _big(rng, n)
    ln = np.where(np.arange(n) % 3 == 0, 1064, 1000).astype(np.uint64)
    flag = port.FEAT["length_difference"]
    om = port.Model([(flag, 0.0, 64.0)], [(0, flag)], [-0.0, -1.0])
    gm = ctx.model(to_desc(capi, om, regression=1))
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    for both in (False, True):
        for rng_ in (None, (7, n - 5)):
            got, flat = _check(ctx, gm, hs, 0.0, both, range=rng_)
            assert (flat["identity"] == 0).all() and np.signbit(flat["identity"]).any()
            mem = got["identity"] != -1.0
            assert np.signbit(got["identity"][mem]).any() and (~np.signbit(got["identity"][mem])).any()


def test_reverse_complements_join_on_strand_1(built_lib, ctx):
    """a database of rows followed by their reverse complements: on both strands complements join forward representatives
    as members on strand 1, and there are fewer clusters than on one strand"""
    capi = built_lib
    from test_gpu_both_strands import _big
    rng = np.random.default_rng(8)
    m = 150
    F, fmag, fln = _big(rng, m)
    H = np.concatenate([F, _rc_rows(F, 5)])
    mag, ln = np.concatenate([fmag, fmag]), np.concatenate([fln, fln])
    om = _model(H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    t = _edge_t(ctx, gm, hs)
    one, _ = _check(ctx, gm, hs, t, False)
    two, _ = _check(ctx, gm, hs, t, True)
    joined = (two["rep"][m:] < m) & (two["strand"][m:] == 1)
    assert joined.any()
    assert two["n_clusters"] < one["n_clusters"]


def test_block_split_on_each_strand(built_lib, ctx):
    """8 000 rows at the smallest positive t: more survivors than one block's scratch holds on each strand, so the block
    loop splits and each row's best in-edge carries across blocks; the result still equals the reference"""
    n = 8000
    gm, hs = _big_case(ctx, built_lib, 97, n, dense=True)
    fwd = ctx.identity_pairs(gm, hs, hs, TINY, 0.9, upper_only=True, max_out=1)
    rev = ctx.identity_pairs(gm, hs.reverse_complement(), hs, TINY, 0.9, upper_only=True, max_out=1)
    assert fwd["n_out"] > SCRATCH and rev["n_out"] > SCRATCH
    for both in (False, True):
        cap = fwd["n_out"] + (rev["n_out"] if both else 0)
        _check(ctx, gm, hs, TINY, both, max_out=cap, structure=False)


def test_errors(built_lib, ctx, golden):
    capi = built_lib
    L = capi.lib()
    H, ln = golden["hist_k5_eb1"][:4], golden["len_k5_eb1"][:4].copy()
    om = port.Model.from_text(weights_text("weights_cfg1_id90"))       # uses length_difference
    gm = ctx.model(to_desc(capi, om, regression=1))
    hs = ctx.hset_from_host(H, 5, length=ln)
    for model, t in ((ctx.model_from_file(weights_path("weights_cfg1_id90")), 0.5), (gm, float("nan"))):
        with pytest.raises(capi.Mc2Error) as e:
            _greedy_call(ctx, model, hs, t)
        assert e.value.status == -1
    for kw in (dict(range=(0, 5)), dict(range=(3, 2)), dict(cutoff=0.0), dict(cutoff=-1.0)):
        with pytest.raises(capi.Mc2Error) as e:
            _greedy_call(ctx, gm, hs, 0.5, **kw)
        assert e.value.status == -1
    out = np.zeros(4, dtype=np.uint64)
    nc = C.c_uint64()
    for args in ((None, out.ctypes.data, C.byref(nc)), (hs.h, None, C.byref(nc)), (hs.h, out.ctypes.data, None)):
        assert L.mc2_identity_greedy_clusters(ctx.h, gm.h, 0.5, 0, args[0], 0, 4, 0.9, args[1], None, None, args[2], None) == -1
    # out_identity, out_strand and n_scored may be NULL
    assert L.mc2_identity_greedy_clusters(ctx.h, gm.h, 0.5, 1, hs.h, 0, 4, 0.9, out.ctypes.data, None, None, C.byref(nc),
                                          None) == 0
    assert 1 <= nc.value <= 4
    ln0 = ln.copy()
    ln0[1] = ln0[2] = 0                                               # (1, 2): an upper-triangle pair in the window
    h0 = ctx.hset_from_host(H, 5, length=ln0)
    for both in (False, True):
        with pytest.raises(capi.Mc2Error) as e:                      # Feature::length_difference throws 123
            _greedy_call(ctx, gm, h0, 0.5, both)
        assert e.value.status == -4
    got = _greedy_call(ctx, gm, hs, 0.5, range=(2, 2))
    assert len(got["rep"]) == 0 and got["n_clusters"] == 0
    one = _greedy_call(ctx, gm, hs, 0.5, True, range=(3, 4))
    assert one["rep"].tolist() == [3] and one["n_clusters"] == 1 and one["strand"].tolist() == [-1]
