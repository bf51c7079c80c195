"""GPU: top-K identity search (mc2_identity_topk).  The reference is mc2_identity_pairs with room for every survivor, sorted
per query on the host by (identity descending, database row ascending) and cut to K; identities are compared bit for bit.
Also against the oracle's predict_pair, on the coarse, full and row-streaming forms of the sweep, at the K edges, on ties,
with the block split forced by more survivors than the scratch holds, and with exclude_self."""
import numpy as np
import pytest

from conftest import weights_path, weights_text
from helpers import all_singles_model, to_desc
from oracle import port
from test_gpu_both_strands import _big, _strand_data
from test_gpu_identity_pairs import FLAGS5, TINY, _legacy, _oracle_identity, _regression, _spread, _window

pytestmark = pytest.mark.gpu

NONE = np.iinfo(np.uint64).max


def _ranges(hq, hd, q_range, d_range):
    return q_range or (0, len(hq)), d_range or (0, len(hd))


def _reference(ctx, gm, hq, hd, t, K, cutoff=0.9, q_range=None, d_range=None, upper=False, exclude_self=False):
    """identity_pairs, sorted per query: dict(d, identity, count, n_hits, n_scored, lists) with lists[i] = (d[], identity[])
    of query q0 + i in the output order"""
    (q0, q1), (d0, d1) = _ranges(hq, hd, q_range, d_range)
    r = ctx.identity_pairs(gm, hq, hd, t, cutoff, q_range=(q0, q1), d_range=(d0, d1), upper_only=upper,
                           max_out=max(1, (q1 - q0) * (d1 - d0)))
    q, d, s = r["q"].astype(np.int64), r["d"].astype(np.int64), r["identity"]
    if exclude_self:
        keep = q != d
        q, d, s = q[keep], d[keep], s[keep]
    order = np.lexsort((d, -s, q))              # numeric: -(-0.0) and -(+0.0) compare equal, so they tie and d decides
    q, d, s = q[order], d[order], s[order]
    nq = q1 - q0
    out = dict(d=np.full((nq, K), NONE, dtype=np.uint64), identity=np.full((nq, K), -1.0), count=np.zeros(nq, dtype=np.uint32),
               n_hits=np.zeros(nq, dtype=np.uint64), n_scored=r["n_scored"], lists=[])
    starts = np.searchsorted(q, np.arange(q0, q1 + 1))
    for i in range(nq):
        a, b = starts[i], starts[i + 1]
        m = min(K, b - a)
        out["d"][i, :m] = d[a:a + m]
        out["identity"][i, :m] = s[a:a + m]
        out["count"][i], out["n_hits"][i] = m, b - a
        out["lists"].append((d[a:b], s[a:b]))
    return out


def _topk(ctx, gm, hq, hd, t, K, cutoff=0.9, q_range=None, d_range=None, upper=False, exclude_self=False):
    return ctx.identity_topk(gm, hq, hd, t, K, cutoff, q_range=q_range, d_range=d_range, upper_only=upper,
                             exclude_self=exclude_self)


def _same(got, want):
    assert np.array_equal(got["d"], want["d"])
    assert np.array_equal(got["identity"].view(np.uint64), want["identity"].view(np.uint64))
    assert np.array_equal(got["count"], want["count"]) and np.array_equal(got["n_hits"], want["n_hits"])
    assert got["n_scored"] == want["n_scored"]


def _check(ctx, gm, hq, hd, t, K, **kw):
    want = _reference(ctx, gm, hq, hd, t, K, **kw)
    got = _topk(ctx, gm, hq, hd, t, K, **kw)
    _same(got, want)
    return got, want


def _check_oracle(om, Q, D, got, t, K, cutoff, q_range, d_range, upper):
    """identities within 1e-9 of predict_pair; the chosen rows are the oracle's top K except pairs within 1e-9 of t or of
    the K-th identity"""
    qs, ds = _window(Q[2], D[2], cutoff, q_range, d_range, upper)
    ref = _oracle_identity(om, Q, D, qs, ds)
    starts = np.searchsorted(qs, np.arange(q_range[0], q_range[1] + 1))
    for i in range(q_range[1] - q_range[0]):
        a, b = starts[i], starts[i + 1]
        v = dict(zip(ds[a:b].tolist(), ref[a:b].tolist()))
        hits = sorted((-s, c) for c, s in v.items() if s >= t)
        top = {c for _, c in hits[:K]}
        kth = -hits[K - 1][0] if len(hits) >= K else None
        edge = {c for c, s in v.items() if abs(s - t) <= 1e-9 or (kth is not None and abs(s - kth) <= 1e-9)}
        n = int(got["count"][i])
        row = got["d"][i, :n].tolist()
        assert set(row) - edge == top - edge, i
        for c, s in zip(row, got["identity"][i, :n]):
            assert abs(s - v[c]) <= 1e-9


@pytest.mark.parametrize("case", ["coarse", "full", "legacy", "u16_big", "k8_u16"])
def test_topk_vs_reference_and_oracle(built_lib, ctx, case):
    """coarse form (t = 0.9, 0.5), full form (t <= 0, the smallest positive double), row-streaming form
    (MC2_SWEEP_LEGACY=1, u16 counts above 255), k = 8 u16 wide rows; upper triangle, ragged rectangle with q_begin > 0,
    and a query set other than the database set"""
    capi = built_lib
    rng = np.random.default_rng(47 if case == "k8_u16" else ["coarse", "full", "legacy", "u16_big"].index(case) + 20)
    k, eb, D, Q = _strand_data(rng, case)
    n, nq = len(D[0]), len(Q[0])
    om = _spread(all_singles_model(FLAGS5, D[0], D[1], D[2], rng, n_combos=4), D[0], D[1], D[2], rng)
    gm = _regression(ctx, capi, om)
    hd = ctx.hset_from_host(D[0], k, mag=D[1], length=D[2])
    hq = ctx.hset_from_host(Q[0], k, mag=Q[1], length=Q[2])
    ts = {"full": (0.0, TINY), "coarse": (0.9, 0.5)}.get(case, (0.5,))
    runs = [(D, hd, (0, n), (0, n), True), (D, hd, (3, n - 7), (5, n - 2), False), (Q, hq, (1, nq - 2), (2, n - 3), False)]

    def go():
        for t in ts:
            for j, (S, hs, qr, dr, upper) in enumerate(runs):
                K = (1, 5, 12)[j]
                ip = ctx.identity_pairs(gm, hs, hd, t, 0.9, q_range=qr, d_range=dr, upper_only=upper, max_out=1)
                sweep = ctx.last_sweep()
                got, want = _check(ctx, gm, hs, hd, t, K, q_range=qr, d_range=dr, upper=upper)
                assert ctx.last_sweep() == sweep            # one block: the diagnostics of the one sweep
                assert int(got["n_hits"].sum()) == ip["n_out"] and got["n_scored"] == ip["n_scored"]
                if case == "coarse":
                    assert sweep["coarse"]
                if t == 0.5:
                    assert got["count"].any() and int(got["n_hits"].sum()) < got["n_scored"]
                _check_oracle(om, S, D, got, t, K, 0.9, qr, dr, upper)
    _legacy(go) if case == "legacy" else go()


def test_k_edges(built_lib, ctx):
    capi = built_lib
    rng = np.random.default_rng(61)
    n = 1500
    H, mag, ln = _big(rng, n)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    sub = dict(q_range=(0, 300), d_range=(0, 300), upper=True)
    want = _reference(ctx, gm, hs, hs, 0.5, 1, **sub)
    hits = want["n_hits"].astype(np.int64)
    assert hits.max() > 1 and (hits == 0).any()
    _same(_topk(ctx, gm, hs, hs, 0.5, 1, **sub), want)
    # K equal to a query's hit count: that row is full, without padding
    r = int(np.argmax(hits))
    K = int(hits[r])
    got, _ = _check(ctx, gm, hs, hs, 0.5, K, **sub)
    assert got["count"][r] == K and (got["d"][r] != NONE).all()
    # K above every hit count: every row padded with d = 2^64 - 1, identity -1.0
    K = K + 3
    got, _ = _check(ctx, gm, hs, hs, 0.5, K, **sub)
    for i in range(300):
        c = int(got["count"][i])
        assert c == hits[i] < K
        assert (got["d"][i, c:] == NONE).all() and (got["identity"][i, c:] == -1.0).all()
    # K = 1024 against rows of about 1 500 hits: the radix select keeps 1 024 and sorts them
    got, want = _check(ctx, gm, hs, hs, 0.0, 1024, cutoff=0.5)     # a window wide enough for every length
    assert (want["n_hits"] == n).all() and (got["count"] == 1024).all()
    assert int(got["n_hits"].sum()) == got["n_scored"]          # t <= 0: every in-window pair is a hit
    for t in (-1.0, -np.inf):
        got = _topk(ctx, gm, hs, hs, t, 3, upper=True)
        assert int(got["n_hits"].sum()) == got["n_scored"] > 0
    for t in (np.nextafter(1.0, 2.0), 1.5, np.inf):              # t > 1: no query has a hit
        got = _topk(ctx, gm, hs, hs, t, 3, upper=True)
        assert not got["count"].any() and not got["n_hits"].any() and got["n_scored"] > 0
        assert (got["d"] == NONE).all() and (got["identity"] == -1.0).all()
    for K in (0, 1025):
        with pytest.raises(capi.Mc2Error) as e:
            _topk(ctx, gm, hs, hs, 0.5, K)
        assert e.value.status == -1
    # empty ranges
    got = _topk(ctx, gm, hs, hs, 0.5, 4, q_range=(7, 7))
    assert got["d"].shape == (0, 4) and got["n_scored"] == 0
    got = _topk(ctx, gm, hs, hs, 0.5, 4, q_range=(7, 10), d_range=(20, 20))
    assert not got["count"].any() and not got["n_hits"].any() and (got["d"] == NONE).all() and (got["identity"] == -1.0).all()


def test_ties_on_duplicated_database_rows(built_lib, ctx):
    """database rows repeated 30 times: equal identities straddle the K-th slot and are taken in database-row order"""
    capi = built_lib
    rng = np.random.default_rng(67)
    B, mb, lb = _big(rng, 12)
    rep = np.repeat(np.arange(12), 30)
    rng.shuffle(rep)
    H, mag, ln = B[rep], mb[rep], lb[rep]
    Q, mq, lq = _big(rng, 40)
    Q[:20] = B[rng.integers(0, 12, 20)]
    mq[:20] = Q[:20].sum(axis=1, dtype=np.uint64)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hd = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    hq = ctx.hset_from_host(Q, 5, mag=mq, length=lq)
    for t, K in ((0.0, 5), (0.3, 17), (0.0, 45)):
        got, want = _check(ctx, gm, hq, hd, t, K)
        straddle = 0
        for i, (d, s) in enumerate(want["lists"]):
            if len(s) > K and s[K - 1] == s[K]:
                straddle += 1
                m = s[:K] == s[K - 1]
                assert np.all(np.diff(got["d"][i, :K][m].astype(np.int64)) > 0)
        assert straddle > 0


def test_negative_and_positive_zero_tie(built_lib, ctx):
    """identity = clamp(-0.0 - f): -0.0 where the length-difference similarity f is 0 (lengths 64 apart), +0.0 where it
    is 1 (equal lengths).  The two zeros compare equal, so each row is ordered by database row alone."""
    capi = built_lib
    rng = np.random.default_rng(71)
    n = 80
    H, mag, _ = _big(rng, n)
    ln = np.where(np.arange(n) % 3 == 0, 1064, 1000).astype(np.uint64)
    flag = port.FEAT["length_difference"]
    om = port.Model([(flag, 0.0, 64.0)], [(0, flag)], [-0.0, -1.0])
    gm = ctx.model(to_desc(capi, om, regression=1))
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    for upper, K in ((False, 10), (True, 7), (False, 200)):
        got, want = _check(ctx, gm, hs, hs, 0.0, K, upper=upper)
        ids = got["identity"][got["identity"] != -1.0]
        assert (ids == 0).all() and np.signbit(ids).any() and (~np.signbit(ids)).any()
        for i in range(n):
            c = int(got["count"][i])
            assert np.all(np.diff(got["d"][i, :c].astype(np.int64)) > 0)
            assert c == min(K, n - (i + 1 if upper else 0))


def test_block_split(built_lib, ctx):
    """5 000 x 5 000 at t <= 0: about 23 M hits, more than the 2^22-pair scratch of one block.  Equal to the reference, and
    bit-identical to the same search run as separate query sub-ranges and concatenated"""
    capi = built_lib
    rng = np.random.default_rng(73)
    n = 5000
    H, mag, ln = _big(rng, n)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    K = 16
    got, want = _check(ctx, gm, hs, hs, 0.0, K)
    assert int(got["n_hits"].sum()) == got["n_scored"] > 2 * (1 << 22)
    parts = [_topk(ctx, gm, hs, hs, 0.0, K, q_range=r) for r in ((0, 1234), (1234, 1235), (1235, 3900), (3900, n))]
    for f in ("d", "identity", "count", "n_hits"):
        cat = np.concatenate([p[f] for p in parts])
        assert np.array_equal(cat.view(np.uint8), got[f].view(np.uint8)), f
    assert sum(p["n_scored"] for p in parts) == got["n_scored"]
    # the same split search with exclude_self: the reference without the pairs (r, r)
    got, _ = _check(ctx, gm, hs, hs, 0.0, K, exclude_self=True)
    assert int(got["n_hits"].sum()) == got["n_scored"] - n


def test_exclude_self(built_lib, ctx):
    capi = built_lib
    rng = np.random.default_rng(79)
    H, mag, ln = _big(rng, 400)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    for t, K, qr in ((0.5, 6, None), (0.0, 400, (17, 333))):
        with_self = _topk(ctx, gm, hs, hs, t, K, q_range=qr)
        got, _ = _check(ctx, gm, hs, hs, t, K, q_range=qr, exclude_self=True)
        q0 = qr[0] if qr else 0
        rows = np.arange(q0, q0 + len(got["d"]), dtype=np.uint64)
        assert not (got["d"] == rows[:, None]).any()
        # exactly the rows whose self pair is an identity_pairs survivor lose one hit (at t <= 0, every row)
        ip = ctx.identity_pairs(gm, hs, hs, t, 0.9, q_range=(q0, q0 + len(rows)), max_out=len(rows) * len(H))
        self_hit = np.isin(rows, ip["q"][ip["q"] == ip["d"]]).astype(np.uint64)
        assert np.array_equal(with_self["n_hits"] - got["n_hits"], self_hit)
        if t <= 0:                  # every row's self pair is a hit, and K holds all of a row's hits
            assert (with_self["d"] == rows[:, None]).any(axis=1).all()
            assert np.array_equal(with_self["n_hits"] - got["n_hits"], np.ones(len(rows), dtype=np.uint64))
    other = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    with pytest.raises(capi.Mc2Error) as e:
        _topk(ctx, gm, hs, other, 0.5, 4, exclude_self=True)
    assert e.value.status == -1


def test_errors(built_lib, ctx, golden):
    capi = built_lib
    H, ln = golden["hist_k5_eb1"][:4], golden["len_k5_eb1"][:4].copy()
    om = port.Model.from_text(weights_text("weights_cfg1_id90"))       # uses length_difference
    gm = ctx.model(to_desc(capi, om, regression=1))
    hs = ctx.hset_from_host(H, 5, length=ln)
    for model, t in ((ctx.model_from_file(weights_path("weights_cfg1_id90")), 0.5), (gm, float("nan"))):
        with pytest.raises(capi.Mc2Error) as e:
            _topk(ctx, model, hs, hs, t, 4)
        assert e.value.status == -1
    with pytest.raises(capi.Mc2Error) as e:
        _topk(ctx, gm, hs, hs, 0.5, 4, q_range=(0, 5))
    assert e.value.status == -1
    ln0 = ln.copy()
    ln0[1] = 0
    hs = ctx.hset_from_host(H, 5, length=ln0)
    with pytest.raises(capi.Mc2Error) as e:                          # Feature::length_difference throws 123
        _topk(ctx, gm, hs, hs, 0.5, 4, q_range=(1, 2), d_range=(0, 4))
    assert e.value.status == -4


def test_all_pairs_step_topk_equals_context_call(built_lib, ctx):
    """multi-GPU driver at world 1 through GpuEngine == Context.identity_topk"""
    import torch
    from meshclust2_b200 import dist as mdist
    from meshclust2_b200 import synth
    capi = built_lib
    seqs, _ = synth.make_set(600, 1000, 30, 0.08, seed=7)
    enc = capi.encode_batch(seqs)
    n = len(seqs)
    cls = ctx.model_from_file(weights_path("weights_cfg1_id90"))
    eng = mdist.GpuEngine(capi, ctx, torch, cls, 5, 1, 0)
    eng.set_local_sequences(ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"]), n, n)
    pts = [port.get_point(s, 5, 1) for s in seqs]
    H = np.stack([p["hist"] for p in pts])
    mag = np.array([p["mag"] for p in pts], dtype=np.uint64)
    ln = np.array([p["len"] for p in pts], dtype=np.uint64)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, np.random.default_rng(3), n_combos=4), H, mag, ln, np.random.default_rng(4))
    gm = _regression(ctx, capi, om)
    res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n, 0.9, upper_only=True, blocks_per_rank=3, identity=(gm, 0.5),
                               top_k=8)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    want = _topk(ctx, gm, hs, hs, 0.5, 8, upper=True)
    assert [b[:2] for b in res["topk"]] == res["blocks"] and len(res["blocks"]) == 3
    for f in ("d", "identity", "count", "n_hits"):
        cat = np.concatenate([tb[f] for _, _, tb in res["topk"]])
        assert np.array_equal(cat.view(np.uint8), want[f].view(np.uint8)), f
    assert res["n_close"] == int(want["n_hits"].sum()) and res["n_scored"] == want["n_scored"]
