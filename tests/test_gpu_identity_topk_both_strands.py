"""GPU: both-strand top-K identity search (mc2_identity_topk_both_strands).  The reference is
mc2_identity_pairs_both_strands with room for every survivor, sorted per query on the host by (identity descending,
database row ascending) and cut to K; d, identity bits and strand are compared exactly.  Also against the oracle's
predict_pair on both strands, against mc2_score_pairs on the reported strand, on the coarse, full and row-streaming forms,
at the K edges, on ties across strands at the K-th slot, with the block split forced on either strand, and with
exclude_self."""
import numpy as np
import pytest

from conftest import weights_path, weights_text
from helpers import all_singles_model, to_desc
from oracle import port
from test_gpu_both_strands import _big, _rc_rows, _strand_data
from test_gpu_identity_pairs import FLAGS5, TINY, _legacy, _oracle_identity, _regression, _spread, _window

pytestmark = pytest.mark.gpu

NONE = np.iinfo(np.uint64).max
SCRATCH = 1 << 22           # survivors one block's sweep of one strand holds (d ranges below it)


def _ranges(hq, hd, q_range, d_range):
    return q_range or (0, len(hq)), d_range or (0, len(hd))


def _reference(ctx, gm, hq, hd, t, K, cutoff=0.9, q_range=None, d_range=None, upper=False, exclude_self=False):
    """identity_pairs_both_strands, sorted per query: dict(d, identity, strand, count, n_hits, n_scored, n_out, lists) with
    lists[i] = (d[], identity[], strand[]) of query q0 + i in the output order"""
    (q0, q1), (d0, d1) = _ranges(hq, hd, q_range, d_range)
    r = ctx.identity_pairs_both_strands(gm, hq, hd, t, cutoff, q_range=(q0, q1), d_range=(d0, d1), upper_only=upper,
                                        max_out=max(1, (q1 - q0) * (d1 - d0)))
    q, d, s, st = r["q"].astype(np.int64), r["d"].astype(np.int64), r["identity"], r["strand"]
    if exclude_self:
        keep = q != d
        q, d, s, st = q[keep], d[keep], s[keep], st[keep]
    order = np.lexsort((d, -s, q))              # numeric: -(-0.0) and -(+0.0) compare equal, so they tie and d decides
    q, d, s, st = q[order], d[order], s[order], st[order]
    nq = q1 - q0
    out = dict(d=np.full((nq, K), NONE, dtype=np.uint64), identity=np.full((nq, K), -1.0),
               strand=np.full((nq, K), -1, dtype=np.int8), count=np.zeros(nq, dtype=np.uint32),
               n_hits=np.zeros(nq, dtype=np.uint64), n_scored=r["n_scored"], n_out=r["n_out"], lists=[])
    starts = np.searchsorted(q, np.arange(q0, q1 + 1))
    for i in range(nq):
        a, b = starts[i], starts[i + 1]
        m = min(K, b - a)
        out["d"][i, :m] = d[a:a + m]
        out["identity"][i, :m] = s[a:a + m]
        out["strand"][i, :m] = st[a:a + m]
        out["count"][i], out["n_hits"][i] = m, b - a
        out["lists"].append((d[a:b], s[a:b], st[a:b]))
    return out


def _topk(ctx, gm, hq, hd, t, K, cutoff=0.9, q_range=None, d_range=None, upper=False, exclude_self=False):
    return ctx.identity_topk_both_strands(gm, hq, hd, t, K, cutoff, q_range=q_range, d_range=d_range, upper_only=upper,
                                          exclude_self=exclude_self)


def _same(got, want):
    assert np.array_equal(got["d"], want["d"])
    assert np.array_equal(got["identity"].view(np.uint64), want["identity"].view(np.uint64))
    assert np.array_equal(got["strand"], want["strand"])
    assert np.array_equal(got["count"], want["count"]) and np.array_equal(got["n_hits"], want["n_hits"])
    assert got["n_scored"] == want["n_scored"]


def _check(ctx, gm, hq, hd, t, K, **kw):
    want = _reference(ctx, gm, hq, hd, t, K, **kw)
    got = _topk(ctx, gm, hq, hd, t, K, **kw)
    _same(got, want)
    return got, want


def _check_oracle(om, Q, D, k, got, t, K, cutoff, q_range, d_range, upper):
    """identities within 1e-9 of max(predict fwd, predict on the reverse-complement rows); the strand agrees where the two
    strands differ by more than 1e-9; the chosen rows are the oracle's top K except pairs within 1e-9 of t or of the K-th
    identity"""
    qs, ds = _window(Q[2], D[2], cutoff, q_range, d_range, upper)
    fwd = _oracle_identity(om, Q, D, qs, ds)
    rev = _oracle_identity(om, (_rc_rows(Q[0], k), Q[1], Q[2]), D, qs, ds)
    starts = np.searchsorted(qs, np.arange(q_range[0], q_range[1] + 1))
    for i in range(q_range[1] - q_range[0]):
        a, b = starts[i], starts[i + 1]
        v = {c: (max(f, r), f, r) for c, f, r in zip(ds[a:b].tolist(), fwd[a:b].tolist(), rev[a:b].tolist())}
        hits = sorted((-s, c) for c, (s, _, _) in v.items() if s >= t)
        top = {c for _, c in hits[:K]}
        kth = -hits[K - 1][0] if len(hits) >= K else None
        edge = {c for c, (s, _, _) in v.items() if abs(s - t) <= 1e-9 or (kth is not None and abs(s - kth) <= 1e-9)}
        n = int(got["count"][i])
        row = got["d"][i, :n].tolist()
        assert set(row) - edge == top - edge, i
        for c, s, st in zip(row, got["identity"][i, :n], got["strand"][i, :n]):
            best, f, r = v[c]
            assert abs(s - best) <= 1e-9
            if abs(f - r) > 1e-9:
                assert st == (1 if r > f else 0), (i, c)


def _check_score_pairs(ctx, gm, hq, hd, got, q_range):
    """every filled slot is the bits mc2_score_pairs gives the pair on its reported strand"""
    filled = got["strand"] >= 0
    assert np.array_equal(filled, got["d"] != NONE)
    rows = np.broadcast_to(np.arange(q_range[0], q_range[1], dtype=np.uint64)[:, None], got["d"].shape)
    for strand, hb in ((0, hq), (1, hq.reverse_complement())):
        sel = got["strand"] == strand
        if sel.any():
            sc = ctx.score_pairs(gm, hd, hb, got["d"][sel], rows[sel], want=("score",))["score"]
            assert np.array_equal(sc.view(np.uint64), got["identity"][sel].view(np.uint64))


@pytest.mark.parametrize("case", ["coarse", "full", "legacy", "u16_big", "k8_u16"])
def test_topk_both_strands_vs_reference_and_oracle(built_lib, ctx, case):
    """coarse form (t = 0.9, 0.5), full form (t <= 0: no reverse sweep; the smallest positive double), row-streaming form
    (MC2_SWEEP_LEGACY=1), u16 counts above 255, k = 8 u16 wide rows; upper triangle, ragged rectangle with q_begin > 0,
    and a query set (half of it reverse complements of database rows) other than the database set"""
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
                ctx.identity_pairs_both_strands(gm, hs, hd, t, 0.9, q_range=qr, d_range=dr, upper_only=upper, max_out=1)
                sweep = ctx.last_sweep()
                got, want = _check(ctx, gm, hs, hd, t, K, q_range=qr, d_range=dr, upper=upper)
                assert ctx.last_sweep() == sweep    # one block: the same sweeps of both strands as the flat call
                assert int(got["n_hits"].sum()) == want["n_out"]
                if case == "coarse":
                    assert sweep["coarse"]
                if t == 0.5:
                    assert got["count"].any() and int(got["n_hits"].sum()) < got["n_scored"]
                if S is Q and t == 0.5:
                    filled = got["strand"][got["strand"] >= 0]
                    assert (filled == 0).any() and (filled == 1).any()
                _check_oracle(om, S, D, k, got, t, K, 0.9, qr, dr, upper)
                _check_score_pairs(ctx, gm, hs, hd, got, qr)
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
    # K above every hit count: every row padded with d = 2^64 - 1, identity -1.0, strand -1
    K = int(hits.max()) + 3
    got, _ = _check(ctx, gm, hs, hs, 0.5, K, **sub)
    for i in range(300):
        c = int(got["count"][i])
        assert c == hits[i] < K
        assert (got["d"][i, c:] == NONE).all() and (got["identity"][i, c:] == -1.0).all() and (got["strand"][i, c:] == -1).all()
    # K = 1024 against rows of about 1 500 hits on each strand: the radix select keeps 1 024 and sorts them
    for t in (0.0, TINY):
        got, want = _check(ctx, gm, hs, hs, t, 1024, cutoff=0.5)   # a window wide enough for every length
        assert np.array_equal(got["count"], np.minimum(want["n_hits"], 1024)) and (want["n_hits"] > 1024).any()
        assert (got["strand"] == 1).any() and (got["strand"] == 0).any()
        if t == 0.0:
            assert (want["n_hits"] == n).all()
    got = _topk(ctx, gm, hs, hs, -np.inf, 3, upper=True)
    assert int(got["n_hits"].sum()) == got["n_scored"] > 0          # t <= 0: every in-window pair is a hit
    for t in (np.nextafter(1.0, 2.0), np.inf):                        # t > 1: no query has a hit
        got = _topk(ctx, gm, hs, hs, t, 3, upper=True)
        assert not got["count"].any() and not got["n_hits"].any() and got["n_scored"] > 0
        assert (got["d"] == NONE).all() and (got["identity"] == -1.0).all() and (got["strand"] == -1).all()
    # empty ranges
    got = _topk(ctx, gm, hs, hs, 0.5, 4, q_range=(7, 7))
    assert got["d"].shape == got["strand"].shape == (0, 4) and got["n_scored"] == 0
    got = _topk(ctx, gm, hs, hs, 0.5, 4, q_range=(7, 10), d_range=(20, 20))
    assert not got["count"].any() and not got["n_hits"].any() and (got["d"] == NONE).all() and (got["strand"] == -1).all()


def test_ties_across_strands_at_the_kth_slot(built_lib, ctx):
    """a database of 12 base rows and their reverse complements, each repeated 15 times, under a model without EMD (its
    features do not change when both operands' bins are permuted alike): id-(q, rc(B)) = id+(q, B) bit for bit, so a base
    row's 30 copies tie, and where one strand of the pair beats the other, the copies of B and of rc(B) report opposite
    strands.  Such ties straddle the K-th slot; the lower database rows win and each entry keeps its own strand."""
    capi = built_lib
    rng = np.random.default_rng(83)
    B, _, lb = _big(rng, 12)
    Bx = np.concatenate([B, _rc_rows(B, 5)])
    rep = np.repeat(np.arange(24), 15)
    rng.shuffle(rep)
    H, ln = Bx[rep], np.concatenate([lb, lb])[rep]
    mag = H.sum(axis=1, dtype=np.uint64)
    Q, _, lq = _big(rng, 40)
    pick = rng.integers(0, 12, 20)
    Q[:20] = B[pick]
    lq[:20] = lb[pick]
    for r in range(20):                                               # near copies, not exact ones
        Q[r, rng.integers(0, 1024, 3)] += 1
    mq = Q.sum(axis=1, dtype=np.uint64)
    flags = [port.FEAT[x] for x in ("euclidean", "manhattan", "pearson", "length_difference")]
    om = _spread(all_singles_model(flags, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hd = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    hq = ctx.hset_from_host(Q, 5, mag=mq, length=lq)
    for t, K in ((0.0, 17), (TINY, 17), (0.0, 45)):
        want = _reference(ctx, gm, hq, hd, t, K, cutoff=0.5)
        cross = 0
        for i, (d, s, st) in enumerate(want["lists"]):
            if len(s) > K and s[K - 1] == s[K]:
                tie = s == s[K - 1]
                cross += set(st[tie].tolist()) == {0, 1}
        assert cross > 0                                              # the reference has ties across strands at slot K
        got = _topk(ctx, gm, hq, hd, t, K, cutoff=0.5)
        _same(got, want)
        for i, (d, s, st) in enumerate(want["lists"]):
            if len(s) > K and s[K - 1] == s[K]:
                m = got["identity"][i, :K] == s[K - 1]
                assert np.all(np.diff(got["d"][i, :K][m].astype(np.int64)) > 0)     # lower database rows first
                # the winners are the tie's lowest rows, each with the strand the flat search reports for it
                strand_of = dict(zip(d.tolist(), st.tolist()))
                assert [strand_of[int(c)] for c in got["d"][i, :K][m]] == got["strand"][i, :K][m].tolist()


def _block_case(ctx, capi, seed):
    rng = np.random.default_rng(seed)
    n = 5000
    H, mag, ln = _big(rng, n)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    return n, gm, ctx.hset_from_host(H, 5, mag=mag, length=ln)


def _split_equals_whole(ctx, gm, hs, n, t, K, got):
    parts = [_topk(ctx, gm, hs, hs, t, K, q_range=r) for r in ((0, 1234), (1234, 1235), (1235, 3900), (3900, n))]
    for f in ("d", "identity", "strand", "count", "n_hits"):
        cat = np.concatenate([p[f] for p in parts])
        assert np.array_equal(cat.view(np.uint8), got[f].view(np.uint8)), f
    assert sum(p["n_scored"] for p in parts) == got["n_scored"]


def test_block_split_forward(built_lib, ctx):
    """5 000 x 5 000 at t <= 0: about 23 M hits, more than one block's forward scratch holds (no reverse sweep).  Equal to
    the reference, and bit-identical to the same search run as separate query sub-ranges and concatenated"""
    n, gm, hs = _block_case(ctx, built_lib, 73)
    K = 16
    got, _ = _check(ctx, gm, hs, hs, 0.0, K)
    assert int(got["n_hits"].sum()) == got["n_scored"] > 2 * SCRATCH
    assert (got["strand"] == 1).any() and (got["strand"] == 0).any()
    _split_equals_whole(ctx, gm, hs, n, 0.0, K, got)


def test_block_split_reverse(built_lib, ctx):
    """5 000 x 5 000 at t = 0.5: the reverse strand alone has more survivors than its scratch holds, so the block loop
    splits on it.  Equal to the reference and to the same search over query sub-ranges; exclude_self on the split search"""
    n, gm, hs = _block_case(ctx, built_lib, 89)
    t, K = 0.5, 10
    rev = ctx.identity_pairs(gm, hs.reverse_complement(), hs, t, 0.9, max_out=1)
    assert rev["n_out"] > SCRATCH
    got, want = _check(ctx, gm, hs, hs, t, K)
    assert want["n_out"] > SCRATCH and (got["strand"] == 1).any() and (got["strand"] == 0).any()
    _split_equals_whole(ctx, gm, hs, n, t, K, got)
    ex, _ = _check(ctx, gm, hs, hs, t, K, exclude_self=True)
    rows = np.arange(n, dtype=np.uint64)
    assert not (ex["d"] == rows[:, None]).any()


def test_exclude_self(built_lib, ctx):
    capi = built_lib
    rng = np.random.default_rng(79)
    H, mag, ln = _big(rng, 400)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    for t, K, qr in ((0.5, 6, None), (0.0, 400, (17, 333)), (TINY, 50, (40, 200))):
        with_self = _topk(ctx, gm, hs, hs, t, K, q_range=qr)
        got, _ = _check(ctx, gm, hs, hs, t, K, q_range=qr, exclude_self=True)
        q0 = qr[0] if qr else 0
        rows = np.arange(q0, q0 + len(got["d"]), dtype=np.uint64)
        assert not (got["d"] == rows[:, None]).any()
        # exactly the rows whose self pair is a hit, on either strand, lose one hit (at t <= 0, every row)
        ip = ctx.identity_pairs_both_strands(gm, hs, hs, t, 0.9, q_range=(q0, q0 + len(rows)), max_out=len(rows) * len(H))
        self_hit = np.isin(rows, ip["q"][ip["q"] == ip["d"]]).astype(np.uint64)
        assert np.array_equal(with_self["n_hits"] - got["n_hits"], self_hit)
        if t <= 0:
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
    for K in (0, 1025):
        with pytest.raises(capi.Mc2Error) as e:
            _topk(ctx, gm, hs, hs, 0.5, K)
        assert e.value.status == -1
    for kw in (dict(q_range=(0, 5)), dict(d_range=(2, 5)), dict(cutoff=0.0)):
        with pytest.raises(capi.Mc2Error) as e:
            _topk(ctx, gm, hs, hs, 0.5, 4, **kw)
        assert e.value.status == -1
    h6 = ctx.hset_from_host(np.ones((4, 4096), dtype=np.uint8), 6, length=ln)
    with pytest.raises(capi.Mc2Error) as e:                          # the two sets differ in k
        _topk(ctx, gm, hs, h6, 0.5, 4)
    assert e.value.status == -1
    ln0 = ln.copy()
    ln0[1] = 0
    hs = ctx.hset_from_host(H, 5, length=ln0)
    with pytest.raises(capi.Mc2Error) as e:                          # Feature::length_difference throws 123
        _topk(ctx, gm, hs, hs, 0.5, 4, q_range=(1, 2), d_range=(0, 4))
    assert e.value.status == -4


def test_all_pairs_step_topk_both_strands_equals_context_call(built_lib, ctx):
    """multi-GPU driver at world 1 through GpuEngine == Context.identity_topk_both_strands"""
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
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, np.random.default_rng(3), n_combos=4), H, mag, ln, np.random.default_rng(4))
    gm = _regression(ctx, capi, om)
    res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n, 0.9, upper_only=True, blocks_per_rank=3,
                               identity=(gm, 0.5, True), top_k=8)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    want = _topk(ctx, gm, hs, hs, 0.5, 8, upper=True)
    assert [b[:2] for b in res["topk"]] == res["blocks"] and len(res["blocks"]) == 3
    for f in ("d", "identity", "strand", "count", "n_hits"):
        cat = np.concatenate([tb[f] for _, _, tb in res["topk"]])
        assert np.array_equal(cat.view(np.uint8), want[f].view(np.uint8)), f
    assert res["n_close"] == int(want["n_hits"].sum()) and res["n_scored"] == want["n_scored"]
    assert 0 < res["n_close"] < res["n_scored"] and len(res["survivors"]) == 0
