"""GPU: the other DNA strand.  mc2_hset_reverse_complement against the oracle counting the mirrored sequences (reverse the
codes, c -> 3 - c, segment [s, e] -> [L-1-e, L-1-s]); mc2_identity_pairs_both_strands against the oracle's predict_pair on
both strands of every in-window pair, against mc2_score_pairs bit for bit on the reported strand, on the coarse, full and
row-streaming forms, with the block split of the reverse sweep forced by millions of survivors."""

import numpy as np
import pytest

from conftest import weights_path, weights_text
from helpers import all_singles_model, synth_hist, to_desc
from oracle import port
from test_gpu_identity_pairs import FLAGS5, TINY, _legacy, _oracle_identity, _regression, _spread, _window

pytestmark = pytest.mark.gpu


def _rc_perm(k):
    """rc[j] = bin of the reverse complement of k-mer j (big-endian base 4, A=0 C=1 G=2 T=3)"""
    j = np.arange(4 ** k, dtype=np.int64)
    r = np.zeros_like(j)
    for p in range(k):
        r = r * 4 + (3 - ((j >> (2 * p)) & 3))
    return r


def _rc_rows(H, k):
    """host reverse complement of histogram rows: out[:, rc(j)] = H[:, j]"""
    out = np.empty_like(H)
    out[:, _rc_perm(k)] = H
    return out


def _mirror(codes, segs):
    L = len(codes)
    c = codes[::-1].copy()
    inside = (c >= 0) & (c <= 3)
    c[inside] = 3 - c[inside]
    s = np.stack([L - 1 - segs[::-1, 1], L - 1 - segs[::-1, 0]], axis=1).astype(np.int32) if len(segs) else segs
    return c, s


def _texts(rng, n, lo=300, hi=900, u8_saturation=False):
    """random reads; some with N runs (several segments), some with runs of A (saturated bins)"""
    out = []
    for i in range(n):
        L = int(rng.integers(lo, hi))
        t = bytearray(rng.choice(list(b"ACGT"), L).astype(np.uint8).tobytes())
        if i % 3 == 1:
            for _ in range(int(rng.integers(1, 4))):
                p, m = int(rng.integers(0, L - 20)), int(rng.integers(1, 15))
                t[p:p + m] = b"N" * m
        if i % 5 == 2:
            p = int(rng.integers(0, L // 2))
            t[p:p + 120] = b"A" * 120
        out.append(bytes(t[:L]))
    if u8_saturation:
        out += [b"A" * 258, b"A" * 259, b"A" * 400, b"C" * 30 + b"A" * 259 + b"G" * 30]   # a count of 254, 255 and above
    return out


def _upload(ctx, encs):
    codes = np.concatenate([e[0] for e in encs]).astype(np.int8)
    seq_off = np.zeros(len(encs) + 1, dtype=np.uint64)
    seq_off[1:] = np.cumsum([len(e[0]) for e in encs])
    segs = np.concatenate([e[1].reshape(-1, 2) for e in encs]).astype(np.int32)
    seg_off = np.zeros(len(encs) + 1, dtype=np.uint64)
    seg_off[1:] = np.cumsum([len(e[1]) for e in encs])
    return ctx.upload_seqs(codes, seq_off, segs, seg_off)


KE = [(1, 1), (2, 2), (3, 4), (5, 8), (5, 1), (6, 2), (8, 1), (8, 2), (9, 4), (11, 1)]


@pytest.mark.parametrize("k,eb", KE, ids=["k%d_u%d" % (k, 8 * eb) for k, eb in KE])
def test_reverse_complement_vs_oracle(built_lib, ctx, k, eb):
    rng = np.random.default_rng(100 * k + eb)
    texts = _texts(rng, 4 if k >= 9 else 24, u8_saturation=eb == 1)
    encs = [port.encode(t)[:2] for t in texts]
    hs = ctx.count_kmers(_upload(ctx, encs), k, eb)
    rc = hs.reverse_complement()
    fwd, got = hs.download(), rc.download()
    for i, (codes, segs) in enumerate(encs):
        mc, ms = _mirror(codes, segs)
        h, m1, _ = port.count(mc, ms, k, eb)
        assert np.array_equal(got["hist"][i], h), i
        assert np.array_equal(got["mers1"][i], m1), i
    assert np.array_equal(got["mers1"], fwd["mers1"][:, ::-1])
    for f in ("mag", "len", "stddev", "max_count"):
        assert np.array_equal(got[f], fwd[f]), f
    assert not got["n_overflow"].any()
    if eb == 1:
        assert fwd["n_overflow"].any() and (fwd["hist"] == 255).any()
    assert rc.largest_count() == hs.largest_count()
    assert np.array_equal(got["hist"], _rc_rows(fwd["hist"], k))
    back = rc.reverse_complement().download()
    assert np.array_equal(back["hist"], fwd["hist"]) and np.array_equal(back["mers1"], fwd["mers1"])


def test_reverse_complement_keeps_stale_magnitudes(built_lib, ctx):
    rng = np.random.default_rng(5)
    H = synth_hist(rng, 50, 6, 2, hi=9)
    ln = rng.integers(900, 1100, 50).astype(np.uint64)
    mag = H.sum(axis=1, dtype=np.uint64) + 13
    rc = ctx.hset_from_host(H, 6, mag=mag, length=ln).reverse_complement().download()
    assert np.array_equal(rc["mag"], mag) and np.array_equal(rc["len"], ln)
    assert np.array_equal(rc["hist"], _rc_rows(H, 6))


def test_reverse_complement_of_text(built_lib, ctx):
    """pure-ACGT reads: reverse complement of the counted set == K1 of the reverse-complemented text"""
    rng = np.random.default_rng(8)
    texts = [bytes(rng.choice(list(b"ACGT"), int(rng.integers(200, 1500))).astype(np.uint8).tobytes()) for _ in range(64)]
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    rct = [t.translate(comp)[::-1] for t in texts]
    for k, eb in ((5, 1), (7, 2)):
        a = ctx.count_kmers(ctx.seqs_from_text(texts), k, eb).reverse_complement().download()
        b = ctx.count_kmers(ctx.seqs_from_text(rct), k, eb).download()
        for f in ("hist", "mers1", "mag", "len"):
            assert np.array_equal(a[f], b[f]), f


# ---- both-strand identity search -------------------------------------------------------------------------------------

def _both(ctx, gm, hq, hd, t, cutoff=0.9, q_range=None, d_range=None, upper=False, max_out=None):
    if max_out is None:
        max_out = max(1, (q_range[1] - q_range[0] if q_range else len(hq)) * (d_range[1] - d_range[0] if d_range else len(hd)))
    return ctx.identity_pairs_both_strands(gm, hq, hd, t, cutoff, q_range=q_range, d_range=d_range, upper_only=upper,
                                           max_out=max_out)


def _check_both(ctx, om, gm, Q, D, hq, hd, k, cutoff, q_range, d_range, upper, t):
    qs, ds = _window(Q[2], D[2], cutoff, q_range, d_range, upper)
    fwd = _oracle_identity(om, Q, D, qs, ds)
    Qr = (_rc_rows(Q[0], k), Q[1], Q[2])
    rev = _oracle_identity(om, Qr, D, qs, ds)
    r = _both(ctx, gm, hq, hd, t, cutoff, q_range, d_range, upper)
    one = ctx.identity_pairs(gm, hq, hd, t, cutoff, q_range=q_range, d_range=d_range, upper_only=upper, max_out=1)
    assert r["n_scored"] == one["n_scored"] == len(qs)
    best = np.maximum(fwd, rev)
    ref = {key: (b, f, v) for key, b, f, v in zip(zip(qs.tolist(), ds.tolist()), best, fwd, rev)}
    got = {(int(q), int(d)): (s, int(st)) for q, d, s, st in zip(r["q"], r["d"], r["identity"], r["strand"])}
    assert r["n_out"] == len(got) == len(r["q"])
    edge = {key for key, (b, _, _) in ref.items() if abs(b - t) <= 1e-9}
    assert set(got) - edge == {key for key, (b, _, _) in ref.items() if b >= t} - edge
    for key, (s, st) in got.items():
        b, f, v = ref[key]
        assert abs(s - b) <= 1e-9
        if abs(f - v) > 1e-9:
            assert st == (1 if v > f else 0), key
    # bit-equal to mc2_score_pairs on the reported strand
    if got:
        hr = hq.reverse_complement()
        for strand, hb in ((0, hq), (1, hr)):
            sel = r["strand"] == strand
            if sel.any():
                sc = ctx.score_pairs(gm, hd, hb, r["d"][sel], r["q"][sel], want=("score",))["score"]
                assert np.array_equal(sc.view(np.uint64), r["identity"][sel].view(np.uint64))
    return r, ref


def _related(rng, n, k, extra, per_row):
    base = np.ones((max(2, n // 8), 4 ** k), dtype=np.int64)
    for r in range(len(base)):
        np.add.at(base[r], rng.integers(0, 4 ** k, extra), 1)
    H = base[rng.integers(0, len(base), n)]
    for r in range(n):
        np.add.at(H[r], rng.integers(0, 4 ** k, per_row), 1)
    return H


def _strand_data(rng, case):
    """database rows D and queries Q of which about half are reverse complements of database rows"""
    k, eb = {"k8_u16": (8, 2), "u16_big": (5, 2)}.get(case, (5, 1))
    if k == 8:
        n, nq = 110, 60
        H = _related(rng, n, 8, 20000, 300)
    else:
        n, nq = 300, 90
        H = _related(rng, n, 5, 400, 40)
    assert H.max() <= 255
    if case == "u16_big":
        H[7, 100] = 300
    Hq = H[rng.integers(0, n, nq)].copy()
    flip = rng.random(nq) < 0.5
    Hq[flip] = _rc_rows(Hq[flip], k)
    Hq[::7] += 1                           # not exact copies
    dt = port.DTYPES[eb]
    H, Hq = H.astype(dt), Hq.astype(dt)
    lnd = rng.integers(900, 1100, n).astype(np.uint64) * (20 if k > 5 else 1)
    lnq = rng.integers(900, 1100, nq).astype(np.uint64) * (20 if k > 5 else 1)
    return k, eb, (H, H.sum(axis=1, dtype=np.uint64), lnd), (Hq, Hq.sum(axis=1, dtype=np.uint64), lnq)


@pytest.mark.parametrize("case", ["coarse", "full", "legacy", "k8_u16", "u16_big"])
def test_both_strands_vs_oracle(built_lib, ctx, case):
    capi = built_lib
    # k8_u16: a seed whose spread model keeps identities inside (0, 1) (median 0.54 over both strands); for others it clamps
    rng = np.random.default_rng(47 if case == "k8_u16" else ["coarse", "full", "legacy", "k8_u16", "u16_big"].index(case) + 20)
    k, eb, D, Q = _strand_data(rng, case)
    n, nq = len(D[0]), len(Q[0])
    om = _spread(all_singles_model(FLAGS5, D[0], D[1], D[2], rng, n_combos=4), D[0], D[1], D[2], rng)
    gm = _regression(ctx, capi, om)
    hd = ctx.hset_from_host(D[0], k, mag=D[1], length=D[2])
    hq = ctx.hset_from_host(Q[0], k, mag=Q[1], length=Q[2])
    ts = {"full": (0.0, TINY)}.get(case, (0.5, 0.8))
    runs = [(D, hd, (0, n), (0, n), True), (D, hd, (3, n - 7), (5, n - 2), False), (Q, hq, (1, nq - 2), (2, n - 3), False)]

    def go():
        for t in ts:
            for S, hs, qr, dr, upper in runs:
                r, ref = _check_both(ctx, om, gm, S, D, hs, hd, k, 0.9, qr, dr, upper, t)
                if t > 0:
                    assert 0 < r["n_out"] < r["n_scored"]
                if S is Q and t > 0:
                    assert (r["strand"] == 1).any() and (r["strand"] == 0).any()
                if case == "coarse":
                    assert ctx.last_sweep()["coarse"]
    _legacy(go) if case == "legacy" else go()


def test_properties(built_lib, ctx):
    """one-strand survivors are both-strand survivors with at least that identity; a palindromic read x + rc(x) reports
    the forward strand; queries found in a database of their own reverse complements are found on the reverse strand"""
    capi = built_lib
    rng = np.random.default_rng(31)
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    xs = [bytes(rng.choice(list(b"ACGT"), int(rng.integers(450, 550))).astype(np.uint8).tobytes()) for _ in range(120)]
    pal = [x + x.translate(comp)[::-1] for x in xs[:40]]
    hx = ctx.count_kmers(ctx.seqs_from_text(xs), 5, 1)
    hrc = ctx.count_kmers(ctx.seqs_from_text([x.translate(comp)[::-1] for x in xs]), 5, 1)
    hp = ctx.count_kmers(ctx.seqs_from_text(pal), 5, 1)
    F = hx.download()
    om = _spread(all_singles_model(FLAGS5, F["hist"], F["mag"], F["len"], rng, n_combos=4), F["hist"], F["mag"], F["len"], rng)
    gm = _regression(ctx, capi, om)
    for t in (0.3, 0.7):
        one = ctx.identity_pairs(gm, hx, hx, t, 0.9, upper_only=True, max_out=120 * 120)
        both = _both(ctx, gm, hx, hx, t, upper=True)
        b = {(int(q), int(d)): s for q, d, s in zip(both["q"], both["d"], both["identity"])}
        for q, d, s in zip(one["q"], one["d"], one["identity"]):
            assert b[(int(q), int(d))] >= s
    r = _both(ctx, gm, hp, hp, TINY, cutoff=0.5)
    assert r["n_out"] > 0 and not r["strand"].any()
    r = _both(ctx, gm, hx, hrc, 0.9, cutoff=0.5)
    one = ctx.identity_pairs(gm, hx, hrc, 0.9, 0.5, max_out=120 * 120)
    fwd_self = {int(q) for q, d in zip(one["q"], one["d"]) if q == d}
    got = {int(q): int(st) for q, d, st in zip(r["q"], r["d"], r["strand"]) if q == d}
    assert set(got) == set(range(120))
    assert all(got[i] == 1 for i in range(120) if i not in fwd_self) and len(fwd_self) < 120


def _big(rng, n):
    H = synth_hist(rng, n, 5, 1, hi=6)
    ln = rng.integers(900, 1100, n).astype(np.uint64)
    return H, H.sum(axis=1, dtype=np.uint64), ln


def test_capacity(built_lib, ctx):
    capi = built_lib
    rng = np.random.default_rng(41)
    H, mag, ln = _big(rng, 400)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    for t in (0.5, 0.0):
        full = _both(ctx, gm, hs, hs, t, upper=True)
        allp = {(int(q), int(d)): (s, st) for q, d, s, st in zip(full["q"], full["d"], full["identity"], full["strand"])}
        assert full["n_out"] == len(allp) > 10
        for cap in (1, full["n_out"] // 2):
            part = _both(ctx, gm, hs, hs, t, upper=True, max_out=cap)
            assert part["n_out"] == full["n_out"] and len(part["q"]) == cap
            for q, d, s, st in zip(part["q"], part["d"], part["identity"], part["strand"]):
                assert allp[(int(q), int(d))] == (s, st)


def test_block_split_of_the_reverse_sweep(built_lib, ctx):
    """2 000 x 2 000 at the smallest positive t: millions of reverse-strand survivors, more than the scratch of one block
    holds, against one unconstrained scoring pass over every in-window pair on both strands"""
    capi = built_lib
    rng = np.random.default_rng(43)
    n = 2000
    H, mag, ln = _big(rng, n)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    hr = hs.reverse_complement()
    qs, ds = _window(ln, ln, 0.9, (0, n), (0, n), False)
    fwd = ctx.score_pairs(gm, hs, hs, ds, qs, want=("score",))["score"]
    rev = ctx.score_pairs(gm, hs, hr, ds, qs, want=("score",))["score"]
    assert (rev >= TINY).sum() > 2 * (1 << 20)
    r = _both(ctx, gm, hs, hs, TINY, max_out=len(qs))
    keep = np.maximum(fwd, rev) >= TINY
    assert r["n_out"] == int(keep.sum()) and r["n_scored"] == len(qs)
    key = lambda q, d: q.astype(np.int64) * n + d.astype(np.int64)
    order = np.argsort(key(r["q"], r["d"]))
    widx = np.flatnonzero(keep)
    worder = np.argsort(key(qs[widx], ds[widx]))
    assert np.array_equal(key(r["q"], r["d"])[order], key(qs[widx], ds[widx])[worder])
    want_id = np.where(rev > fwd, rev, fwd)[widx][worder]
    assert np.array_equal(r["identity"][order].view(np.uint64), want_id.view(np.uint64))
    assert np.array_equal(r["strand"][order], (rev > fwd)[widx][worder].astype(np.int8))


def test_errors(built_lib, ctx, golden):
    capi = built_lib
    H, ln = golden["hist_k5_eb1"][:4], golden["len_k5_eb1"][:4].copy()
    om = port.Model.from_text(weights_text("weights_cfg1_id90"))       # uses length_difference
    gm = ctx.model(to_desc(capi, om, regression=1))
    hs = ctx.hset_from_host(H, 5, length=ln)
    for model, t in ((ctx.model_from_file(weights_path("weights_cfg1_id90")), 0.5), (gm, float("nan"))):
        with pytest.raises(capi.Mc2Error) as e:
            ctx.identity_pairs_both_strands(model, hs, hs, t, 0.9)
        assert e.value.status == -1
    ln0 = ln.copy()
    ln0[1] = 0
    hs = ctx.hset_from_host(H, 5, length=ln0)
    with pytest.raises(capi.Mc2Error) as e:
        ctx.identity_pairs_both_strands(gm, hs, hs, 0.5, 0.9, q_range=(1, 2), d_range=(0, 4))
    assert e.value.status == -4


def test_all_pairs_step_both_strands_equals_context_call(built_lib, ctx):
    """multi-GPU driver at world 1 through GpuEngine == Context.identity_pairs_both_strands"""
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
    try:
        res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n, 0.9, upper_only=True, max_out=n * n,
                                   identity=(gm, 0.5, True))
        s = res["survivors"]
        got = {(int(q), int(d)): (v, int(st)) for (q, d), v, st in zip(s.tolist(), s.scores().view(np.uint64), s.strands())}
    finally:
        for slot in eng._surv_slots:
            for b in slot[3]:
                capi.host_unregister(b)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    r = _both(ctx, gm, hs, hs, 0.5, upper=True)
    want = {(int(q), int(d)): (v, int(st)) for q, d, v, st in zip(r["q"], r["d"], r["identity"].view(np.uint64), r["strand"])}
    assert got == want and res["n_close"] == r["n_out"] and res["n_scored"] == r["n_scored"] and 0 < len(want) < r["n_scored"]
