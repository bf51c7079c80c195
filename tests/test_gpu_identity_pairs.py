"""GPU: identity search (mc2_identity_pairs): every in-window pair scored with a regression model (Predictor<T>::similarity,
Predictor.cpp:284-300: the GLM sum clamped to [0, 1]), survivors = identity >= t.  Against the oracle's predict_pair over
all in-window pairs (FC_Runner.cpp:435-444 window, compute(database c, query r)), against mc2_score_pairs bit for bit, on
the tile form and the row-streaming form."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import weights_path, weights_text
from helpers import FAST, all_singles_model, synth_hist, to_desc
from oracle import port

pytestmark = pytest.mark.gpu

TINY = np.nextafter(0.0, 1.0)      # fastcar's `sim > 0`


def _window(lnq, lnd, cutoff, q_range, d_range, upper):
    """in-window (q, d) pairs of the reference's work() loop, q-major"""
    qs, ds = [], []
    d = np.arange(*d_range)
    for q in range(*q_range):
        lo, hi = int(float(lnq[q]) * cutoff), int(float(lnq[q]) / cutoff)
        ok = (lnd[d].astype(np.int64) >= lo) & (lnd[d].astype(np.int64) <= hi)
        if upper:
            ok &= d > q
        qs.append(np.full(int(ok.sum()), q))
        ds.append(d[ok])
    return np.concatenate(qs).astype(np.int64), np.concatenate(ds).astype(np.int64)


def _oracle_identity(om, Q, D, qs, ds):
    """oracle identities of pairs (query qs[i], database ds[i]) -- compute(database, query); Q / D = (H, mag, len)"""
    cm = om.cmodel()
    L = port.lib()
    out = np.empty(len(qs))
    v = C.c_double()
    Hq, mq, lq = Q
    Hd, md, ld = D
    for i, (q, d) in enumerate(zip(qs, ds)):
        a = port._pt(Hd[d], int(md[d]), int(ld[d]))
        b = port._pt(Hq[q], int(mq[q]), int(lq[q]))
        rc = L.mc2o_predict_pair(C.byref(cm), Hd.dtype.itemsize, C.c_uint64(Hd.shape[1]), C.byref(a), C.byref(b), C.byref(v))
        assert rc == 0
        out[i] = v.value
    return out


def _sums(om, H, mag, ln, rng, m=400):
    """unclamped GLM sums (intercept left out) of random pairs, through the classifier form: logit(logistic(sum))"""
    n = len(H)
    ia, ib = rng.integers(0, n, m), rng.integers(0, n, m)
    w0 = om.weights[0]
    om.weights[0] = 0.0
    s = np.clip(port.score_pairs(om, H, mag, ln, ia, ib, want_cache=False)["score"], 1e-15, 1 - 1e-15)
    om.weights[0] = w0
    return np.log(s / (1 - s))


def _spread(om, H, mag, ln, rng, lo=-0.2, hi=1.2):
    """rescale the weights affinely so that the sums of sampled pairs spread over about [lo, hi] (otherwise nearly every
    identity clamps to 0 or 1)"""
    s = _sums(om, H, mag, ln, rng)
    a, b = np.quantile(s, 0.05), np.quantile(s, 0.95)
    f = (hi - lo) / max(b - a, 1e-6)
    om.weights = [lo - f * a] + [w * f for w in om.weights[1:]]
    return om


def _regression(ctx, capi, om):
    return ctx.model(to_desc(capi, om, regression=1))


def _check_vs_oracle(ctx, capi, om, gm, Q, D, hq, hd, cutoff, q_range, d_range, upper, t):
    qs, ds = _window(Q[2], D[2], cutoff, q_range, d_range, upper)
    want = _oracle_identity(om, Q, D, qs, ds)
    r = ctx.identity_pairs(gm, hq, hd, t, cutoff, q_range=q_range, d_range=d_range, upper_only=upper, max_out=max(1, len(qs)))
    assert r["n_scored"] == len(qs)
    a = ctx.all_pairs(ctx.model(to_desc(capi, om)), hq, hd, cutoff, q_range=q_range, d_range=d_range, upper_only=upper, max_out=1)
    assert a["n_scored"] == len(qs)
    got = {(int(q), int(d)): s for q, d, s in zip(r["q"], r["d"], r["identity"])}
    assert r["n_out"] == len(got)
    ref = dict(zip(zip(qs.tolist(), ds.tolist()), want.tolist()))
    wset = {k for k, s in ref.items() if s >= t}
    edge = {k for k, s in ref.items() if abs(s - t) <= 1e-9}
    assert set(got) - edge == wset - edge
    for k, s in got.items():
        assert abs(s - ref[k]) <= 1e-9
    return r, ref


def _wide_hist(rng, n, k, eb, mean_extra):
    N = 4 ** k
    H = np.ones((n, N), dtype=np.int64)
    for r in range(n):
        np.add.at(H[r], rng.integers(0, N, mean_extra), 1)
    return H


def _related(rng, n, k, eb, extra, per_row=300):
    base = _wide_hist(rng, max(2, n // 8), k, eb, extra)
    H = base[rng.integers(0, len(base), n)]
    for r in range(n):
        np.add.at(H[r], rng.integers(0, 4 ** k, per_row), 1)
    return H


FLAGS5 = [port.FEAT[x] for x in ("euclidean", "emd", "manhattan", "pearson", "length_difference")]


@pytest.mark.parametrize("case", ["k5_u8", "k6_u16", "k7_u16", "k8_u16", "synth500"])
def test_identity_vs_oracle(built_lib, ctx, case):
    """tile form shapes: one slab, wide rows of uint16 bins <= 255, a synth_hist set; upper and rectangular sweeps over
    ranges that are not multiples of 64 / 256, and a query set other than the database set"""
    capi = built_lib
    cases = {"k5_u8": (5, 1), "k6_u16": (6, 2), "k7_u16": (7, 2), "k8_u16": (8, 2), "synth500": (5, 1)}
    rng = np.random.default_rng(list(cases).index(case))
    k, eb = cases[case]
    if case == "synth500":
        n = 500
        H = synth_hist(rng, n + 90, 5, 1, hi=6).astype(np.int64)
    elif k == 5:
        n = 300
        H = _related(rng, n + 90, 5, 1, 400, 40)
    else:
        n = 150 if k < 8 else 110
        H = _related(rng, n + 90, k, eb, 20000)
    assert H.max() <= 255
    H = H.astype(port.DTYPES[eb])
    ln = rng.integers(900, 1100, len(H)).astype(np.uint64) * (20 if k > 5 else 1)
    mag = H.sum(axis=1, dtype=np.uint64)
    Hq, Hd = H[n:], H[:n]                      # query set (90 rows) != database set
    Q, D = (Hq, mag[n:], ln[n:]), (Hd, mag[:n], ln[:n])
    om = _spread(all_singles_model(FLAGS5, Hd, D[1], D[2], rng, n_combos=4), Hd, D[1], D[2], rng)
    gm = _regression(ctx, capi, om)
    hd = ctx.hset_from_host(Hd, k, mag=D[1], length=D[2])
    hq = ctx.hset_from_host(Hq, k, mag=Q[1], length=Q[2])
    runs = [((0, n), (0, n), True, 0.5), ((3, n - 7), (0, n), False, 0.3), ((5, 70), (60, n - 1), True, 0.7)]
    for qr, dr, upper, t in runs:
        r, ref = _check_vs_oracle(ctx, capi, om, gm, D, D, hd, hd, 0.9, qr, dr, upper, t)
        assert 0 < r["n_out"] < r["n_scored"]
    r, ref = _check_vs_oracle(ctx, capi, om, gm, Q, D, hq, hd, 0.9, (1, 89), (2, n - 3), False, 0.5)
    assert 0 < r["n_out"] < r["n_scored"]


def _big_set(rng, n):
    H = synth_hist(rng, n, 5, 1, hi=6)
    ln = rng.integers(900, 1100, n).astype(np.uint64)
    return H, H.sum(axis=1, dtype=np.uint64), ln


def test_identity_same_bits_as_score_pairs(built_lib, ctx):
    """~3 000 rows (many tiles, several super-rows of the schedule): every survivor's identity is mc2_score_pairs' score
    bit for bit, and exactly the in-window pairs scoring >= t survive"""
    capi = built_lib
    rng = np.random.default_rng(42)
    n = 3000
    H, mag, ln = _big_set(rng, n)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    qs, ds = _window(ln, ln, 0.9, (0, n), (0, n), True)
    sc = ctx.score_pairs(gm, hs, hs, ds, qs, want=("score",))["score"]    # compute(database, query)
    for t in (0.5, 0.9, TINY):
        r = ctx.identity_pairs(gm, hs, hs, t, 0.9, upper_only=True, max_out=len(qs))
        assert r["n_scored"] == len(qs)
        keep = sc >= t
        assert r["n_out"] == int(keep.sum()) and 0 < r["n_out"] < len(qs)
        got = np.stack([r["q"].astype(np.int64), r["d"].astype(np.int64)], axis=1)
        key = lambda a, b: a * n + b
        order = np.argsort(key(got[:, 0], got[:, 1]))
        want_idx = np.flatnonzero(keep)
        want_order = np.argsort(key(qs[want_idx], ds[want_idx]))
        assert np.array_equal(key(got[order, 0], got[order, 1]), key(qs[want_idx], ds[want_idx])[want_order])
        assert np.array_equal(r["identity"][order].view(np.uint64), sc[want_idx][want_order].view(np.uint64))


def _boundary_pairs(ctx, capi, om, H, mag, ln, want=60):
    """pairs whose identity lies strictly inside (0, 1), with that identity"""
    n = len(H)
    qs, ds = _window(ln, ln, 0.9, (0, n), (0, n), True)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    sc = ctx.score_pairs(gm, hs, hs, ds, qs, want=("score",))["score"]
    inside = np.flatnonzero((sc > 0) & (sc < 1))
    pick = inside[np.linspace(0, len(inside) - 1, min(want, len(inside))).astype(np.int64)]
    return gm, hs, qs[pick], ds[pick], sc[pick]


@pytest.mark.parametrize("kind", ["plain", "large_weights", "three_single_combo"])
def test_screen_at_the_boundary(built_lib, ctx, kind):
    """t = a pair's identity keeps it, nextafter(identity, 2) drops it: the fp32 screen never rejects a survivor, also with
    weights up to 10^3 and with a model outside the screen's form (every pair takes the exact path)"""
    capi = built_lib
    rng = np.random.default_rng(7)
    H, mag, ln = _big_set(rng, 400)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    if kind == "large_weights":
        s = _sums(om, H, mag, ln, rng)
        med = float(np.median(s))
        f = 1e3 / max(abs(w) for w in om.weights[1:])
        om.weights = [0.5 - f * med] + [w * f for w in om.weights[1:]]
        assert max(abs(w) for w in om.weights) <= 2e3
    elif kind == "three_single_combo":
        om.combos.append((0, FLAGS5[0] | FLAGS5[1] | FLAGS5[2]))
        om.weights.append(0.25)
    gm, hs, qs, ds, ids = _boundary_pairs(ctx, capi, om, H, mag, ln)
    assert len(qs) >= 50
    for q, d, s in zip(qs, ds, ids):
        for t, n_want in ((s, 1), (np.nextafter(s, 2.0), 0)):
            r = ctx.identity_pairs(gm, hs, hs, float(t), 0.9, q_range=(int(q), int(q) + 1), d_range=(int(d), int(d) + 1), max_out=4)
            assert r["n_scored"] == 1 and r["n_out"] == n_want, (q, d, s, t)
            if n_want:
                assert r["identity"][0] == s


@pytest.mark.parametrize("seed", [0, 1, 2, 3, 4, 5])
def test_random_regression_models(built_lib, ctx, seed):
    """random models over the fast singles (every reduction mix), stale magnitudes on odd seeds"""
    capi = built_lib
    rng = np.random.default_rng(seed)
    n = 260
    H = synth_hist(rng, n, 5, 1, hi=5)
    ln = rng.integers(900, 1100, n).astype(np.uint64)
    mag = H.sum(axis=1, dtype=np.uint64)
    if seed % 2:
        mag = mag.copy()
        mag[::3] += 13
    flags = [int(f) for f in rng.choice(FAST, size=int(rng.integers(1, 6)), replace=False)]
    om = all_singles_model(flags, H, mag, ln, rng, n_combos=int(rng.integers(1, 5)))
    om = _spread(om, H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    S = (H, mag, ln)
    r, _ = _check_vs_oracle(ctx, capi, om, gm, S, S, hs, hs, 0.9, (0, n), (0, n), True, 0.5)
    assert 0 < r["n_out"] < r["n_scored"]


def _legacy(fn):
    os.environ["MC2_SWEEP_LEGACY"] = "1"
    try:
        return fn()
    finally:
        os.environ.pop("MC2_SWEEP_LEGACY", None)


@pytest.mark.parametrize("case", ["u16_big_bin", "u32", "u64", "k4", "jeffrey", "jensen_shannon"])
def test_shapes_outside_the_tile_form(built_lib, ctx, case):
    """the row-streaming kernels serve what the tile form declines"""
    capi = built_lib
    rng = np.random.default_rng(len(case))
    n = 160
    k, eb = {"u16_big_bin": (5, 2), "u32": (5, 4), "u64": (5, 8), "k4": (4, 1)}.get(case, (5, 1))
    H = synth_hist(rng, n, k, 1, hi=6).astype(np.int64)
    if case == "u16_big_bin":
        H[7, 100] = 300
    H = H.astype(port.DTYPES[eb])
    ln = rng.integers(900, 1100, n).astype(np.uint64)
    mag = H.sum(axis=1, dtype=np.uint64)
    flags = FLAGS5[:3]
    if case == "jeffrey":
        flags = [port.FEAT["jefferey_divergence"]] + FLAGS5[:1]
    elif case == "jensen_shannon":
        flags = [port.FEAT["jensen_shannon"]] + FLAGS5[2:3]
    om = all_singles_model(flags, H, mag, ln, rng, n_combos=3)
    om = _spread(om, H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, k, mag=mag, length=ln)
    S = (H, mag, ln)
    r, _ = _check_vs_oracle(ctx, capi, om, gm, S, S, hs, hs, 0.9, (0, n), (0, n), True, 0.5)
    assert 0 < r["n_out"] < r["n_scored"]


def test_tile_and_row_forms_agree(built_lib, ctx):
    """same survivors and identity bits from the tile form and the row-streaming form on a shape both serve"""
    capi = built_lib
    rng = np.random.default_rng(9)
    H, mag, ln = _big_set(rng, 700)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    for upper, t in ((True, 0.5), (False, 0.8)):
        a = ctx.identity_pairs(gm, hs, hs, t, 0.9, upper_only=upper, max_out=700 * 700)
        b = _legacy(lambda: ctx.identity_pairs(gm, hs, hs, t, 0.9, upper_only=upper, max_out=700 * 700))
        ga = {(int(q), int(d)): s for q, d, s in zip(a["q"], a["d"], a["identity"].view(np.uint64))}
        gb = {(int(q), int(d)): s for q, d, s in zip(b["q"], b["d"], b["identity"].view(np.uint64))}
        assert ga == gb and a["n_scored"] == b["n_scored"] and 0 < len(ga) < a["n_scored"]


@pytest.mark.parametrize("legacy", [False, True])
def test_thresholds_and_capacity(built_lib, ctx, legacy):
    capi = built_lib
    rng = np.random.default_rng(13)
    H, mag, ln = _big_set(rng, 300)
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)

    def run(t, max_out=300 * 300):
        f = lambda: ctx.identity_pairs(gm, hs, hs, t, 0.9, upper_only=True, max_out=max_out)
        return _legacy(f) if legacy else f()
    qs, _ = _window(ln, ln, 0.9, (0, 300), (0, 300), True)
    for t in (0.0, -1.0, -np.inf):
        r = run(t)
        assert r["n_out"] == r["n_scored"] == len(qs)
    for t in (np.nextafter(1.0, 2.0), 1.5, np.inf):
        r = run(t)
        assert r["n_out"] == 0 and r["n_scored"] == len(qs)
    full = run(0.5)
    assert 10 < full["n_out"] < len(qs)
    part = run(0.5, max_out=7)
    assert part["n_out"] == full["n_out"] and len(part["q"]) == 7
    allp = {(int(q), int(d)): s for q, d, s in zip(full["q"], full["d"], full["identity"])}
    for q, d, s in zip(part["q"], part["d"], part["identity"]):
        assert allp[(int(q), int(d))] == s


def test_errors(built_lib, ctx, golden):
    capi = built_lib
    H, ln = golden["hist_k5_eb1"][:4], golden["len_k5_eb1"][:4].copy()
    om = port.Model.from_text(weights_text("weights_cfg1_id90"))       # uses length_difference and pearson
    gm = ctx.model(to_desc(capi, om, regression=1))
    hs = ctx.hset_from_host(H, 5, length=ln)
    for model, t in ((ctx.model_from_file(weights_path("weights_cfg1_id90")), 0.5), (gm, float("nan"))):
        with pytest.raises(capi.Mc2Error) as e:
            ctx.identity_pairs(model, hs, hs, t, 0.9)
        assert e.value.status == -1
    ln0 = ln.copy()
    ln0[1] = 0
    hs = ctx.hset_from_host(H, 5, length=ln0)
    with pytest.raises(capi.Mc2Error) as e:                          # Feature::length_difference throws 123
        ctx.identity_pairs(gm, hs, hs, 0.5, 0.9, q_range=(1, 2), d_range=(0, 4))   # row 1's window [0, 0] holds itself
    assert e.value.status == -4
    Hc = H.copy()
    Hc[2, :] = 1                                                     # zero variance -> pearson NaN -> reference throws
    hs = ctx.hset_from_host(Hc, 5, length=np.full(4, 1000, dtype=np.uint64))
    with pytest.raises(capi.Mc2Error) as e:
        ctx.identity_pairs(gm, hs, hs, 0.5, 0.9)
    assert e.value.status == -4


def test_all_pairs_step_identity_equals_context_call(built_lib, ctx):
    """multi-GPU driver at world 1 through GpuEngine == Context.identity_pairs"""
    import torch
    from meshclust2_b200 import dist as mdist
    from meshclust2_b200 import synth
    capi = built_lib
    seqs, _ = synth.make_set(700, 1000, 40, 0.08, seed=5)
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
        res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n, 0.9, upper_only=True, max_out=n * n, identity=(gm, 0.5))
        got = {(int(q), int(d)): s for (q, d), s in zip(res["survivors"].tolist(), res["survivors"].scores().view(np.uint64))}
    finally:
        # the engine page-locks its survivor buffers for its whole life; they must not be freed while still registered
        for slot in eng._surv_slots:
            for b in slot[3]:
                capi.host_unregister(b)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    r = ctx.identity_pairs(gm, hs, hs, 0.5, 0.9, upper_only=True, max_out=n * n)
    want = {(int(q), int(d)): s for q, d, s in zip(r["q"], r["d"], r["identity"].view(np.uint64))}
    assert got == want and res["n_close"] == r["n_out"] and res["n_scored"] == r["n_scored"] and 0 < len(want) < r["n_scored"]
