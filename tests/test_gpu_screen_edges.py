"""GPU: the tile sweep's fp32 rejection screen (build_screen in csrc/mc2_api.cu, screen_pairs and make_rowf in
csrc/tile_sweep.cu) at its exact decision boundary and at the limits of what it admits.

The screen is a proof: a pair it rejects has an exact GLM sum below the threshold.  A hole in it can only show as a
survivor that goes missing at the boundary, so these tests put pairs exactly there and compare every sweep, with no
pair exempted, against
  1. dense mc2_score_pairs over every in-window pair (compute(database, query)), whose close flag and score come from the
     same fp64 epilogue: equal survivors, bit-identical scores;
  2. the row-streaming form (MC2_SWEEP_LEGACY=1), which has no screen: equal survivors and bits;
  3. the oracle on a sample of query rows: scores within 1e-9.
Placing a pair on the boundary: for a classifier, the intercept w0* at which the pair just turns close (bisection over
doubles in their order); for a regression model, an identity search at t = the pair's identity (kept) and
nextafter(t, 2) (dropped)."""
import os

import numpy as np
import pytest

from conftest import weights_text
from helpers import all_singles_model, synth_hist, to_desc
from oracle import port

pytestmark = pytest.mark.gpu

F = port.FEAT
EMD, LD = F["emd"], F["length_difference"]
XY, XY2, X2Y, X2Y2 = 0, 1, 2, 3
SIM = {F[x] for x in ("normalized_vectors", "pearson", "intersection", "kulczynski2", "simratio")}
EPS = 2.0 ** -23
CUTOFF = 0.9
BIASES = (0.0, 0.3, -0.3, 0.4999989, -0.4999989)
MC2_ERR_FEATURE = -4
PLACED = 45


def _legacy(fn):
    os.environ["MC2_SWEEP_LEGACY"] = "1"
    try:
        return fn()
    finally:
        os.environ.pop("MC2_SWEEP_LEGACY", None)


def _window(ln, upper=True):
    """in-window (q, d) pairs of the sweep over one set, q-major (FC_Runner.cpp:435-444: size_t truncation)"""
    n = len(ln)
    qs, ds = [], []
    d = np.arange(n)
    L = ln.astype(np.int64)
    for q in range(n):
        lo, hi = int(float(ln[q]) * CUTOFF), int(float(ln[q]) / CUTOFF)
        ok = (L >= lo) & (L <= hi)
        if upper:
            ok &= d > q
        qs.append(np.full(int(ok.sum()), q))
        ds.append(d[ok])
    return np.concatenate(qs).astype(np.int64), np.concatenate(ds).astype(np.int64)


def _key(x):
    """doubles -> integers in the same order (int64 bit patterns, negatives mirrored)"""
    i = int(np.float64(x).view(np.int64))
    return i if i >= 0 else -(i & 0x7FFFFFFFFFFFFFFF)


def _val(k):
    return float(np.int64(k).view(np.float64)) if k >= 0 else float(np.int64(-k | -0x8000000000000000).view(np.float64))


def _threshold(bias):
    """the classifier's decision on the sum: logistic(sum) >= 0.5 - bias (Predictor.cpp:323-333)"""
    p = 0.5 - bias
    return float(np.log(p / (1.0 - p)))


def _model_of(singles, combos, weights, bias=0.0):
    """an oracle model over (flag, min, max) singles; they are kept in the order the combos look them up (add_feature,
    Feature.cpp:102-127) and only if a combo uses them"""
    norm = {f: (lo, hi) for f, lo, hi in singles}
    look = []
    for _, fl in combos:
        for b in range(64):
            if fl >> b & 1 and (1 << b) not in look:
                look.append(1 << b)
    return port.Model([(f,) + norm[f] for f in look], combos, weights, bias, k=5, ident=0.9, datatype="uint8_t")


def _with(om, w0=None, bias=None):
    return port.Model(om.singles, om.combos, [om.weights[0] if w0 is None else w0] + om.weights[1:],
                      om.bias if bias is None else bias, k=5, ident=0.9, datatype="uint8_t")


def _widen_emd(om, case):
    """the coarse form bounds the EMD inside an interval 32 T wide (T: the smaller row total once the pseudo-count is
    out); an EMD range at least 16 times that keeps the interval within 1/16 in normalised units, so that the screen
    still rejects pairs"""
    H, mag, _ = case.S
    base = 1 if int(H.sum(axis=1).max()) >= 65536 else 0
    width = 512.0 * float(np.median(H.sum(axis=1, dtype=np.int64) - base * H.shape[1]))
    om.singles = [(f, lo, max(hi, lo + width)) if f == EMD else (f, lo, hi) for f, lo, hi in om.singles]
    return om


def _moderate_b(om, bmax=50.0):
    """ranges widened where min / range would put the offset b of x = a raw + b beyond bmax (normalized_vectors or
    pearson of rows with sums near 65 536 span a few 1e-4 near 1): such models are outside the screen's form"""
    out = []
    for f, lo, hi in om.singles:
        out.append((f, lo, lo + max(hi - lo, abs(lo) / (bmax - 1))))
    om.singles = out
    return om


def _power(kind, nidx):
    return {XY: nidx, X2Y2: 2 * nidx, XY2: 3, X2Y: 3}[kind]


def _combo_values(om, cache):
    """the combos of om over the oracle's normalised singles (pairs x singles) -> pairs x combos"""
    out = []
    for (kind, _), ix in zip(om.combos, om.combo_indices()):
        x = cache[:, ix]
        if kind == XY:
            v = np.prod(x, axis=1)
        elif kind == X2Y2:
            v = np.prod(x * x, axis=1)
        elif kind == XY2:
            v = x[:, 0] * x[:, 1] * x[:, 1]
        else:
            v = x[:, 0] * x[:, 0] * x[:, 1]
        out.append(v)
    return np.stack(out, axis=1)


def _rest(om, S, ds, qs):
    """the oracle's GLM sum without the intercept, and u = 1 + max |x| over the singles, of pairs (database ds, query qs)"""
    H, mag, ln = S
    cache = port.score_pairs(om, H, mag, ln, ds, qs, want_cache=True)["cache"]
    return _combo_values(om, cache) @ np.array(om.weights[1:]), 1 + np.abs(cache).max(axis=1)


def _k1(om):
    """build_screen's K1 (|fp32 sum - exact| <= eps (K1 u^4 + K0)) for the model's singles and combos"""
    beta = 0.0
    for f, lo, hi in om.singles:
        r = hi - lo
        beta = max(beta, abs(-lo / r if f in SIM else 1 + lo / r))
    gamma = 18 * max(1.0, 2 * beta)
    nc = len(om.combos)
    return sum(abs(w) * (1.01 * _power(kind, len(ix)) * gamma + _power(kind, len(ix)) + 2 + nc + 1)
               for w, (kind, _), ix in zip(om.weights[1:], om.combos, om.combo_indices()))


def _scale_to_bound(om, u, e):
    """combo weights scaled so that the screen's bound 2 eps K1 u^4 is e at u"""
    f = e / (2 * EPS * _k1(om) * u ** 4)
    om.weights = [om.weights[0]] + [w * f for w in om.weights[1:]]
    return om


def _model(ctx, capi, om, regression):
    return ctx.model(to_desc(capi, om, regression=int(regression)))


def _sweep(ctx, gm, hs, t, **kw):
    if t is None:
        r = ctx.all_pairs(gm, hs, hs, CUTOFF, **kw)
    else:
        r = ctx.identity_pairs(gm, hs, hs, t, CUTOFF, **kw)
        r["score"] = r["identity"]
    return r


def _bits(r):
    return {(int(q), int(d)): int(s) for q, d, s in zip(r["q"], r["d"], r["score"].view(np.uint64))}


class Case:
    """one set (rows, side-band, hset, in-window pairs) and the checks against the three references"""

    def __init__(self, ctx, capi, H, mag, ln):
        self.ctx, self.capi = ctx, capi
        self.S = (H, mag, ln)
        self.n = len(H)
        self.hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
        self.qs, self.ds = _window(ln)

    def dense(self, gm, t):
        """reference 1: {(q, d): score bits} of the survivors among every in-window pair"""
        r = self.ctx.score_pairs(gm, self.hs, self.hs, self.ds, self.qs, want=("score", "close"))
        keep = r["close"] != 0 if t is None else r["score"] >= t
        return {(int(q), int(d)): int(s) for q, d, s in zip(self.qs[keep], self.ds[keep], r["score"][keep].view(np.uint64))}, r["score"]

    def check(self, gm, t=None, coarse=None, screened=True, om=None, oracle_rows=0):
        """the whole-set sweep == reference 1 == reference 2 (and the oracle on oracle_rows query rows); coarse / screened:
        the form the sweep must take and whether the screen must reject pairs (n_exact < n_scored)"""
        m = len(self.qs)
        a = _sweep(self.ctx, gm, self.hs, t, upper_only=True, max_out=max(1, m))
        st = self.ctx.last_sweep()
        want, sc = self.dense(gm, t)
        assert a["n_scored"] == m and a["n_out"] == len(want)
        assert _bits(a) == want
        b = _legacy(lambda: _sweep(self.ctx, gm, self.hs, t, upper_only=True, max_out=max(1, m)))
        assert b["n_scored"] == m and _bits(b) == want
        if coarse is not None:
            assert st["coarse"] == coarse, st
        if screened:
            assert st["n_exact"] < a["n_scored"], st
        if om is not None and oracle_rows:
            self.oracle(om, sc, t, oracle_rows)
        return a, st

    def oracle(self, om, sc, t, rows):
        """reference 3: the oracle's scores (classifier) or identities (regression) of every in-window pair of a few query
        rows against the dense scores, within 1e-9"""
        H, mag, ln = self.S
        sel = np.isin(self.qs, np.linspace(0, self.n - 2, rows).astype(np.int64))
        qs, ds = self.qs[sel], self.ds[sel]
        if t is None:
            want = port.score_pairs(om, H, mag, ln, ds, qs, want_cache=False)["score"]
        else:
            want = np.array([port.predict_pair(om, H[d], H[q], int(mag[d]), int(mag[q]), int(ln[d]), int(ln[q]))
                             for q, d in zip(qs, ds)])
        assert np.abs(sc[sel] - want).max() <= 1e-9

    def pair_score(self, gm, q, d):
        return self.ctx.score_pairs(gm, self.hs, self.hs, [d], [q], want=("score", "close"))

    def one_pair(self, gm, q, d, t=None):
        r = _sweep(self.ctx, gm, self.hs, t, q_range=(q, q + 1), d_range=(d, d + 1), max_out=4)
        assert r["n_scored"] == 1
        return r


def _place_classifier(case, om, q, d, rest, bias):
    """w0* = the smallest double intercept at which pair (q, d) is close under om with this bias"""
    ctx, capi = case.ctx, case.capi

    def close(w0):
        return bool(case.pair_score(_model(ctx, capi, _with(om, w0, bias), False), q, d)["close"][0])
    g = _threshold(bias) - rest
    span = 1e-9 * (1 + abs(g) + abs(rest))
    lo, hi = g - span, g + span
    for _ in range(40):
        if not close(lo):
            break
        lo -= span
        span *= 4
    for _ in range(40):
        if close(hi):
            break
        hi += span
        span *= 4
    assert not close(lo) and close(hi)
    klo, khi = _key(lo), _key(hi)
    while khi - klo > 1:
        mid = (klo + khi) // 2
        if close(_val(mid)):
            khi = mid
        else:
            klo = mid
    return _val(khi)


def _pick(rest, count, lo=0.02, hi=0.98):
    """indices of count pairs spread over the range of rest (between its lo and hi quantiles)"""
    order = np.argsort(rest, kind="stable")
    n = len(order)
    return order[np.linspace(int(lo * n), int(hi * (n - 1)), count).astype(np.int64)]


def _place_all(case, om, count=PLACED, coarse=None, pairs=None, per_pair_model=None, oracle_every=9):
    """place count pairs (spread over the sums' range) on the boundary, alternately as classifier (cycling the biases)
    and regression pairs; for each: the one-pair sweep keeps it at the boundary and drops it at the neighbour, and the
    whole-set sweep with that model equals the references.  per_pair_model(i) -> a model for pair i (else om)."""
    ctx, capi = case.ctx, case.capi
    if pairs is None:
        sub = np.random.default_rng(0).choice(len(case.qs), size=min(3000, len(case.qs)), replace=False)
        rest, _ = _rest(om, case.S, case.ds[sub], case.qs[sub])
        pairs = sub[_pick(rest, count)]
    n_screened = 0
    for i, j in enumerate(pairs):
        q, d = int(case.qs[j]), int(case.ds[j])
        m = per_pair_model(i, q, d) if per_pair_model else om
        rest = float(_rest(m, case.S, np.array([d]), np.array([q]))[0][0])
        check_oracle = oracle_every and i % oracle_every == 0
        if i % 3 == 2:
            # regression: an intercept that puts the identity inside (0, 1), then t = that identity
            target = 0.05 + 0.9 * ((i * 0.37) % 1.0)
            mr = _with(m, target - rest, 0.0)
            gm = _model(ctx, capi, mr, True)
            s = float(case.pair_score(gm, q, d)["score"][0])
            assert 0 < s < 1, (q, d, s)
            r = case.one_pair(gm, q, d, s)
            assert r["n_out"] == 1 and r["score"][0] == s, (q, d, s)
            assert case.one_pair(gm, q, d, float(np.nextafter(s, 2.0)))["n_out"] == 0, (q, d, s)
            _, st = case.check(gm, s, coarse, screened=False, om=mr if check_oracle else None, oracle_rows=6)
        else:
            bias = BIASES[i % len(BIASES)]
            w0 = _place_classifier(case, m, q, d, rest, bias)
            at, below = _with(m, w0, bias), _with(m, float(np.nextafter(w0, -np.inf)), bias)
            gm = _model(ctx, capi, at, False)
            s = case.pair_score(gm, q, d)["score"][0]
            r = case.one_pair(gm, q, d)
            assert r["n_out"] == 1 and r["score"].view(np.uint64)[0] == np.float64(s).view(np.uint64), (q, d, w0, bias)
            assert case.one_pair(_model(ctx, capi, below, False), q, d)["n_out"] == 0, (q, d, w0, bias)
            _, st = case.check(gm, None, coarse, screened=False, om=at if check_oracle else None, oracle_rows=6)
        n_screened += st["n_exact"] < len(case.qs)
    return n_screened


# ---------------------------------------------------------------------------------------------------------------------
# rows and models of the regimes
# ---------------------------------------------------------------------------------------------------------------------
def _rows(rng, dtype, n=192):
    """uint8 rows (bins 1..6, near-duplicates), or uint16 rows of one slab whose sums lie just above 65 536 (the
    pseudo-count is taken out of the cumulative rows)"""
    if dtype == "u8":
        # k-mer counts of about 1 kb sequences: eight templates, each row one of them with a tenth of its bins moved by 1
        base = rng.poisson(1.0, (8, 1024))
        H = base[rng.integers(0, 8, n)] + rng.integers(-1, 2, (n, 1024)) * (rng.random((n, 1024)) < 0.1)
        H = np.clip(H, 0, 255).astype(np.uint8)
        H[H.sum(axis=1) == 0, 0] = 1
    else:
        H = (64 + (rng.random((n, 1024)) < 0.5)).astype(np.uint16)
        H[: n // 2] = H[rng.integers(0, 8, n // 2)]
        H[: n // 2] += (rng.random((n // 2, 1024)) < 0.03).astype(np.uint16)
        assert (H.sum(axis=1) > 65536).all() and (H.sum(axis=1) < 65536 + 1024).all()
    ln = rng.integers(900, 1100, n).astype(np.uint64)
    return H, H.sum(axis=1, dtype=np.uint64), ln


FULL_FLAGS = [F[x] for x in ("euclidean", "manhattan", "pearson", "normalized_vectors", "intersection", "kulczynski2",
                             "simratio", "length_difference")]


# singles that still vary between rows of 64 / 65 counts (normalized_vectors, pearson, intersection, kulczynski2 and
# simratio stay within 1e-3 of 1 there)
U16_FLAGS = [F["euclidean"], F["manhattan"]]


def _flags(rng, coarse, dtype, k=4):
    """EMD for the coarse form, length_difference (the lengths spread the sums whatever the rows), and random others"""
    pool = [f for f in (FULL_FLAGS if dtype == "u8" else U16_FLAGS) if f != LD]
    f = [int(x) for x in rng.choice(pool, size=min(len(pool), k - 1 - int(coarse)), replace=False)]
    return ([EMD] if coarse else []) + [LD] + f


def _typical_u(om, case):
    sub = np.random.default_rng(1).choice(len(case.qs), size=min(800, len(case.qs)), replace=False)
    return float(np.median(_rest(om, case.S, case.ds[sub], case.qs[sub])[1]))


def _regime_model(regime, coarse, dtype, case, rng):
    H, mag, ln = case.S
    if regime == "trained":
        om = port.Model.from_text(weights_text("weights_cfg1_id90"))
        if not coarse:
            # the full form: the trained model's combos without EMD
            keep = [i for i, (_, fl) in enumerate(om.combos) if not fl & EMD]
            om = _model_of(om.singles, [om.combos[i] for i in keep], [om.weights[0]] + [om.weights[i + 1] for i in keep])
        return om
    if regime == "squared":
        # X2Y2 with two singles, XY2, X2Y, a single squared; both weight signs
        fl = _flags(rng, coarse, dtype, 3)
        a, b, c = fl
        om = all_singles_model(fl, H, mag, ln, rng, n_combos=1)
        om = _model_of(om.singles, [(X2Y2, a | b), (XY2, a | c), (X2Y, b | c), (X2Y2, a), (X2Y2, c)],
                       [0.0, 1.5, -2.0, 1.0, -1.2, 0.8])
        return _widen_emd(_moderate_b(om), case)
    om = _widen_emd(_moderate_b(all_singles_model(_flags(rng, coarse, dtype), H, mag, ln, rng, n_combos=4)), case)
    if regime == "large_weights":
        # weights as large as the screen still works with: its bound e reaches about 0.6 at a typical pair, 1 (no
        # rejection) at the wider ones
        return _scale_to_bound(om, _typical_u(om, case), 0.6)
    if regime == "wide_norm":
        # ranges narrowed so normalised values reach about +-20, |b| kept below the gamma limit (582.5): the u^4 term
        # dominates the bound; weights scaled so that it stays usable
        singles = []
        for f, lo, hi in om.singles:
            mid, r = (lo + hi) / 2, max((hi - lo) / 40, 1e-6)
            r = max(r, abs(mid) / 570)
            singles.append((f, mid - r if f in SIM else mid + r, (mid - r if f in SIM else mid + r) + r))
        om.singles = singles
        return _scale_to_bound(om, _typical_u(om, case), 0.3)
    return om


# ---------------------------------------------------------------------------------------------------------------------
# 1 + 2: pairs on the boundary, per regime and tile form
# ---------------------------------------------------------------------------------------------------------------------
REGIMES = ["trained", "random", "large_weights", "wide_norm", "squared"]
# the trained model's EMD range (about 2.8e5) is far narrower than the coarse interval of rows summing to 65 536 (about
# 2.1e6), so the coarse form could not reject a pair there: it runs on uint8 rows only
BOUNDARY_CASES = [(r, f, d) for r in REGIMES for f in ("full", "coarse") for d in ("u8", "u16")
                  if (r, f, d) != ("trained", "coarse", "u16")]


@pytest.mark.parametrize("regime,form,dtype", BOUNDARY_CASES)
def test_pairs_on_the_boundary(built_lib, ctx, regime, form, dtype):
    """45 pairs per regime on the exact decision boundary (classifier with bias 0, +-0.3, +-0.4999989, and regression):
    kept there, dropped one double below; every whole-set sweep equals the references"""
    rng = np.random.default_rng(BOUNDARY_CASES.index((regime, form, dtype)))
    coarse = form == "coarse"
    case = Case(ctx, built_lib, *_rows(rng, dtype))
    om = _regime_model(regime, coarse, dtype, case, rng)
    assert any(f == EMD for f, _, _ in om.singles) == coarse
    # the screen runs and rejects pairs: a classifier that keeps the top 5 % of the sums
    sub = rng.choice(len(case.qs), size=1000, replace=False)
    top = float(np.quantile(_rest(om, case.S, case.ds[sub], case.qs[sub])[0], 0.95))
    cm = _with(om, -top, 0.0)
    case.check(_model(ctx, built_lib, cm, False), None, coarse, screened=True, om=cm, oracle_rows=8)
    n_screened = _place_all(case, om, coarse=coarse)
    assert n_screened >= PLACED // 3


def test_emd_squared_spanning_zero(built_lib, ctx):
    """coarse form, EMD^2 and EMD^2 x with negative weights: the normalised EMD x = 1 - (emd - min) / range is set to
    vanish at each placed pair's exact EMD (max = that EMD), so x changes sign inside the pair's coarse interval and
    only the spans-0 rule keeps the screen's upper bound above the exact sum"""
    capi = built_lib
    rng = np.random.default_rng(5)
    for dtype in ("u8", "u16"):
        case = Case(ctx, capi, *_rows(rng, dtype))
        H, mag, ln = case.S
        base = _widen_emd(all_singles_model([EMD, F["euclidean"], F["pearson"]], H, mag, ln, rng, n_combos=1), case)
        width = next(hi - lo for f, lo, hi in base.singles if f == EMD)
        eu, pe = F["euclidean"], F["pearson"]
        variants = [
            ([(X2Y2, EMD), (XY, eu)], [0.0, -3.0, 1.5]),
            ([(XY2 if EMD > eu else X2Y, EMD | eu), (XY, pe)], [0.0, -2.5, 1.0]),
            ([(XY2 if EMD > pe else X2Y, EMD | pe), (X2Y2, EMD), (XY, eu)], [0.0, -1.5, -1.0, 1.0]),
        ]
        sub = rng.choice(len(case.qs), size=1500, replace=False)
        emd = np.array([port.raw_single(EMD, H[d], H[q], int(mag[d]), int(mag[q])) for q, d in zip(case.qs[sub], case.ds[sub])])
        pairs = sub[_pick(emd, PLACED)]

        def model_for(i, q, d):
            combos, w = variants[i % len(variants)]
            e = port.raw_single(EMD, H[d], H[q], int(mag[d]), int(mag[q]))
            return _model_of([(EMD, e - width, e)] + [s for s in base.singles if s[0] != EMD], combos, w)

        n_screened = _place_all(case, None, coarse=True, pairs=pairs, per_pair_model=model_for)
        assert n_screened >= PLACED // 3


# ---------------------------------------------------------------------------------------------------------------------
# 3: rows the screen must not touch (make_rowf's `big`)
# ---------------------------------------------------------------------------------------------------------------------
def _touching(case, rows):
    big = np.zeros(case.n, dtype=bool)
    big[rows] = True
    return int((big[case.qs] | big[case.ds]).sum())


@pytest.mark.parametrize("form", ["full", "coarse"])
def test_lengths_around_2_24(built_lib, ctx, form):
    """lengths 2^24 - 3 .. 2^24 + 3 (differences 0-6) with length_difference normalised over [0, 8]: from 2^24 on, float
    lengths are no longer exact (2^24 + 1 and 2^24 + 2 differ by 1, their floats by 2), so those rows must take the
    exact path; pairs placed on the boundary where the float difference is the larger one"""
    capi = built_lib
    coarse = form == "coarse"
    rng = np.random.default_rng(11 + coarse)
    H, mag, _ = _rows(rng, "u8")
    # three quarters of the rows below 2^24, in length order: a warp whose rows all stay below it screens its pairs
    ln = np.sort((1 << 24) + rng.choice([-3, -2, -1, 0, 1, 2, 3], len(H), p=[.25, .25, .25, .07, .06, .06, .06])).astype(np.uint64)
    case = Case(ctx, capi, H, mag, ln)
    flags = ([EMD] if coarse else []) + [F["euclidean"], LD]
    om = all_singles_model(flags, H, mag, ln, rng, n_combos=1)
    eu = F["euclidean"]
    combos = [(XY, LD), (XY, eu)] + ([(XY, EMD)] if coarse else [])
    om = _model_of([(f, 0.0, 8.0) if f == LD else (f, lo, hi) for f, lo, hi in _widen_emd(om, case).singles], combos,
                   [0.0, 2.0, -1.0] + ([-0.7] if coarse else []))
    big = np.flatnonzero(ln >= (1 << 24))
    lf = ln.astype(np.float32).astype(np.float64)
    exact = np.abs(ln[case.qs].astype(np.int64) - ln[case.ds].astype(np.int64))
    fl = np.abs(lf[case.qs] - lf[case.ds])
    worse = np.flatnonzero(fl > exact)     # float rounding would lower x = 1 - ld / 8, and the weight on it is positive
    assert len(worse) > 100
    rest, _ = _rest(om, case.S, case.ds[worse], case.qs[worse])
    _place_all(case, om, coarse=coarse, pairs=worse[_pick(rest, 40, 0.0, 1.0)])
    rest, _ = _rest(om, case.S, case.ds, case.qs)
    cm = _with(om, -float(np.quantile(rest, 0.95)), 0.0)
    _, st = case.check(_model(ctx, capi, cm, False), None, coarse, screened=True, om=cm, oracle_rows=6)
    assert st["n_exact"] >= _touching(case, big)


@pytest.mark.parametrize("form", ["full", "coarse"])
def test_stale_magnitudes(built_lib, ctx, form):
    """pseudo-magnitudes 2^26 - 1 (still screened), 2^26 and 2^40 (exact path) on rows whose bins sum to far less"""
    capi = built_lib
    coarse = form == "coarse"
    rng = np.random.default_rng(21 + coarse)
    H, mag, ln = _rows(rng, "u8")
    mag = mag.copy()
    edge = np.arange(0, len(H), 6)
    mag[edge] = (1 << 26) - 1
    mag[3::12] = 1 << 26
    mag[5::12] = 1 << 40
    case = Case(ctx, capi, H, mag, ln)
    flags = ([EMD] if coarse else []) + [F[x] for x in ("intersection", "kulczynski2", "pearson", "euclidean")]
    om = _widen_emd(all_singles_model(flags, H, mag, ln, rng, n_combos=4), case)
    big = np.flatnonzero(mag >= (1 << 26))
    # boundary pairs among those that touch a 2^26 - 1 row but no big one
    touch = np.isin(case.qs, edge) | np.isin(case.ds, edge)
    clean = ~(np.isin(case.qs, big) | np.isin(case.ds, big))
    cand = np.flatnonzero(touch & clean)
    rest, _ = _rest(om, case.S, case.ds[cand], case.qs[cand])
    _place_all(case, om, coarse=coarse, pairs=cand[_pick(rest, 30)])
    _place_all(case, om, count=15, coarse=coarse)
    cm = _with(om, -float(np.median(rest)), 0.0)
    _, st = case.check(_model(ctx, capi, cm, False), None, coarse, screened=True, om=cm, oracle_rows=6)
    assert st["n_exact"] >= _touching(case, big)


@pytest.mark.parametrize("form", ["full", "coarse"])
@pytest.mark.parametrize("which", ["len0", "mag0"])
def test_zero_length_and_magnitude(built_lib, ctx, form, which):
    """len = 0 or mag = 0 rows: the sweep reports what mc2_score_pairs and the oracle report (MC2_ERR_FEATURE where the
    reference throws), and otherwise the same survivors and bits"""
    capi = built_lib
    coarse = form == "coarse"
    rng = np.random.default_rng(31 + coarse + 2 * (which == "mag0"))
    H, mag, ln = _rows(rng, "u8", n=96)
    flags = ([EMD] if coarse else []) + [F[x] for x in ("intersection", "kulczynski2", "euclidean", "length_difference")]
    om = all_singles_model(flags, H, mag, ln, rng, n_combos=4)
    mag, ln = mag.copy(), ln.copy()
    if which == "len0":
        zero = [4, 9, 40]           # in one another's window [0, 0]: length_difference throws
        ln[zero] = 0
    else:
        zero = [4, 40]              # out of each other's window; kulczynski2 against them is infinite, not NaN
        mag[zero] = 0
        ln[zero] = (920, 1080)
    case = Case(ctx, capi, H, mag, ln)
    gm = _model(ctx, capi, om, False)

    def status(fn):
        try:
            fn()
            return 0
        except capi.Mc2Error as e:
            return e.status
    m = max(1, len(case.qs))
    got = status(lambda: ctx.all_pairs(gm, case.hs, case.hs, CUTOFF, upper_only=True, max_out=m))
    ref = status(lambda: ctx.score_pairs(gm, case.hs, case.hs, case.ds, case.qs, want=("score", "close")))
    leg = status(lambda: _legacy(lambda: ctx.all_pairs(gm, case.hs, case.hs, CUTOFF, upper_only=True, max_out=m)))
    try:
        port.score_pairs(om, H, mag, ln, case.ds, case.qs, want_cache=False)
        orc = 0
    except ValueError:
        orc = MC2_ERR_FEATURE
    assert got == ref == leg == orc, (got, ref, leg, orc)
    if which == "len0":
        assert got == MC2_ERR_FEATURE
    else:
        assert got == 0
        _, st = case.check(gm, None, coarse, screened=False)
        assert st["n_exact"] >= _touching(case, zero)


def test_every_row_big(built_lib, ctx):
    """a few thousand rows, every one of length >= 2^24, in the coarse form: every in-window pair goes through the
    exact-EMD flush of the epilogue"""
    capi = built_lib
    rng = np.random.default_rng(41)
    n = 2500
    H = synth_hist(rng, n, 5, 1, hi=6)
    mag = H.sum(axis=1, dtype=np.uint64)
    ln = rng.integers(1 << 24, 1 << 25, n).astype(np.uint64)
    case = Case(ctx, capi, H, mag, ln)
    flags = [EMD, F["euclidean"], F["pearson"], F["manhattan"]]
    om = _widen_emd(all_singles_model(flags, H, mag, ln, rng, n_combos=4), case)
    sub = rng.choice(len(case.qs), size=1500, replace=False)
    rest, _ = _rest(om, case.S, case.ds[sub], case.qs[sub])
    cm = _with(om, -float(np.quantile(rest, 0.9)), 0.0)
    a, st = case.check(_model(ctx, capi, cm, False), None, True, screened=False, om=cm, oracle_rows=4)
    assert st["n_exact"] == a["n_scored"] == len(case.qs) and 0 < a["n_out"] < a["n_scored"]


# ---------------------------------------------------------------------------------------------------------------------
# 4: what build_screen admits
# ---------------------------------------------------------------------------------------------------------------------
def _desc_of(capi, om, singles=None, combos=None, weights=None, bias=None):
    """a model description straight from lists (for models the oracle's flag notation cannot state)"""
    s = singles if singles is not None else om.singles
    c = combos if combos is not None else [(kind, ix) for (kind, _), ix in zip(om.combos, om.combo_indices())]
    w = weights if weights is not None else om.weights
    return capi.make_desc(s, c, w, om.bias if bias is None else bias, 0)


LIMITS = ["w", "w0", "gamma", "bias", "bias_neg", "combos", "three_singles", "power3", "repeated_single", "jeffrey",
          "jensen_shannon"]


@pytest.mark.parametrize("limit", LIMITS)
def test_admission_limits(built_lib, ctx, limit):
    """a model just inside and just outside each limit of build_screen: the same survivors and bits as the references
    on both sides; inside, the screen runs (coarse form); outside it does not (every pair exact, or the row-streaming
    form for a model the tile sweep does not serve)"""
    capi = built_lib
    rng = np.random.default_rng(LIMITS.index(limit))
    H = synth_hist(rng, 160, 5, 1, hi=6)        # no empty bin: the log singles have a value on every pair
    case = Case(ctx, capi, H, H.sum(axis=1, dtype=np.uint64), rng.integers(900, 1100, 160).astype(np.uint64))
    H, mag, ln = case.S
    eu, pe, ma = F["euclidean"], F["pearson"], F["manhattan"]
    om = _widen_emd(all_singles_model([EMD, eu, pe, ma], H, mag, ln, rng, n_combos=1), case)
    om = _model_of(om.singles, [(XY, EMD | eu), (XY2, eu | pe), (XY, ma)], [0.0, 1.0, -1.5, 0.8])
    sub = rng.choice(len(case.qs), size=1000, replace=False)
    rest, _ = _rest(om, case.S, case.ds[sub], case.qs[sub])
    om.weights[0] = -float(np.median(rest))
    idx = {f: i for i, (f, _, _) in enumerate(om.singles)}
    ci = [(kind, ix) for (kind, _), ix in zip(om.combos, om.combo_indices())]
    row_form = False
    if limit == "w":
        inside = _desc_of(capi, om, weights=[om.weights[0], 999999.9] + om.weights[2:])
        outside = _desc_of(capi, om, weights=[om.weights[0], 1e6] + om.weights[2:])
    elif limit == "w0":
        inside = _desc_of(capi, om, weights=[-999999.9] + om.weights[1:])
        outside = _desc_of(capi, om, weights=[-1e6] + om.weights[1:])
    elif limit == "gamma":
        # euclidean is distance-like: x = 1 - (raw - min) / range, b = 1 + min / range; gamma = 18 max(1, 2 max|b|) and
        # 4 eps gamma < 0.01 bound |b| below 582.54
        lo, hi = next((a, b) for f, a, b in om.singles if f == eu)
        r = hi - lo

        def at(b):
            return _desc_of(capi, om, singles=[(f, (b - 1) * r, (b - 1) * r + r) if f == eu else (f, a, c)
                                               for f, a, c in om.singles])
        inside, outside = at(582.0), at(583.0)
    elif limit in ("bias", "bias_neg"):
        sg = 1 if limit == "bias" else -1
        inside, outside = _desc_of(capi, om, bias=sg * 0.4999989), _desc_of(capi, om, bias=sg * 0.499999)
    elif limit == "combos":
        extra = [(XY, [idx[eu]]), (XY, [idx[pe]]), (X2Y2, [idx[ma]]), (XY, [idx[EMD], idx[pe]]), (X2Y, [idx[pe], idx[ma]]),
                 (XY, [idx[EMD]])]
        w = [0.3, -0.2, 0.1, 0.25, -0.15, 0.05]
        inside = _desc_of(capi, om, combos=ci + extra[:5], weights=om.weights + w[:5])
        outside = _desc_of(capi, om, combos=ci + extra, weights=om.weights + w)
    elif limit == "three_singles":
        inside = _desc_of(capi, om)
        outside = _desc_of(capi, om, combos=ci + [(XY, [idx[EMD], idx[eu], idx[pe]])], weights=om.weights + [0.2])
    elif limit == "power3":
        inside = _desc_of(capi, om, combos=ci + [(X2Y2, [idx[pe]])], weights=om.weights + [0.2])
        outside = _desc_of(capi, om, combos=ci + [(XY2, [idx[pe], idx[pe]])], weights=om.weights + [0.2])
    elif limit == "repeated_single":
        # the same single twice (fast_epi = 0): the tile sweep does not serve it
        row_form = True
        inside = _desc_of(capi, om)
        outside = _desc_of(capi, om, singles=om.singles + [next(s for s in om.singles if s[0] == ma)],
                           combos=ci + [(XY, [len(om.singles)])], weights=om.weights + [0.2])
    else:
        # a log single: the row-streaming kernels serve the model
        row_form = True
        f = F["jefferey_divergence" if limit == "jeffrey" else "jensen_shannon"]
        vals = [port.raw_single(f, H[d], H[q], int(mag[d]), int(mag[q])) for q, d in zip(case.qs[:64], case.ds[:64])]
        inside = _desc_of(capi, om)
        outside = _desc_of(capi, om, singles=om.singles + [(f, min(vals), max(vals))],
                           combos=ci + [(XY, [len(om.singles)])], weights=om.weights + [0.4])
    if limit == "combos":
        assert inside.n_combos == 8 and outside.n_combos == 9
    gi, go = ctx.model(inside), ctx.model(outside)
    case.check(gi, None, True, screened=False)
    a, st = case.check(go, None, False, screened=False)
    if row_form:
        assert st["n_exact"] == 0
    else:
        assert st["n_exact"] == a["n_scored"]
