"""GPU: the coarse form of the tile sweep (csrc/tile_sweep.cu, COARSE): the fp32 screen bounds the EMD by an interval from
64 sampled cumulative bins per row, and the pairs it keeps get the exact EMD from the full cumulative rows.  Survivors
and score bits must be those of the row-streaming form (MC2_SWEEP_LEGACY=1) and of the oracle, for the bench's shapes,
random models over EMD, adversarial rows and identity searches."""
import os

import numpy as np
import pytest

from conftest import weights_path, weights_text
from helpers import all_singles_model, synth_hist, to_desc
from oracle import port

pytestmark = pytest.mark.gpu

EMD = port.FEAT["emd"]
XY, XY2, X2Y, X2Y2 = 0, 1, 2, 3


def _legacy(fn):
    os.environ["MC2_SWEEP_LEGACY"] = "1"
    try:
        return fn()
    finally:
        os.environ.pop("MC2_SWEEP_LEGACY", None)


def _bits(r, key="score"):
    return {(int(q), int(d)): int(s) for q, d, s in zip(r["q"], r["d"], r[key].view(np.uint64))}


def _oracle_close(om, H, mag, ln, cutoff, q_range, d_range, upper):
    """the reference's work() loop through the oracle: {(q, d): score} of the close pairs, #scored"""
    out, scored = {}, 0
    for q in range(*q_range):
        lo, hi = int(float(ln[q]) * cutoff), int(float(ln[q]) / cutoff)
        cand = [d for d in range(*d_range) if lo <= int(ln[d]) <= hi and (not upper or d > q)]
        if not cand:
            continue
        cand = np.array(cand)
        r = port.score_pairs(om, H, mag, ln, cand, np.full(len(cand), q))
        scored += len(cand)
        for d, s, c in zip(cand, r["score"], r["close"]):
            if c:
                out[(q, int(d))] = s
    return out, scored


def _check_sweep(ctx, gm, hs, n, cutoff=0.9, om=None, H=None, mag=None, ln=None, oracle_rows=None, want_coarse=True):
    """coarse form == row-streaming form bit for bit (and == the oracle on the first oracle_rows query rows)"""
    a = ctx.all_pairs(gm, hs, hs, cutoff, upper_only=True, max_out=n * n)
    st = ctx.last_sweep()
    assert st["coarse"] == want_coarse
    b = _legacy(lambda: ctx.all_pairs(gm, hs, hs, cutoff, upper_only=True, max_out=n * n))
    assert not ctx.last_sweep()["coarse"]
    assert a["n_scored"] == b["n_scored"] and a["n_out"] == b["n_out"]
    assert _bits(a) == _bits(b)
    if om is not None:
        m = oracle_rows or n
        r = ctx.all_pairs(gm, hs, hs, cutoff, q_range=(0, m), upper_only=True, max_out=n * n)
        want, scored = _oracle_close(om, H, mag, ln, cutoff, (0, m), (0, n), True)
        got = {(int(q), int(d)): s for q, d, s in zip(r["q"], r["d"], r["score"])}
        assert r["n_scored"] == scored
        edge = {k for k, s in want.items() if abs(s - 0.5) <= 1e-9}
        assert set(got) - edge == set(want) - edge
        for k in set(got) & set(want):
            assert abs(got[k] - want[k]) <= 1e-9
    return a, st


def _count(ctx, seqs, k, eb):
    from meshclust2_b200 import capi
    enc = capi.encode_batch(seqs)
    sq = ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"])
    hs = ctx.count_kmers(sq, k, eb)
    got = hs.download()
    return hs, got["hist"], got["mag"], got["len"]


@pytest.mark.parametrize("cfg,n", [("cfg3", 1500), ("cfg2", 1200)])
def test_bench_shapes(built_lib, ctx, cfg, n):
    """subsets of the bench's cfg3 / cfg2 sets with the bench model: the coarse form runs, sends only a small share of
    the scored pairs through the exact epilogue (cfg3) and keeps the row-streaming form's survivors and bits"""
    from meshclust2_b200 import synth
    seqs, _, k, eb = synth.make_config_range(cfg, lo=0, hi=n)
    assert (k, eb) == (5, 1)
    hs, H, mag, ln = _count(ctx, seqs, k, eb)
    gm = ctx.model_from_file(weights_path("weights_cfg1_id90"))
    om = port.Model.from_text(weights_text("weights_cfg1_id90"))
    a, st = _check_sweep(ctx, gm, hs, n, om=om, H=H, mag=mag, ln=ln, oracle_rows=150)
    assert a["n_out"] > 0
    if cfg == "cfg3":
        assert st["n_exact"] < 0.01 * a["n_scored"], st


def _emd_model(H, mag, ln, rng, form, sign, other="euclidean"):
    """a model over EMD (and one other single) in the given form; the intercept puts about 5 % of the pairs above the
    classifier's threshold"""
    flags = [EMD, port.FEAT[other]]
    base = all_singles_model(flags, H, mag, ln, rng, n_combos=1)
    rng_of = {f: (lo, hi) for f, lo, hi in base.singles}
    o = port.FEAT[other]
    combos = {"emd": [(XY, EMD)], "emd2": [(X2Y2, EMD)],
              "emd_x": [(XY, EMD | o)], "emd2_x": [(XY2 if EMD > o else X2Y, EMD | o), (XY, o)]}[form]
    look = []
    for _, fl in combos:
        for b in range(64):
            if fl >> b & 1 and (1 << b) not in look:
                look.append(1 << b)
    singles = [(f,) + rng_of[f] for f in look]
    w = [0.0] + [sign * float(abs(x) + 0.5) for x in rng.standard_normal(len(combos))]
    om = port.Model(singles, combos, w, 0.0, k=5, ident=0.9, datatype="uint8_t")
    n = len(H)
    ia, ib = rng.integers(0, n, 600), rng.integers(0, n, 600)
    s = np.clip(port.score_pairs(om, H, mag, ln, ia, ib, want_cache=False)["score"], 1e-15, 1 - 1e-15)
    sums = np.log(s / (1 - s))
    om.weights[0] = -float(np.quantile(sums, 0.95))
    return om


@pytest.mark.parametrize("form", ["emd", "emd2", "emd_x", "emd2_x"])
@pytest.mark.parametrize("sign", [1, -1])
def test_random_emd_models(built_lib, ctx, form, sign):
    """EMD alone, EMD^2, EMD * x, EMD^2 * x with both weight signs: the interval screen never drops a close pair"""
    from meshclust2_b200 import capi
    rng = np.random.default_rng(17 + 5 * sign + len(form))
    n = 400
    H = synth_hist(rng, n, 5, 1, hi=6)
    ln = rng.integers(900, 1100, n).astype(np.uint64)
    mag = H.sum(axis=1, dtype=np.uint64)
    om = _emd_model(H, mag, ln, rng, form, sign)
    gm = ctx.model(to_desc(capi, om))
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    a, _ = _check_sweep(ctx, gm, hs, n, om=om, H=H, mag=mag, ln=ln, oracle_rows=120)
    assert 0 < a["n_out"] < a["n_scored"]


def _adversarial(rng, n):
    """uint8 rows (sums < 65536, base 0): all mass in one 16-bin block, flat rows (every bin = the base 0, and constant
    rows), very different totals, and near-duplicates of a few templates"""
    H = synth_hist(rng, n, 5, 1, hi=8).astype(np.int64)
    for r in range(0, 40):
        H[r] = 0
        b = int(rng.integers(0, 64))
        H[r, 16 * b:16 * b + 16] = rng.integers(0, 256, 16)
    H[40:48] = 0
    H[48:56] = 3
    H[56:60] = 60 - (rng.random((4, H.shape[1])) < 0.5)  # sums about 60 900
    H[60:64] = 0
    H[60:64, 0] = 1      # sum 1
    H[64:72, 1000:] = 255
    H[72:80] = H[0:8]
    H[72:80, 16 * 63:] += 1
    return H.astype(np.uint8)


def test_adversarial_rows(built_lib, ctx):
    """the widest intervals (one heavy 16-bin block), flat rows, totals from 1 to 61 k: bench model and an EMD-only
    model, coarse == row-streaming == oracle"""
    from meshclust2_b200 import capi
    rng = np.random.default_rng(23)
    n = 360
    H = _adversarial(rng, n)
    ln = np.full(n, 1000, dtype=np.uint64)
    mag = H.sum(axis=1, dtype=np.uint64)
    # the bench model's normalized_vectors / pearson have no value on flat rows (the reference throws): its set keeps
    # the other adversarial rows
    Hb = H.copy()
    Hb[40:56] = H[0:16]
    hb = ctx.hset_from_host(Hb, 5, mag=Hb.sum(axis=1, dtype=np.uint64), length=ln)
    gm = ctx.model_from_file(weights_path("weights_cfg1_id90"))
    om = port.Model.from_text(weights_text("weights_cfg1_id90"))
    _check_sweep(ctx, gm, hb, n, om=om, H=Hb, mag=Hb.sum(axis=1, dtype=np.uint64), ln=ln, oracle_rows=100)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    for form, sign in (("emd", 1), ("emd2", -1), ("emd2_x", 1)):
        om = _emd_model(H, mag, ln, rng, form, sign, other="manhattan")
        gm = ctx.model(to_desc(capi, om))
        a, _ = _check_sweep(ctx, gm, hs, n, om=om, H=H, mag=mag, ln=ln, oracle_rows=100)
        assert a["n_out"] > 0


@pytest.mark.parametrize("eb", [1, 2])
def test_rows_with_the_pseudo_count_taken_out(built_lib, ctx, eb):
    """row sums just above 65 536 with every bin >= 1: cumulative rows of (bin - 1), samples from cum_wide_kernel (uint8
    rows and the uint16 byte plane)"""
    from meshclust2_b200 import capi
    rng = np.random.default_rng(31 + eb)
    n = 300
    H = (64 + (rng.random((n, 1024)) < 0.5)).astype(port.DTYPES[eb])
    H[: n // 2] = H[rng.integers(0, 8, n // 2)]
    assert (H.sum(axis=1) >= 65536).all() and (H.sum(axis=1) - 1024 < 65536).all()
    ln = rng.integers(950, 1050, n).astype(np.uint64)
    mag = H.sum(axis=1, dtype=np.uint64)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    om = _emd_model(H.astype(np.int64), mag, ln, rng, "emd_x", 1)
    gm = ctx.model(to_desc(capi, om))
    a, _ = _check_sweep(ctx, gm, hs, n)
    assert a["n_out"] > 0


def _regression(ctx, capi, om, H, mag, ln, rng, lo=-0.2, hi=1.2):
    """the model as a regression model whose sums spread over about [lo, hi]"""
    n = len(H)
    ia, ib = rng.integers(0, n, 400), rng.integers(0, n, 400)
    w0 = om.weights[0]
    om.weights[0] = 0.0
    s = np.clip(port.score_pairs(om, H, mag, ln, ia, ib, want_cache=False)["score"], 1e-15, 1 - 1e-15)
    om.weights[0] = w0
    s = np.log(s / (1 - s))
    a, b = np.quantile(s, 0.05), np.quantile(s, 0.95)
    f = (hi - lo) / max(b - a, 1e-6)
    om.weights = [lo - f * a] + [w * f for w in om.weights[1:]]
    return om, ctx.model(to_desc(capi, om, regression=1))


def test_identity_search(built_lib, ctx):
    """identity search at t = 0.5, 0.9, 1.0 takes the coarse form, t <= 0 the full one; the same survivors and identity
    bits as the row-streaming form, and a pair whose identity sits just above the threshold is kept"""
    from meshclust2_b200 import capi
    rng = np.random.default_rng(41)
    n = 500
    H = synth_hist(rng, n, 5, 1, hi=6)
    ln = rng.integers(900, 1100, n).astype(np.uint64)
    mag = H.sum(axis=1, dtype=np.uint64)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    om = all_singles_model([port.FEAT[x] for x in ("euclidean", "emd", "pearson", "length_difference")], H, mag, ln, rng,
                           n_combos=4)
    om, gm = _regression(ctx, capi, om, H, mag, ln, rng)
    probe = ctx.identity_pairs(gm, hs, hs, 1e-300, 0.9, upper_only=True, max_out=n * n)
    ids = probe["identity"]
    inner = ids[(ids > 0.2) & (ids < 0.95)]
    assert len(inner) > 0
    t_edge = float(np.nextafter(inner[0], -np.inf))
    for t, coarse in ((0.5, True), (0.9, True), (1.0, True), (t_edge, True), (0.0, False), (-1.0, False)):
        a = ctx.identity_pairs(gm, hs, hs, t, 0.9, upper_only=True, max_out=n * n)
        assert ctx.last_sweep()["coarse"] == coarse, t
        b = _legacy(lambda: ctx.identity_pairs(gm, hs, hs, t, 0.9, upper_only=True, max_out=n * n))
        assert a["n_scored"] == b["n_scored"] and a["n_out"] == b["n_out"], t
        assert _bits(a, "identity") == _bits(b, "identity"), t
        if t == t_edge:
            assert float(inner[0]) in set(a["identity"].tolist())
