"""GPU: refinement of the coarse tile sweep's candidates (csrc/tile_sweep.cu).  The sweep writes the pairs its screen keeps
to a candidate buffer of 2^23 records and refine_kernel gives them the exact epilogue after the sweep; pairs beyond the
buffer are refined inside the sweep, as before.  Both paths must give the row-streaming form's (MC2_SWEEP_LEGACY=1)
survivors and score bits, keep the max_out contract, and serve the identity, top-K and both-strand searches."""
import os

import numpy as np
import pytest

from conftest import weights_path
from helpers import all_singles_model, synth_hist, to_desc
from oracle import port

pytestmark = pytest.mark.gpu

CAND_CAP = 1 << 23


def _legacy(fn):
    os.environ["MC2_SWEEP_LEGACY"] = "1"
    try:
        return fn()
    finally:
        os.environ.pop("MC2_SWEEP_LEGACY", None)


def _sorted(r, key):
    """(q, d, score bits) sorted by (q, d)"""
    o = np.lexsort((r["d"], r["q"]))
    return r["q"][o], r["d"][o], np.ascontiguousarray(r[key][o]).view(np.uint64)


def _same(a, b, key="score"):
    assert a["n_out"] == b["n_out"] and a["n_scored"] == b["n_scored"]
    for x, y in zip(_sorted(a, key), _sorted(b, key)):
        assert np.array_equal(x, y)


def _cfg3(ctx, n):
    from meshclust2_b200 import capi, synth
    seqs, _, k, eb = synth.make_config_range("cfg3", lo=0, hi=n)
    enc = capi.encode_batch(seqs)
    sq = ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"])
    hs = ctx.count_kmers(sq, k, eb)
    got = hs.download()
    return hs, got["hist"], got["mag"], got["len"]


def _regression(ctx, H, mag, ln, rng, lo=-0.2, hi=1.2):
    """a regression model over EMD and three other singles whose sums spread over about [lo, hi]"""
    from meshclust2_b200 import capi
    om = all_singles_model([port.FEAT[x] for x in ("euclidean", "emd", "pearson", "length_difference")], H, mag, ln, rng,
                           n_combos=4)
    n = len(H)
    ia, ib = rng.integers(0, n, 400), rng.integers(0, n, 400)
    om.weights[0] = 0.0
    s = np.clip(port.score_pairs(om, H, mag, ln, ia, ib, want_cache=False)["score"], 1e-15, 1 - 1e-15)
    s = np.log(s / (1 - s))
    a, b = np.quantile(s, 0.05), np.quantile(s, 0.95)
    f = (hi - lo) / max(b - a, 1e-6)
    om.weights = [lo - f * a] + [w * f for w in om.weights[1:]]
    return ctx.model(to_desc(capi, om, regression=1))


def test_buffer_only(built_lib, ctx):
    """a cfg3 subset with the bench model: every candidate goes through the buffer, none inline, and the survivors and
    their bits are the row-streaming form's; the same for an identity search on the same rows"""
    n = 4000
    hs, H, mag, ln = _cfg3(ctx, n)
    gm = ctx.model_from_file(weights_path("weights_cfg1_id90"))
    a = ctx.all_pairs(gm, hs, hs, 0.9, upper_only=True, max_out=n * n)
    st = ctx.last_sweep()
    assert st["coarse"] and st["n_exact"] > 0 and st["n_inline"] == 0, st
    assert a["n_out"] > 0
    b = _legacy(lambda: ctx.all_pairs(gm, hs, hs, 0.9, upper_only=True, max_out=n * n))
    assert not ctx.last_sweep()["coarse"]
    _same(a, b)
    rm = _regression(ctx, H, mag, ln, np.random.default_rng(5))
    for t in (0.5, 0.9):
        a = ctx.identity_pairs(rm, hs, hs, t, 0.9, upper_only=True, max_out=n * n)
        st = ctx.last_sweep()
        assert st["coarse"] and st["n_inline"] == 0, (t, st)
        b = _legacy(lambda: ctx.identity_pairs(rm, hs, hs, t, 0.9, upper_only=True, max_out=n * n))
        _same(a, b, "identity")


def test_overflow_inline(built_lib, ctx):
    """a square identity search whose screen keeps more than 2^23 pairs: the pairs beyond the buffer are refined inside the
    sweep (n_inline > 0), and the result is the row-streaming form's"""
    rng = np.random.default_rng(17)
    n = 6000
    H = synth_hist(rng, n, 5, 1, hi=6)
    ln = rng.integers(950, 1050, n).astype(np.uint64)
    mag = H.sum(axis=1, dtype=np.uint64)
    hs = ctx.hset_from_host(H, 5, mag=mag, length=ln)
    rm = _regression(ctx, H, mag, ln, rng)
    t = 0.05
    a = ctx.identity_pairs(rm, hs, hs, t, 0.9, max_out=n * n)
    st = ctx.last_sweep()
    assert st["coarse"] and st["n_exact"] > CAND_CAP and st["n_inline"] > 0, st
    assert st["n_inline"] < st["n_exact"]
    b = _legacy(lambda: ctx.identity_pairs(rm, hs, hs, t, 0.9, max_out=n * n))
    _same(a, b, "identity")


def test_max_out_truncation(built_lib, ctx):
    """more survivors than max_out: the count stays exact and the pairs returned are distinct survivors with their bits"""
    n = 3000
    hs, H, mag, ln = _cfg3(ctx, n)
    gm = ctx.model_from_file(weights_path("weights_cfg1_id90"))
    full = ctx.all_pairs(gm, hs, hs, 0.9, upper_only=True, max_out=n * n)
    assert full["n_out"] > 100
    want = {(int(q), int(d)): int(s) for q, d, s in zip(full["q"], full["d"], full["score"].view(np.uint64))}
    for cap in (1, 37, int(full["n_out"]) // 3, int(full["n_out"]) - 1):
        r = ctx.all_pairs(gm, hs, hs, 0.9, upper_only=True, max_out=cap)
        assert ctx.last_sweep()["coarse"]
        assert r["n_out"] == full["n_out"] and r["n_scored"] == full["n_scored"]
        got = {(int(q), int(d)): int(s) for q, d, s in zip(r["q"][:cap], r["d"][:cap], r["score"][:cap].view(np.uint64))}
        assert len(got) == cap
        assert all(want[k] == v for k, v in got.items())


def test_topk_and_strands(built_lib, ctx):
    """identity top-K, both-strand pairs and both-strand top-K on the coarse form equal the row-streaming form's"""
    n = 3000
    hs, H, mag, ln = _cfg3(ctx, n)
    rm = _regression(ctx, H, mag, ln, np.random.default_rng(9))
    for t in (0.5, 0.9):
        a = ctx.identity_topk(rm, hs, hs, t, 10, 0.9, exclude_self=True)
        assert ctx.last_sweep()["coarse"]
        b = _legacy(lambda: ctx.identity_topk(rm, hs, hs, t, 10, 0.9, exclude_self=True))
        for key in ("d", "count", "n_hits"):
            assert np.array_equal(a[key], b[key]), (t, key)
        assert np.array_equal(a["identity"].view(np.uint64), b["identity"].view(np.uint64)), t

        a = ctx.identity_pairs_both_strands(rm, hs, hs, t, 0.9, upper_only=True, max_out=n * n)
        assert ctx.last_sweep()["coarse"]
        b = _legacy(lambda: ctx.identity_pairs_both_strands(rm, hs, hs, t, 0.9, upper_only=True, max_out=n * n))
        assert a["n_out"] == b["n_out"]
        oa, ob = np.lexsort((a["d"], a["q"])), np.lexsort((b["d"], b["q"]))
        for key in ("q", "d", "strand"):
            assert np.array_equal(a[key][oa], b[key][ob]), (t, key)
        assert np.array_equal(a["identity"][oa].view(np.uint64), b["identity"][ob].view(np.uint64)), t

        a = ctx.identity_topk_both_strands(rm, hs, hs, t, 10, 0.9, upper_only=True)
        assert ctx.last_sweep()["coarse"]
        b = _legacy(lambda: ctx.identity_topk_both_strands(rm, hs, hs, t, 10, 0.9, upper_only=True))
        for key in ("d", "strand", "count", "n_hits"):
            assert np.array_equal(a[key], b[key]), (t, key)
        assert np.array_equal(a["identity"].view(np.uint64), b["identity"].view(np.uint64)), t
