"""GPU: staged greedy clustering (mc2_greedy_*, Context.greedy_begin) against the single call mc2_identity_greedy_clusters.
A block loop on the host sweeps each query-row block part by part (shares from dist.block_shares, as the ranks of
all_pairs_step(greedy=True) would), splits a block whose parts overflow, and adds it; rep, the bits of identity, strand,
n_clusters and the summed n_scored must equal the single call's, for every sweep form, both strands, row ranges, 1 to 8
parts simulated on one GPU, fixed and random block tilings with other calls between stages, and overflowing parts.  Also
the argument errors and a corrupted slot."""
import ctypes as C

import numpy as np
import pytest

from conftest import weights_path
from helpers import all_singles_model
from meshclust2_b200 import dist as mdist
from test_gpu_both_strands import _strand_data
from test_gpu_identity_components import _big_case, _edge_t
from test_gpu_identity_greedy import _flat, _greedy_call
from test_gpu_identity_pairs import FLAGS5, TINY, _legacy, _regression, _spread

pytestmark = pytest.mark.gpu


def _staged(ctx, gm, hs, t, both=False, rows=None, n_parts=1, blocks=None, cap=0, between=None, cutoff=0.9):
    """the block loop of all_pairs_step(greedy=True) with every part swept on this GPU.  blocks: None = the grow / shrink
    policy from a whole-range first block, else the block sizes to try in turn (an overflowing one is split)"""
    b0, b1 = rows or (0, len(hs))
    g = ctx.greedy_begin(gm, hs, t, cutoff, both_strands=both, range=(b0, b1), n_parts=n_parts, part_capacity=cap)
    try:
        capacity = g.part_arrays(0)["capacity"]
        sizes = iter(blocks) if blocks is not None else None
        qb, size, want, n_scored, splits = b0, b1 - b0, None, 0, 0
        while qb < b1:
            if sizes is not None and want is None:
                want = next(sizes)
            qe = qb + min(want if sizes is not None else size, b1 - qb)
            shares = mdist.block_shares(qb, qe, b1, n_parts)
            res = [g.sweep_part(p, *shares[p]) for p in range(n_parts)]
            counts = [r[0] for r in res]
            most = max(counts)
            if most > capacity:
                span = qe - qb
                size = want = max(1, min(span // 2, int(float(span) * float(capacity // 2) / float(most))))
                splits += 1
                continue
            g.add_block(qb, qe, shares, counts)
            if between is not None:
                between()
            n_scored += sum(r[1] for r in res)
            qb, want = qe, None
            if most < capacity // 4:
                size = min(size * 2, b1 - b0)
        out = g.end()
    finally:
        g.free()
    out.update(n_scored=n_scored, splits=splits)
    return out


def _same(got, want):
    assert got["rep"].dtype == np.uint64 and np.array_equal(got["rep"], want["rep"])
    assert np.array_equal(got["identity"].view(np.uint64), want["identity"].view(np.uint64))
    assert np.array_equal(got["strand"], want["strand"])
    assert got["n_clusters"] == want["n_clusters"] and got["n_scored"] == want["n_scored"]


def _case(ctx, capi, case):
    """the sets of test_gpu_identity_greedy.test_greedy_vs_reference: about a quarter of the rows are other rows' reverse
    complements"""
    rng = np.random.default_rng(47 if case == "k8_u16" else ["coarse", "full", "legacy", "u16_big"].index(case) + 20)
    k, eb, D, Q = _strand_data(rng, case)
    H = np.concatenate([D[0], Q[0]])
    mag, ln = np.concatenate([D[1], Q[1]]), np.concatenate([D[2], Q[2]])
    om = _spread(all_singles_model(FLAGS5, H, mag, ln, rng, n_combos=4), H, mag, ln, rng)
    gm = _regression(ctx, capi, om)
    hs = ctx.hset_from_host(H, k, mag=mag, length=ln)
    ts = (0.0, TINY) if case == "full" else (0.9, 0.5, _edge_t(ctx, gm, hs))
    return gm, hs, ts


@pytest.mark.parametrize("case", ["coarse", "full", "legacy", "u16_big", "k8_u16"])
def test_one_part_equals_single_call(built_lib, ctx, case):
    """n_parts = 1 and the default capacity: every sweep form, one and both strands, the whole set and begin > 0"""
    gm, hs, ts = _case(ctx, built_lib, case)
    n = len(hs)
    seen = []

    def go():
        for t in ts:
            for rng_ in ((0, n), (5, n - 3)):
                for both in (False, True):
                    want = _greedy_call(ctx, gm, hs, t, both, rng_)
                    got = _staged(ctx, gm, hs, t, both, rng_)
                    _same(got, want)
                    seen.append(1 < got["n_clusters"] < rng_[1] - rng_[0])
    _legacy(go) if case == "legacy" else go()
    assert case == "full" or any(seen)


def test_sweep_part_reports_the_flat_sweep(built_lib, ctx):
    """a whole-range part sweep makes the flat call's sweep (mc2_debug_last_sweep) and finds its edges"""
    gm, hs, _ = _case(ctx, built_lib, "coarse")
    n = len(hs)
    for both in (False, True):
        flat = _flat(ctx, gm, hs, 0.5, both, (0, n), 0.9)
        sweep = ctx.last_sweep()
        g = ctx.greedy_begin(gm, hs, 0.5, 0.9, both_strands=both)
        ne, ns = g.sweep_part(0, 0, n)
        assert ctx.last_sweep()["n_exact"] == sweep["n_exact"] and ctx.last_sweep()["coarse"] == sweep["coarse"]
        assert (ne, ns) == (flat["n_out"], flat["n_scored"])
        g.free()


@pytest.mark.parametrize("n_parts", [2, 3, 8])
def test_parts_simulated_on_one_gpu(built_lib, ctx, n_parts):
    """n_parts shares per block from dist.block_shares, with the grow / shrink policy and with blocks of 5 rows (fewer rows
    than parts at 8: empty shares)"""
    gm, hs, ts = _case(ctx, built_lib, "coarse")
    n = len(hs)
    for t in ts:
        for both in (False, True):
            for rng_ in ((0, n), (7, n)):
                want = _greedy_call(ctx, gm, hs, t, both, rng_)
                _same(_staged(ctx, gm, hs, t, both, rng_, n_parts=n_parts), want)
                _same(_staged(ctx, gm, hs, t, both, rng_, n_parts=n_parts, blocks=[5] * n), want)


def test_tilings_with_other_calls_between(built_lib, ctx):
    """seeded random block tilings, with identity_pairs on another set, identity_components on the same set and a top-K
    between the stages (they share the context's scratch)"""
    gm, hs, ts = _case(ctx, built_lib, "coarse")
    gm2, hs2, _ = _case(ctx, built_lib, "u16_big")
    n = len(hs)
    rng = np.random.default_rng(5)

    def between():
        ctx.identity_pairs(gm2, hs2, hs2, 0.5, 0.9, upper_only=True, max_out=1 << 16)
        ctx.identity_components(gm, hs, 0.5, 0.9, both_strands=True)
        ctx.identity_topk(gm, hs, hs, 0.5, 4, 0.9, upper_only=True)

    for t in ts:
        for both in (False, True):
            want = _greedy_call(ctx, gm, hs, t, both)
            for n_parts in (1, 3):
                blocks = rng.integers(1, max(2, n // 4), size=n).tolist()
                _same(_staged(ctx, gm, hs, t, both, n_parts=n_parts, blocks=blocks, between=between), want)


def test_overflow_splits_and_resweeps(built_lib, ctx):
    """3 000 rows at the smallest positive t with part_capacity = n: most in-window pairs are edges, parts overflow, the
    loop splits and sweeps again, and the result is still the single call's"""
    n = 3000
    gm, hs = _big_case(ctx, built_lib, 97, n, dense=True)
    for both, n_parts in ((False, 1), (False, 2), (True, 2)):
        want = _greedy_call(ctx, gm, hs, TINY, both)
        got = _staged(ctx, gm, hs, TINY, both, n_parts=n_parts, cap=n)
        assert got["splits"] > 0
        _same(got, want)


def test_errors(built_lib, ctx):
    import torch
    capi = built_lib
    gm, hs, _ = _case(ctx, capi, "coarse")
    n = len(hs)

    def err(fn, *a, **kw):
        with pytest.raises(capi.Mc2Error) as e:
            fn(*a, **kw)
        assert e.value.status == -1

    err(ctx.greedy_begin, gm, hs, 0.5, 0.9, n_parts=0)
    err(ctx.greedy_begin, gm, hs, 0.5, 0.9, part_capacity=n - 1)
    err(ctx.greedy_begin, ctx.model_from_file(weights_path("weights_cfg1_id90")), hs, 0.5, 0.9)
    err(ctx.greedy_begin, gm, hs, float("nan"), 0.9)
    err(ctx.greedy_begin, gm, hs, 0.5, 0.9, range=(0, n + 1))
    g = ctx.greedy_begin(gm, hs, 0.5, 0.9, n_parts=2, range=(4, n))
    err(g.sweep_part, 2, 4, 10)                              # part index >= n_parts
    err(g.sweep_part, 0, 3, 10)                              # below begin
    err(g.sweep_part, 0, 10, n + 1)                          # past end
    err(g.end)                                               # rows undecided
    assert g.sweep_part(0, 4, 4) == (0, 0)
    assert g.sweep_part(1, 4, 4) == (0, 0)
    g.add_block(4, 4, [(4, 4), (4, 4)], [0, 0])             # an empty block changes nothing
    cap = g.part_arrays(0)["capacity"]
    mid = n // 2
    shares = mdist.block_shares(4, mid, n, 2)
    s = shares[0][1]
    counts = [g.sweep_part(p, *shares[p])[0] for p in range(2)]
    assert counts[1] > 0
    err(g.add_block, 5, mid, [(5, s), (s, mid)], counts)                # not the next undecided row
    err(g.add_block, 4, n + 1, [(4, s), (s, n + 1)], counts)            # past end
    err(g.add_block, 4, mid, [(4, s), (s + 1, mid)], counts)            # a gap
    err(g.add_block, 4, mid, [(s, mid), (4, s)], counts)                # out of part order
    err(g.add_block, 4, mid, [(4, s), (s, mid - 1)], counts)            # short of qe
    err(g.add_block, 4, mid, shares, [counts[0], cap + 1])              # a count above capacity
    # a record of part 1 whose r lies in part 0's range: refused before any state changes
    rec = torch.as_tensor(g.part_arrays(1)["records"], device="cuda")
    keep = rec[0].clone()
    r32 = rec.view(torch.int32)
    r32[0, 0] = shares[0][0] - 4
    torch.cuda.synchronize()
    err(g.add_block, 4, mid, shares, counts)
    rec[0] = keep
    r32[0, 1] = r32[0, 0]                                               # c outside (r, end) is refused as well
    torch.cuda.synchronize()
    err(g.add_block, 4, mid, shares, counts)
    rec[0] = keep
    torch.cuda.synchronize()
    g.add_block(4, mid, shares, counts)
    err(g.sweep_part, 0, mid - 1, n)                                    # below the next undecided row
    shares = mdist.block_shares(mid, n, n, 2)
    counts = [g.sweep_part(p, *shares[p])[0] for p in range(2)]
    g.add_block(mid, n, shares, counts)
    got = g.end()
    g.free()
    _same(dict(got, n_scored=0), dict(_greedy_call(ctx, gm, hs, 0.5, range=(4, n)), n_scored=0))
    # the C entry points' NULL checks
    L = capi.lib()
    h = C.c_void_p()
    assert L.mc2_greedy_begin(ctx.h, gm.h, 0.5, 0, hs.h, 0, n, 0.9, 1, 0, None) == -1
    assert L.mc2_greedy_begin(ctx.h, gm.h, 0.5, 0, hs.h, 0, n, 0.9, 1, 0, C.byref(h)) == 0
    assert L.mc2_greedy_sweep_part(ctx.h, h, 0, 0, 1, None, None) == -1
    assert L.mc2_greedy_end(ctx.h, h, None, None, None, None) == -1
    L.mc2_greedy_free(h)
