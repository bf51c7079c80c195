"""GPU: every K1 (k-mer histogram) route against the reference, every row and every field, on whole batches.

The routes of kmer_count.cu are picked per batch (average length, k, width, longest read, batch size), so each test
builds the batch that reaches the route it is about and compares every row with exact references:
  * histograms: the C oracle (oracle.port.count_batch), which restates the reference's fill_table;
  * sum, sumsq, mag, mers1, len, max_count and the per-segment overflow count: exact integer arithmetic in numpy from
    k-mer counts taken over the same segments (a second, independent count), cross-checked against the oracle's
    histogram, port.count's overflow count and port.largest_count;
  * stddev: bit-equal to sqrt(float(N*sumsq - sum^2)) / N (what the device computes) and within 1e-12 of the oracle's
    two-pass value.
sum and sumsq are read straight from the device side-band with cudaMemcpy on the CUDA runtime torch loads.
"""
import ctypes
import math

import numpy as np
import pytest

from oracle import port
from meshclust2_b200 import synth

pytestmark = pytest.mark.gpu

TMAX = {1: 0xFF, 2: 0xFFFF, 4: 0xFFFFFFFF, 8: 0xFFFFFFFFFFFFFFFF}
FIELDS = ("hist", "mag", "sum", "sumsq", "len", "mers1", "stddev", "n_overflow", "max_count")


# ---------------------------------------------------------------------------------------------------------------------
# batches: concatenated codes + sequence-relative segment lists, as ctx.upload_seqs takes them
# ---------------------------------------------------------------------------------------------------------------------
def _batch(items):
    """items: [(codes int8[L], segs int32[m, 2])] -> dict(codes, seq_off, segs, seg_off)"""
    n = len(items)
    seq_off = np.zeros(n + 1, dtype=np.uint64)
    seg_off = np.zeros(n + 1, dtype=np.uint64)
    if n:
        seq_off[1:] = np.cumsum([len(c) for c, _ in items])
        seg_off[1:] = np.cumsum([len(s) for _, s in items])
    codes = np.concatenate([np.asarray(c, dtype=np.int8) for c, _ in items] + [np.zeros(0, dtype=np.int8)])
    segs = np.concatenate([np.asarray(s, dtype=np.int32).reshape(-1, 2) for _, s in items] + [np.zeros((0, 2), np.int32)])
    return dict(codes=codes, seq_off=seq_off, segs=segs, seg_off=seg_off)


def _encode(texts):
    return _batch([port.encode(t)[:2] for t in texts])


def _rows(b, lo, hi):
    """rows [lo, hi) of a batch as a batch of their own"""
    so, go = b["seq_off"], b["seg_off"]
    return dict(codes=b["codes"][int(so[lo]):int(so[hi])], seq_off=so[lo:hi + 1] - so[lo],
                segs=b["segs"][int(go[lo]):int(go[hi])], seg_off=go[lo:hi + 1] - go[lo])


def _row(b, i):
    so, go = b["seq_off"], b["seg_off"]
    return b["codes"][int(so[i]):int(so[i + 1])], b["segs"][int(go[i]):int(go[i + 1])]


def _upload(ctx, b):
    return ctx.upload_seqs(b["codes"], b["seq_off"], b["segs"], b["seg_off"])


# ---------------------------------------------------------------------------------------------------------------------
# the device side-band, read back with a plain cudaMemcpy
# ---------------------------------------------------------------------------------------------------------------------
_RT = []


def _cudart():
    if not _RT:
        import torch
        torch.cuda.init()
        path = "libcudart.so.12"
        with open("/proc/self/maps") as f:
            for line in f:
                if "libcudart.so" in line:
                    path = line.split()[-1]
                    break
        rt = ctypes.CDLL(path)
        rt.cudaMemcpy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
        rt.cudaMemcpy.restype = ctypes.c_int
        _RT.append(rt)
    return _RT[0]


def device_sideband(hs, which, first=0, count=None):
    """rows [first, first + count) of side-band column `which` (0 mag, 1 len, 2 sum, 3 sumsq) via cudaMemcpy D2H"""
    count = len(hs) - first if count is None else count
    out = np.zeros(count, dtype=np.uint64)
    if count:
        src = hs.device_sideband(which) + 8 * first
        rc = _cudart().cudaMemcpy(out.ctypes.data, src, count * 8, 2)  # cudaMemcpyDeviceToHost
        assert rc == 0, "cudaMemcpy failed: %d" % rc
    return out


def _device(hs, first=0, count=None):
    got = hs.download(first, count)
    got["sum"] = device_sideband(hs, 2, first, count)
    got["sumsq"] = device_sideband(hs, 3, first, count)
    return got


# ---------------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------------
def _exact_counts(b, k, r0, r1):
    """Exact k-mer counts (int64, no init, no saturation) of rows [r0, r1) from the codes inside their segments:
    per row [r1 - r0, N], per segment [segments of those rows, N] (with each segment's row), and per row the effective
    length and the 1-mer counts [r1 - r0, 4]."""
    N = 4 ** k
    so, go = b["seq_off"].astype(np.int64), b["seg_off"].astype(np.int64)
    p0, p1 = so[r0], so[r1]
    g0, g1 = go[r0], go[r1]
    nseg, nrow = int(g1 - g0), r1 - r0
    codes = b["codes"][p0:p1].astype(np.int64) & 3
    T = len(codes)
    seg_row = np.repeat(np.arange(nrow), np.diff(go[r0:r1 + 1]))
    segs = b["segs"][g0:g1].astype(np.int64)
    gs = so[r0:r1][seg_row] - p0 + segs[:, 0]
    ge = so[r0:r1][seg_row] - p0 + segs[:, 1]
    length = np.bincount(seg_row, weights=ge - gs + 1, minlength=nrow).astype(np.int64)
    # every position inside a segment, tagged with 1 + its segment's index (segments are disjoint)
    sid = np.arange(nseg, dtype=np.int64)
    tag = np.zeros(T + 1, dtype=np.int64)
    np.add.at(tag, gs, sid + 1)
    np.add.at(tag, ge + 1, -(sid + 1))
    tag = np.cumsum(tag)[:T]
    inside = np.nonzero(tag)[0]
    mers1 = np.bincount(seg_row[tag[inside] - 1] * 4 + codes[inside], minlength=4 * nrow).reshape(nrow, 4)
    # k-mer starts: gs .. ge - k + 1 of the segments that hold >= k bases
    starts = inside[inside + k - 1 <= ge[tag[inside] - 1]]
    idx = np.zeros(len(starts), dtype=np.int64)
    for t in range(k):
        idx = idx * 4 + codes[starts + t]
    per_seg = np.bincount((tag[starts] - 1) * N + idx, minlength=nseg * N).reshape(nseg, N)
    per_row = np.zeros((nrow, N), dtype=np.int64)
    have = np.nonzero(np.diff(go[r0:r1 + 1]))[0]
    if len(have):
        per_row[have] = np.add.reduceat(per_seg, go[r0:r1][have] - g0, axis=0)
    return per_row, per_seg, seg_row, length, mers1


def _reference(b, k, ebs, init=1):
    """{eb: dict(FIELDS..., sd_two_pass)} for every row of batch b, with the table init count_kmers uses (1)."""
    N = 4 ** k
    n = len(b["seq_off"]) - 1
    so, go = b["seq_off"].astype(np.int64), b["seg_off"].astype(np.int64)
    out = {}
    for eb in ebs:
        out[eb] = dict(hist=port.count_batch(b["codes"], b["seq_off"], b["segs"], b["seg_off"], k, eb, threads=8)[0],
                       mag=np.zeros(n, np.uint64), sum=np.zeros(n, np.uint64), sumsq=np.zeros(n, np.uint64),
                       len=np.zeros(n, np.uint64), mers1=np.zeros((n, 4), np.uint64), n_overflow=np.zeros(n, np.int32),
                       max_count=np.zeros(n, np.uint32), stddev=np.zeros(n), sd_two_pass=np.zeros(n),
                       ovf_closed=np.zeros(n, np.int32))
    # chunks of rows: [rows + segments, N] int64 near 32 MB, at most 4 M bases
    cap = max(1, (4 << 20) // N)
    r0 = 0
    while r0 < n:
        r1 = r0 + 1
        while r1 < n and (r1 + 1 - r0) + (go[r1 + 1] - go[r0]) <= cap and so[r1 + 1] - so[r0] <= (4 << 20):
            r1 += 1
        per_row, per_seg, srow, length, mers1 = _exact_counts(b, k, r0, r1)
        mx = per_row.max(axis=1)
        # each segment's running total within its read: cum[s] - cum[last segment of the previous read]
        cum = np.cumsum(per_seg, axis=0)
        first = (go[r0:r1] - go[r0])[srow]
        cum -= np.where((first > 0)[:, None], cum[np.maximum(first - 1, 0)], 0)
        for eb in ebs:
            o = out[eb]
            tmax = TMAX[eb]
            h = np.minimum(init + per_row, tmax) if eb <= 4 else init + per_row
            # segment s overflows iff some bin occurs in s and init + its occurrences up to and including s > max(T)
            seg_ovf = ((per_seg > 0) & (init + cum > tmax)).any(axis=1) if eb <= 4 else np.zeros(len(per_seg), bool)
            assert np.array_equal(h, o["hist"][r0:r1].astype(np.int64)), "reference counts disagree with the oracle"
            o["sum"][r0:r1] = h.sum(axis=1)
            o["sumsq"][r0:r1] = (h * h).sum(axis=1)
            o["max_count"][r0:r1] = mx
            o["len"][r0:r1] = length
            o["mers1"][r0:r1] = 1 + mers1
            o["ovf_closed"][r0:r1] = np.bincount(srow, weights=seg_ovf, minlength=r1 - r0).astype(np.int32)
        r0 = r1
    for eb in ebs:
        o = out[eb]
        o["mag"] = o["sum"].copy()
        for i in range(n):
            s, q = int(o["sum"][i]), int(o["sumsq"][i])
            o["stddev"][i] = math.sqrt(float(N * q - s * s)) / N
            o["sd_two_pass"][i] = port.point_stats(o["hist"][i])[1]
            c, sg = _row(b, i)
            o["n_overflow"][i] = port.count(c, sg, k, eb)[2]
        assert np.array_equal(o["n_overflow"], o["ovf_closed"]), "closed-form overflow count disagrees with the oracle"
    # largest_count is defined where every segment holds >= k bases
    o = out[ebs[0]]
    for i in range(n):
        c, sg = _row(b, i)
        if len(sg) and (sg[:, 1] - sg[:, 0] + 1 >= k).all():
            assert port.largest_count(c, sg, k) - 1 == o["max_count"][i], i
    return out


def _first_bad(a, w):
    bad = np.nonzero((a != w).reshape(len(a), -1).any(axis=1))[0]
    return int(bad[0]) if len(bad) else None


def _check(got, want, tag, sd_tol=1e-12):
    """every row, every field: bits, and the stddev within sd_tol (relative) of the oracle's two-pass value"""
    for f in FIELDS:
        a, w = got[f], want[f]
        assert a.shape[0] == w.shape[0], (tag, f)
        if f == "stddev":
            ok = a.view(np.uint64) == w.view(np.uint64)
        else:
            assert a.dtype == w.dtype, (tag, f, a.dtype, w.dtype)
            ok = (a == w).reshape(len(a), -1).all(axis=1)
        if not ok.all():
            i = int(np.nonzero(~ok)[0][0])
            if f == "hist":
                d = np.nonzero(a[i] != w[i])[0]
                extra = " bins %s: got %s want %s" % (d[:6].tolist(), a[i][d[:6]].tolist(), w[i][d[:6]].tolist())
            else:
                extra = ": got %s want %s" % (a[i], w[i])
            pytest.fail("%s: field %s differs in %d rows, first row %d%s" % (tag, f, int((~ok).sum()), i, extra))
    sd, ref = got["stddev"], want["sd_two_pass"]
    far = np.nonzero(np.abs(sd - ref) > sd_tol * np.abs(ref))[0]
    assert len(far) == 0, "%s: stddev of row %d is %r, the two-pass value %r" % (tag, far[0], sd[far[0]], ref[far[0]])


def _same(a, b, tag):
    """two device results hold the same bits in every field"""
    for f in FIELDS:
        x, y = a[f], b[f]
        if f == "stddev":
            x, y = x.view(np.uint64), y.view(np.uint64)
        if not np.array_equal(x, y):
            pytest.fail("%s: field %s differs, first row %s" % (tag, f, _first_bad(x, y)))


def _count(ctx, b, k, eb):
    hs = ctx.count_kmers(_upload(ctx, b), k, eb)
    return hs, _device(hs)


# ---------------------------------------------------------------------------------------------------------------------
# 1. whole batches
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cfg3", "cfg2"])
def test_config_sets_every_row(ctx, name):
    """cfg3: 100k x 950-1 050 bases (straddling the 1 008-base common path), cfg2: 10k x 1.5 kb; k = 5, uint8."""
    seqs, _, k, eb = synth.make_config_range(name)
    b = _encode(seqs)
    del seqs
    _, got = _count(ctx, b, k, eb)
    _check(got, _reference(b, k, (eb,))[eb], name)


def _random_codes(rng, n):
    return rng.integers(0, 4, n).astype(np.int8)


def _text(rng, n):
    return np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].tobytes()


def _mixed_texts(n, seed):
    """Reads whose shapes are drawn at random, so every transition between shapes happens inside one warp's walk."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        u = rng.random()
        if u < 0.002:                                              # long: 20-80 kb
            out.append(_text(rng, int(rng.integers(20000, 80001))))
        elif u < 0.35:                                             # common: one segment from 0, <= 1 008 bases
            out.append(_text(rng, int(rng.integers(21, 1009))))
        elif u < 0.55:                                             # generic single segment: 1 009-4 000 bases
            out.append(_text(rng, int(rng.integers(1009, 4001))))
        elif u < 0.70:                                             # leading N run of 1-40
            out.append(b"N" * int(rng.integers(1, 41)) + _text(rng, int(rng.integers(21, 1500))))
        elif u < 0.85:                                             # several segments split by N runs >= 10
            parts = [_text(rng, int(rng.integers(20, 700))) for _ in range(int(rng.integers(2, 6)))]
            seps = [b"N" * int(rng.integers(10, 40)) for _ in parts[1:]]
            t = parts[0] + b"".join(s + p for s, p in zip(seps, parts[1:]))
            out.append(t.lower() if rng.random() < 0.2 else t)
        elif u < 0.90:                                             # all N
            out.append(b"N" * int(rng.integers(1, 300)))
        elif u < 0.95:                                             # empty
            out.append(b"")
        else:                                                      # shorter than k (for k >= 2)
            out.append(_text(rng, int(rng.integers(1, 6))))
    return out


_CACHE = {}


@pytest.fixture(scope="module")
def mixed(ctx):
    """at least 3 x 64 x sm_count reads: 64 resident warps per SM at most, so every warp walks >= 3 reads"""
    n = 3 * 64 * ctx.sm_count + 101
    texts = _mixed_texts(n, seed=2024)
    return texts, _encode(texts)


def _mixed_ref(mixed, k, eb):
    key = ("mixed", k)
    if key not in _CACHE:
        _CACHE.clear()
        _CACHE[key] = _reference(mixed[1], k, (1, 2, 4, 8) if k == 5 else (1, 2))
    return _CACHE[key][eb]


@pytest.mark.parametrize("k,eb", [(1, 1), (1, 2), (3, 1), (3, 2), (5, 1), (5, 2), (5, 4), (5, 8), (6, 1), (6, 2)])
def test_mixed_batch_every_row(ctx, mixed, k, eb):
    """u8/u16: count_warp_kernel with its next-sequence pipeline; u32/u64: count_kernel's warp form"""
    _, got = _count(ctx, mixed[1], k, eb)
    _check(got, _mixed_ref(mixed, k, eb), "mixed k=%d eb=%d" % (k, eb))


@pytest.mark.parametrize("k,eb", [(5, 2), (3, 1)])
def test_mixed_batch_in_uneven_slices(ctx, mixed, k, eb):
    """the same reads counted in slices of uneven size (some small enough to change route) give the same bits"""
    b = mixed[1]
    n = len(b["seq_off"]) - 1
    _, whole = _count(ctx, b, k, eb)
    cuts = [0, 1, 38, 1038, 1039, 7777, n - 5, n]
    parts = [_count(ctx, _rows(b, lo, hi), k, eb)[1] for lo, hi in zip(cuts[:-1], cuts[1:])]
    joined = {f: np.concatenate([p[f] for p in parts]) for f in FIELDS}
    _same(joined, whole, "slices k=%d eb=%d" % (k, eb))


# ---------------------------------------------------------------------------------------------------------------------
# 2. segment lengths and offsets
# ---------------------------------------------------------------------------------------------------------------------
def _segment_shapes(k, seed):
    rng = np.random.default_rng(seed)
    items = []
    for L in range(1, 1101):                                      # every length, s0 = 0: 1 008 / 1 009 route change
        items.append((_random_codes(rng, L), [[0, L - 1]]))
    for s0 in range(48):                                          # s0 0..47 against e0 at every residue mod 16
        for r in range(16):
            for j in (0, 1, 3, 31, 63, 66):
                e0 = 16 * (s0 // 16 + j) + r
                if e0 < s0:
                    e0 += 16
                items.append((_random_codes(rng, e0 + 1 + int(rng.integers(0, 20))), [[s0, e0]]))
    for d in (-1, 0, 1):                                          # k - 1, k and k + 1 bases
        for s0 in (0, 1, 7, 15, 16, 31, 40, 1000, 1015):
            ln = k + d
            if ln >= 1:
                items.append((_random_codes(rng, s0 + ln + int(rng.integers(0, 3))), [[s0, s0 + ln - 1]]))
    for _ in range(40):                                           # segments separated by one base
        segs, p = [], int(rng.integers(0, 20))
        for _ in range(int(rng.integers(2, 12))):
            ln = int(rng.integers(1, 60))
            segs.append([p, p + ln - 1])
            p += ln + 1
        items.append((_random_codes(rng, p + int(rng.integers(0, 5))), segs))
    segs, p = [], 3                                               # one read with 200 segments
    for _ in range(200):
        ln = int(rng.integers(1, 40))
        segs.append([p, p + ln - 1])
        p += ln + int(rng.integers(1, 6))
    items.append((_random_codes(rng, p), segs))
    perm = rng.permutation(len(items))                            # neighbours of every shape inside one warp's walk
    return _batch([items[i] for i in perm])


@pytest.mark.parametrize("k", [1, 2, 5, 6, 7])
def test_segment_lengths_and_offsets(ctx, k):
    b = _segment_shapes(k, seed=70 + k)
    ref = _reference(b, k, (1, 2))
    for eb in (1, 2):
        _, got = _count(ctx, b, k, eb)
        _check(got, ref[eb], "segments k=%d eb=%d" % (k, eb))


# ---------------------------------------------------------------------------------------------------------------------
# 3. dispatch boundaries: each pair differs only in the route
# ---------------------------------------------------------------------------------------------------------------------
def _pad(b, row, extra, code=2):
    """the same batch with `extra` bases appended to one read outside its segments"""
    items = [_row(b, i) for i in range(len(b["seq_off"]) - 1)]
    c, s = items[row]
    items[row] = (np.concatenate([c, np.full(extra, code, np.int8)]), s)
    return _batch(items)


def _count_launches(ctx, b, k, eb):
    sq = _upload(ctx, b)
    l0 = ctx.launches
    hs = ctx.count_kmers(sq, k, eb)
    return ctx.launches - l0, _device(hs)


@pytest.mark.parametrize("eb", [1, 2, 4])
def test_average_length_4096_against_4097(ctx, eb):
    """total_bases / n == 4 096 takes the warp route, 4 097 the CTA route (one read padded outside its segments)"""
    rng = np.random.default_rng(4096)
    items = []
    for i in range(40):
        c = _random_codes(rng, 4096)
        if i % 4 == 0:
            segs = [[0, 4095]]
        elif i % 4 == 1:
            segs = [[int(rng.integers(1, 40)), 4095 - int(rng.integers(0, 30))]]
        elif i % 4 == 2:
            segs = [[0, 999], [1010, 2500], [2520, 4095]]
        else:
            c[:] = 0
            segs = [[0, 4095]]                                    # poly-A: saturates u8
        items.append((c, segs))
    b4096 = _batch(items)
    b4097 = _pad(b4096, 7, 40)
    assert b4096["seq_off"][-1] // 40 == 4096 and b4097["seq_off"][-1] // 40 == 4097
    ref = _reference(b4096, 5, (eb,))[eb]
    _, warp = _count(ctx, b4096, 5, eb)
    _, cta = _count(ctx, b4097, 5, eb)
    _check(warp, ref, "avg 4096")
    _check(cta, ref, "avg 4097")


@pytest.mark.parametrize("k,eb", [(5, 1), (5, 2), (6, 1), (6, 2)])
def test_long_poly_a_among_short_reads(ctx, k, eb):
    """A 70 000-base poly-A among 120 x 1 kb reads keeps the average below 4 096, so the warp kernel counts it (u16
    saturates). A second long read adds 400 x AAAAAC to the poly-A: bins 0 and 1 then share a lane of the narrowing pass
    whose u16 sum of squares passes 2^32. Counted alone, each long read takes the CTA route."""
    rng = np.random.default_rng(70000 + k)
    longs = {57: b"A" * 70000, 90: b"A" * 70000 + b"AAAAAC" * 400}
    texts = [_text(rng, 1000) for _ in range(120)]
    for i in sorted(longs):
        texts.insert(i, longs[i])
    b = _encode(texts)
    ref = _reference(b, k, (eb,))[eb]
    if eb == 2:
        lanes = ref["hist"][90].astype(np.int64).reshape(-1, 32, 4)          # lane l narrows bins 4l..4l+3 of each 128
        assert ((lanes * lanes).sum(axis=(0, 2)) >= 1 << 32).any()
    _, got = _count(ctx, b, k, eb)
    _check(got, ref, "long among short")
    for i, t in longs.items():
        _, one = _count(ctx, _encode([t]), k, eb)
        _check(one, {f: v[i:i + 1] for f, v in ref.items()}, "long read %d alone" % i)
        assert got["n_overflow"][i] == 1 and int(got["hist"][i].max()) == TMAX[eb]


def _k8_reads(rng, longest, in_segment):
    """a poly-A read of `longest` bases whose segment holds `in_segment` of them, plus short and multi-segment reads"""
    c = np.zeros(longest, np.int8)
    items = [(c, [[0, in_segment - 1]]), (_random_codes(rng, 3000), [[0, 2999]]),
             (_random_codes(rng, 5000), [[0, 1199], [1300, 1320], [1340, 4999]]), (_random_codes(rng, 7), [[0, 6]]),
             (_random_codes(rng, 900), [[11, 899]])]
    return _batch(items)


@pytest.mark.parametrize("eb", [1, 2, 4])
def test_k8_packed_at_its_limit(ctx, eb):
    """k = 8: a longest read of 65 534 bases keeps init + max_len <= 65 535 (packed 16-bit shared histogram); the same
    segments in a 65 535-base read take the global path"""
    rng = np.random.default_rng(65534)
    packed = _k8_reads(rng, 65534, 65534)
    glob = _pad(packed, 0, 1, code=0)
    ref = _reference(packed, 8, (eb,))[eb]
    lp, got_p = _count_launches(ctx, packed, 8, eb)
    lg, got_g = _count_launches(ctx, glob, 8, eb)
    _check(got_p, ref, "k8 packed")
    _check(got_g, ref, "k8 global")
    assert lp == lg


def _short_reads(rng, n, with_long=None):
    items = []
    for i in range(n):
        L = int(rng.integers(40, 400))
        c = _random_codes(rng, L)
        if i % 5 == 1:
            segs = [[int(rng.integers(1, 20)), L - 1]]
        elif i % 5 == 2:
            segs = [[0, L // 3], [L // 3 + 2, L - 1]]
        else:
            segs = [[0, L - 1]]
        items.append((c, segs))
    if with_long is not None:
        row, L = with_long
        items[row] = (np.zeros(L, np.int8), [[0, L - 1]])
    return items


def test_k9_global_second_launch(ctx):
    """k = 9 counts in launches of 1 024 reads: 1 025 reads make a second launch with seq_begin = 1 024"""
    rng = np.random.default_rng(9)
    items = _short_reads(rng, 1025)
    items[1024] = (np.zeros(600, np.int8), [[0, 299], [301, 599]])    # saturates u8 in both segments
    b1025 = _batch(items)
    b1024 = _rows(b1025, 0, 1024)
    ref = _reference(b1025, 9, (1,))[1]
    l4, got4 = _count_launches(ctx, b1024, 9, 1)
    _check(got4, {f: v[:1024] for f, v in ref.items()}, "k9 1024")
    del got4
    l5, got5 = _count_launches(ctx, b1025, 9, 1)
    _check(got5, ref, "k9 1025")
    assert l5 == l4 + 1, (l4, l5)
    assert got5["n_overflow"][1024] == 2


def test_k8_global_second_launch(ctx):
    """k = 8 with a 65 535-base read counts in global memory in launches of 4 096 reads"""
    rng = np.random.default_rng(8)
    items = _short_reads(rng, 4097, with_long=(100, 65535))
    items[4096] = (np.zeros(700, np.int8), [[5, 300], [320, 699]])
    b4097 = _batch(items)
    b4096 = _rows(b4097, 0, 4096)
    ref = _reference(b4097, 8, (1,))[1]
    l6, got6 = _count_launches(ctx, b4096, 8, 1)
    _check(got6, {f: v[:4096] for f, v in ref.items()}, "k8 4096")
    del got6
    l7, got7 = _count_launches(ctx, b4097, 8, 1)
    _check(got7, ref, "k8 4097")
    assert l7 == l6 + 1, (l6, l7)


# ---------------------------------------------------------------------------------------------------------------------
# 4. saturation and overflow at the threshold
# ---------------------------------------------------------------------------------------------------------------------
def _runs_case(k, tmax, a_counts, lead=0, other=False):
    """One read of A-runs, one segment per entry of a_counts: segment s holds a_counts[s] occurrences of the all-A
    k-mer (and nothing else), or, with other=True and a count of 0, a C/G/T segment without it. Segments are separated
    by one C outside every segment."""
    codes, segs, p = [np.full(lead, 1, np.int8)], [], lead
    for c in a_counts:
        if c == 0 and other:
            run = np.tile(np.array([1, 2, 3], np.int8), 50)
        else:
            run = np.zeros(c + k - 1, np.int8)
        codes.append(run)
        segs.append([p, p + len(run) - 1])
        p += len(run)
        codes.append(np.ones(1, np.int8))
        p += 1
    return np.concatenate(codes), segs


def _threshold_cases(k, eb):
    """(items, expected n_overflow) with init 1: a bin reaching max(T) does not overflow, max(T) + 1 does"""
    T = TMAX[eb]
    cases = [
        ([T - 1], 0, 0), ([T], 0, 1),                       # single segment from base 0: flag from the bins' maximum
        ([T - 1], 13, 0), ([T], 13, 1),                     # single segment off a word boundary
        ([T - 1, 5], 0, 1), ([T, 5], 0, 2),                 # segment 2 has more of the saturated bin
        ([T - 1, 0], 0, 0), ([T, 0], 0, 1),                 # segment 2 has none of it
        ([T - 2, 1], 0, 0), ([T - 2, 2], 0, 1),             # segment 2 is the only one to overflow, or just reaches max
        ([T - 1, 1], 0, 1), ([5, T - 7, 1], 0, 0), ([5, T - 6, 1], 0, 1), ([5, T - 5, 1], 0, 2),
    ]
    items, want = [], []
    for counts, lead, novf in cases:
        items.append(_runs_case(k, T, counts, lead, other=True))
        want.append(novf)
    return items, want


@pytest.mark.parametrize("k,eb", [(5, 1), (5, 2), (6, 1), (6, 2), (7, 1), (7, 2), (8, 1), (8, 2), (9, 1), (9, 2)])
def test_saturation_and_overflow_threshold(ctx, k, eb):
    """k = 5, 6: warp kernel (short fillers keep the average <= 4 096); k = 7: CTA; k = 8: packed u8 / global u16;
    k = 9: global"""
    items, want = _threshold_cases(k, eb)
    rng = np.random.default_rng(100 * k + eb)
    if k <= 6:
        total = sum(len(c) for c, _ in items)
        fill = max(0, -(-(total - 1000 * len(items)) // 3000)) + 20
        items = items + [(_random_codes(rng, 1000), [[0, 999]]) for _ in range(fill)]
    b = _batch(items)
    ref = _reference(b, k, (eb,))[eb]
    assert ref["n_overflow"][:len(want)].tolist() == want
    if k <= 6:
        assert b["seq_off"][-1] // (len(b["seq_off"]) - 1) <= 4096
    _, got = _count(ctx, b, k, eb)
    # k >= 8, u16: the oracle's two-pass fp64 sum over 4^k bins with one bin at 65 535 loses ~1e-12 relative to
    # cancellation (the device's integer identity is exact up to the final rounding)
    _check(got, ref, "threshold k=%d eb=%d" % (k, eb), sd_tol=1e-12 if k < 8 else 1e-9)


@pytest.mark.parametrize("eb,inits", [(1, (254, 255)), (2, (65534, 65535))])
@pytest.mark.parametrize("k", [2, 6, 8])
def test_kmer_table_increment_at_max_init(ctx, k, eb, inits):
    rng = np.random.default_rng(k + eb)
    codes = np.concatenate([_random_codes(rng, 150), np.zeros(40, np.int8), _random_codes(rng, 110)])
    tmax = TMAX[eb]
    for init in inits:
        for first, last in ((0, 300 - k), (3, 3), (150, 150 + 39 - k + 1), (151, 151), (17, 200)):
            vals, ret = ctx.kmer_table_increment(codes, first, last, k, eb, init)
            want = np.full(4 ** k, init, dtype=np.int64)
            wret = 0
            for p in range(first, last + 1):
                h = 0
                for t in range(k):
                    h = h * 4 + int(codes[p + t])
                if want[h] < tmax:
                    want[h] += 1
                else:
                    wret = -1
            assert np.array_equal(vals.astype(np.int64), want), (k, eb, init, first, last)
            assert ret == wret, (k, eb, init, first, last)


# ---------------------------------------------------------------------------------------------------------------------
# 5. the same histograms through other entry points
# ---------------------------------------------------------------------------------------------------------------------
def test_count_into_across_route_switches(ctx):
    """one set refilled by count_kmers_into from batches that switch route: warp -> CTA -> warp"""
    rng = np.random.default_rng(55)
    short1 = _encode([_text(rng, int(rng.integers(100, 1500))) for _ in range(64)])
    long_ = _encode([_text(rng, int(rng.integers(5000, 9000))) if i % 3 else b"A" * 6000 for i in range(64)])
    short2 = _encode(_mixed_texts(64, seed=56))
    for eb in (1, 2):
        dst = None
        for tag, b in (("warp", short1), ("cta", long_), ("warp again", short2)):
            sq = _upload(ctx, b)
            if dst is None:
                dst = ctx.count_kmers(sq, 5, eb)
            else:
                ctx.count_kmers_into(sq, dst)
            fresh = ctx.count_kmers(sq, 5, eb)
            _same(_device(dst), _device(fresh), "count_into %s eb=%d" % (tag, eb))
            assert dst.largest_count() == fresh.largest_count()
        _check(_device(dst), _reference(short2, 5, (eb,))[eb], "count_into final eb=%d" % eb)


def test_count_into_rows_then_refresh(ctx):
    rng = np.random.default_rng(77)
    a = _encode(_mixed_texts(300, seed=78))
    b = _encode([_text(rng, int(rng.integers(4000, 12000))) for _ in range(9)])
    for eb in (1, 2):
        h = ctx.hset_alloc(3 + 300 + 4 + 9 + 2, 5, eb)
        ctx.count_kmers_into_rows(_upload(ctx, a), h, 3)
        ctx.count_kmers_into_rows(_upload(ctx, b), h, 307)
        h.refresh()
        for first, src in ((3, a), (307, b)):
            n = len(src["seq_off"]) - 1
            _same(_device(h, first, n), _device(ctx.count_kmers(_upload(ctx, src), 5, eb)), "rows at %d eb=%d" % (first, eb))
        for first, n in ((0, 3), (303, 4), (316, 2)):
            rest = _device(h, first, n)
            assert not rest["hist"].any() and not rest["sum"].any() and not rest["sumsq"].any()


def test_seqs_from_text_matches_upload(ctx, mixed):
    texts = mixed[0]
    sub = list(range(0, len(texts), 7))
    tx = [texts[i] for i in sub]
    bb = _encode(tx)
    for k, eb in ((5, 1), (6, 2), (3, 4)):
        _same(_device(ctx.count_kmers(ctx.seqs_from_text(tx), k, eb)), _device(ctx.count_kmers(_upload(ctx, bb), k, eb)),
              "seqs_from_text k=%d eb=%d" % (k, eb))


@pytest.mark.parametrize("k,eb", [(5, 1), (6, 2), (3, 2)])
def test_legacy_count_kernel_matches(ctx, mixed, monkeypatch, k, eb):
    """MC2_K1_LEGACY=1 puts count_kernel in place of count_warp_kernel (read on every call)"""
    sq = _upload(ctx, mixed[1])
    plain = _device(ctx.count_kmers(sq, k, eb))
    monkeypatch.setenv("MC2_K1_LEGACY", "1")
    legacy = _device(ctx.count_kmers(sq, k, eb))
    monkeypatch.delenv("MC2_K1_LEGACY")
    _same(legacy, plain, "legacy k=%d eb=%d" % (k, eb))


# ---------------------------------------------------------------------------------------------------------------------
# 6. width detection at the exact limits
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("largest,width", [(255, 1), (256, 2), (65535, 2), (65536, 4)])
def test_auto_width_at_the_limits(ctx, largest, width):
    """Largest count = 1 + the largest multiplicity: a poly-A of largest + 3 bases at k = 5"""
    rng = np.random.default_rng(largest)
    texts = [_text(rng, int(rng.integers(300, 1200))) for _ in range(50)]
    texts.insert(17, b"A" * (largest + 3))
    b = _encode(texts)
    hs, got_largest, eb = ctx.count_kmers_auto(_upload(ctx, b), 5)
    assert (got_largest, eb, hs.elem_bytes, hs.largest_count()) == (largest, width, width, largest)
    _check(_device(hs), _reference(b, 5, (eb,))[eb], "auto %d" % largest)
