"""Both-strand top-K identity search (mc2_identity_topk_both_strands) against the flat both-strand list
(mc2_identity_pairs_both_strands) and the one-strand top-K (mc2_identity_topk) on the cfg3 shape: 100 k x 1 kb, k = 5,
uint8, cutoff 0.9, the regression model of tests/test_integrated_fastcar.py (tools/identity_bench.py).

Two shapes: the upper triangle, and the full square with exclude_self for both top-K calls (the flat list keeps the self
pairs).  For t = 0.9 and 0.5 and K = 1, 10 and 100, the three calls are timed alternately in the same session (one step
of each in turn, the order rotating every step), with CUDA events and the L2 overwritten before every timed call; every
output goes to page-locked host buffers.  Then, in a separate profiled call of each (torch.profiler CUDA activity), the
device time of the selection kernels (topk_count / topk_scatter / seg_scan / topk_select) and the number of sweep launches.
Prints one JSON line, with the card name, power limit and maximum SM clock read by nvidia-smi in the same run.

    python tools/strand_topk_bench.py [--warmup 5] [--steps 10] [--n N] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from identity_bench import CUTOFF, MAX_OUT, WEIGHTS, gpu_info  # noqa: E402
from meshclust2_b200 import capi, synth  # noqa: E402
from test_integrated_fastcar import REGRESSION_SECTION  # noqa: E402
from topk_bench import profile_call  # noqa: E402

KS = (1, 10, 100)


def alternated(ctx, calls, warmup, steps):
    """{name: ms per step (mean, min, max), n_out, n_scored} of each call() (returning (n_out, n_scored)), one step of each in
    turn with the order rotating every step, the L2 overwritten before each"""
    names = list(calls)
    for _ in range(warmup):
        for nm in names:
            ctx.flush_l2(256 << 20)
            calls[nm]()
    ms = {nm: [] for nm in names}
    res = {}
    for s in range(steps):
        for j in range(len(names)):
            nm = names[(s + j) % len(names)]
            ctx.flush_l2(256 << 20)
            ctx.sync()
            ctx.timer_start()
            res[nm] = calls[nm]()
            ms[nm].append(ctx.timer_stop())
    out = {}
    for nm in names:
        mean = float(np.mean(ms[nm]))
        out[nm] = dict(ms_per_step=round(mean, 3), ms_min=round(min(ms[nm]), 3), ms_max=round(max(ms[nm]), 3),
                       n_out=int(res[nm][0]), n_scored=int(res[nm][1]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--n", type=int, default=None, help="rows (default: cfg3's 100 k)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if a.steps < 10:
        ap.error("--steps must be >= 10")
    import tempfile

    import torch
    info = gpu_info()
    seqs, _, k, eb = synth.make_config("cfg3", n=a.n)
    n = len(seqs)
    ctx = capi.Context(0)
    enc = capi.encode_batch(seqs)
    hs = ctx.count_kmers(ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"]), k, eb)
    with tempfile.TemporaryDirectory() as tmp:
        w3 = os.path.join(tmp, "w3.txt")
        with open(w3, "w") as f:
            f.write(open(WEIGHTS).read().replace("mode: 1", "mode: 3").rstrip("\n") + "\n\n" + REGRESSION_SECTION)
        reg = ctx.model_from_file(w3, which=1)
    flat = (np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT),
            np.zeros(MAX_OUT, dtype=np.int8))
    one = {K: (np.zeros((n, K), dtype=np.uint64), np.zeros((n, K)), np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint64))
           for K in KS}
    both = {K: (np.zeros((n, K), dtype=np.uint64), np.zeros((n, K)), np.zeros((n, K), dtype=np.int8),
                np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint64)) for K in KS}
    pinned = list(flat) + [b for K in KS for b in one[K] + both[K]]
    for b in pinned:
        capi.host_register(b)

    def flat_call(t, upper):
        def call():
            r = ctx.identity_pairs_both_strands(reg, hs, hs, t, CUTOFF, upper_only=upper, max_out=MAX_OUT, out=flat)
            return r["n_out"], r["n_scored"]
        return call

    def one_call(t, K, upper):
        def call():
            r = ctx.identity_topk(reg, hs, hs, t, K, CUTOFF, upper_only=upper, exclude_self=not upper, out=one[K])
            return int(r["n_hits"].sum()), r["n_scored"]
        return call

    def both_call(t, K, upper):
        def call():
            r = ctx.identity_topk_both_strands(reg, hs, hs, t, K, CUTOFF, upper_only=upper, exclude_self=not upper,
                                               out=both[K])
            return int(r["n_hits"].sum()), r["n_scored"]
        return call

    out = dict(tool="strand_topk_bench",
               shape="cfg3: %d x 1 kb, k=%d, uint%d, cutoff %.1f, L2 flushed per call, calls alternated" % (n, k, 8 * eb, CUTOFF),
               gpu=info, warmup=a.warmup, steps=a.steps, max_out=MAX_OUT, scratch_pairs_per_strand=max(n, 1 << 22))
    for shape, upper in (("upper_triangle", True), ("square_exclude_self", False)):
        res = {}
        for t in (0.9, 0.5):
            row = {}
            for K in KS:
                calls = dict(flat_both_strands=flat_call(t, upper), topk_one_strand=one_call(t, K, upper),
                             topk_both_strands=both_call(t, K, upper))
                tm = alternated(ctx, calls, a.warmup, a.steps)
                both_call(t, K, upper)()
                sweep = ctx.last_sweep()
                for nm, call in calls.items():
                    sel_ms, sweeps = profile_call(torch, call)
                    tm[nm]["sweep_launches"] = sweeps
                    if nm != "flat_both_strands":
                        tm[nm]["selection_kernels_ms"] = round(sel_ms, 3)
                tb = tm["topk_both_strands"]
                tb.update(hits=tb.pop("n_out"), strand_reverse=int((both[K][2] == 1).sum()),
                          kept=int(np.minimum(both[K][4], K).sum()), n_exact=sweep["n_exact"], coarse=sweep["coarse"],
                          over_flat_both_strands=round(tb["ms_per_step"] / tm["flat_both_strands"]["ms_per_step"], 4),
                          over_topk_one_strand=round(tb["ms_per_step"] / tm["topk_one_strand"]["ms_per_step"], 4))
                tm["topk_one_strand"]["hits"] = tm["topk_one_strand"].pop("n_out")
                row["K_%d" % K] = tm
            res["t_%g" % t] = row
        out[shape] = res
    for b in pinned:
        capi.host_unregister(b)
    hs.free()
    ctx.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
