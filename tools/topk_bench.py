"""Top-K identity search (mc2_identity_topk) against the flat survivor list (mc2_identity_pairs) on the cfg3 shape:
100 k x 1 kb, k = 5, uint8, cutoff 0.9, the regression model of tests/test_integrated_fastcar.py (tools/identity_bench.py).

Two shapes: the upper triangle, and the full square with exclude_self (a neighbour table without the self hit; the flat
list of that square keeps the self pairs, which add one survivor per row).  For t = 0.9 and 0.5, identity_pairs once and
identity_topk for K = 1, 10 and 100, with CUDA events and the L2 overwritten before every timed call (the 100 MB set
otherwise sits in the 126 MB L2); every output goes to page-locked host buffers.  Then, in a separate profiled call per
configuration (torch.profiler CUDA activity), the device time of the selection kernels (topk_count / topk_scatter /
seg_scan / topk_select) and the number of sweep launches (block sweeps).
Prints one JSON line, with the card name, power limit and maximum SM clock read by nvidia-smi in the same run.

    python tools/topk_bench.py [--warmup 5] [--steps 10] [--n N] [--out FILE]
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

from identity_bench import CUTOFF, MAX_OUT, WEIGHTS, gpu_info, timed  # noqa: E402
from meshclust2_b200 import capi, synth  # noqa: E402
from test_integrated_fastcar import REGRESSION_SECTION  # noqa: E402

KS = (1, 10, 100)
SELECT_KERNELS = ("topk_count_kernel", "topk_scatter_kernel", "seg_scan_kernel", "topk_select_kernel")


def profile_call(torch, call):
    """(selection kernels' device ms, sweep launches) of one call"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    sel_us, sweeps = 0.0, 0
    for e in prof.events():
        if any(k in e.name for k in SELECT_KERNELS):
            sel_us += e.time_range.elapsed_us()
        elif "sweep" in e.name and "kernel" in e.name:      # tile_sweep_kernel or a row-streaming sweep_*kernel
            sweeps += 1
    return sel_us / 1e3, sweeps


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
    pinned = [np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT)]
    tables = {K: (np.zeros((n, K), dtype=np.uint64), np.zeros((n, K)), np.zeros(n, dtype=np.uint32),
                  np.zeros(n, dtype=np.uint64)) for K in KS}
    for K in KS:
        pinned += list(tables[K])
    for b in pinned:
        capi.host_register(b)
    flat = tuple(pinned[:3])

    def pairs_call(t, upper):
        def call():
            r = ctx.identity_pairs(reg, hs, hs, t, CUTOFF, upper_only=upper, max_out=MAX_OUT, out=flat)
            return r["n_out"], r["n_scored"]
        return call

    def topk_call(t, K, upper):
        def call():
            r = ctx.identity_topk(reg, hs, hs, t, K, CUTOFF, upper_only=upper, exclude_self=not upper, out=tables[K])
            return int(r["n_hits"].sum()), r["n_scored"]
        return call

    out = dict(tool="topk_bench", shape="cfg3: %d x 1 kb, k=%d, uint%d, cutoff %.1f, L2 flushed per call" % (n, k, 8 * eb, CUTOFF),
               gpu=info, warmup=a.warmup, steps=a.steps, max_out=MAX_OUT, scratch_pairs=max(n, 1 << 22))
    for shape, upper in (("upper_triangle", True), ("square_exclude_self", False)):
        res = {}
        for t in (0.9, 0.5):
            base = timed(ctx, pairs_call(t, upper), a.warmup, a.steps)
            row = dict(identity_pairs=base)
            for K in KS:
                tk = timed(ctx, topk_call(t, K, upper), a.warmup, a.steps)
                sweep = ctx.last_sweep()
                sel_ms, sweeps = profile_call(torch, topk_call(t, K, upper))
                tk.update(hits=tk.pop("n_out"), kept=int(np.minimum(tables[K][3], K).sum()),
                          over_identity_pairs=round(tk["ms_per_step"] / base["ms_per_step"], 4),
                          selection_kernels_ms=round(sel_ms, 3), block_sweeps=sweeps, n_exact=sweep["n_exact"],
                          coarse=sweep["coarse"])
                tk.pop("survivor_fraction", None)
                row["K_%d" % K] = tk
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
