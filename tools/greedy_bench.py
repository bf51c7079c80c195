"""Greedy representative clustering (mc2_identity_greedy_clusters) against the flat survivor lists a user would otherwise copy
to the host (mc2_identity_pairs, mc2_identity_pairs_both_strands) and the single-linkage call (mc2_identity_components), on
the cfg3 shape: 100 k x 1 kb, k = 5, uint8, cutoff 0.9, upper triangle, the regression model of
tests/test_integrated_fastcar.py (tools/identity_bench.py).

For t = 0.9 and 0.5, on one strand and on both: the flat list (max_out 2^24, page-locked outputs), the components call and
the greedy call, alternating in one session with CUDA events and the L2 overwritten before every timed call (the 100 MB set
otherwise sits in the 126 MB L2).  Then, in a separate profiled call per configuration (torch.profiler CUDA activity), the
device time of the greedy call's bucket (count + scatter), resolve and assign kernels and the number of sweep launches.
Prints one JSON line, with the card name, power limit and maximum SM clock read by nvidia-smi in the same run.

    python tools/greedy_bench.py [--warmup 5] [--steps 10] [--n N] [--out FILE]
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

GROUPS = dict(bucket=("topk_count_kernel", "topk_scatter_kernel"), resolve=("greedy_resolve_kernel",),
              assign=("greedy_assign_kernel",), init_finish=("greedy_init_kernel", "greedy_finish_kernel"))


def profile_call(torch, call):
    """(device ms per kernel group, sweep launches) of one call"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    us = {g: 0.0 for g in GROUPS}
    sweeps = 0
    for e in prof.events():
        for g, names in GROUPS.items():
            if any(k in e.name for k in names):
                us[g] += e.time_range.elapsed_us()
        if "sweep" in e.name and "kernel" in e.name:        # tile_sweep_kernel or a row-streaming sweep_*kernel
            sweeps += 1
    return {g + "_ms": round(v / 1e3, 3) for g, v in us.items()}, sweeps


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
    pinned = [np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT),
              np.zeros(MAX_OUT, dtype=np.int8)]
    for b in pinned:
        capi.host_register(b)

    def flat_call(t, both):
        def call():
            if both:
                r = ctx.identity_pairs_both_strands(reg, hs, hs, t, CUTOFF, upper_only=True, max_out=MAX_OUT, out=tuple(pinned))
            else:
                r = ctx.identity_pairs(reg, hs, hs, t, CUTOFF, upper_only=True, max_out=MAX_OUT, out=tuple(pinned[:3]))
            return r["n_out"], r["n_scored"]
        return call

    def comp_call(t, both):
        def call():
            r = ctx.identity_components(reg, hs, t, CUTOFF, both_strands=both)
            return r["n_components"], r["n_scored"]
        return call

    def greedy_call(t, both):
        def call():
            r = ctx.identity_greedy_clusters(reg, hs, t, CUTOFF, both_strands=both)
            return r["n_clusters"], r["n_scored"]
        return call

    out = dict(tool="greedy_bench", shape="cfg3: %d x 1 kb, k=%d, uint%d, upper triangle, cutoff %.1f, L2 flushed per call"
               % (n, k, 8 * eb, CUTOFF), gpu=info, warmup=a.warmup, steps=a.steps, max_out=MAX_OUT,
               scratch_pairs_per_strand=max(n, 1 << 24))

    def merge(rs):
        ms = [r["ms_per_step"] for r in rs]
        d = dict(rs[-1])
        d.update(ms_per_step=round(float(np.mean(ms)), 3), ms_min=min(r["ms_min"] for r in rs), ms_max=max(r["ms_max"] for r in rs))
        d.pop("pairs_per_s", None)
        d.pop("survivor_fraction", None)
        return d

    for t in (0.9, 0.5):
        row = {}
        for both in (False, True):
            tag = "both_strands" if both else "one_strand"
            # alternate the three calls so that drift on the shared host hits them alike
            fl, cc, gr = [], [], []
            for _ in range(2):
                fl.append(timed(ctx, flat_call(t, both), a.warmup, a.steps // 2))
                cc.append(timed(ctx, comp_call(t, both), a.warmup, a.steps // 2))
                gr.append(timed(ctx, greedy_call(t, both), a.warmup, a.steps // 2))
            sweep = ctx.last_sweep()
            f, c, g = merge(fl), merge(cc), merge(gr)
            f["survivors"] = f.pop("n_out")
            c["n_components"] = c.pop("n_out")
            g["n_clusters"] = g.pop("n_out")
            c["over_flat"] = round(c["ms_per_step"] / f["ms_per_step"], 4)
            kern, sweeps = profile_call(torch, greedy_call(t, both))
            g.update(over_flat=round(g["ms_per_step"] / f["ms_per_step"], 4),
                     over_components=round(g["ms_per_step"] / c["ms_per_step"], 4), sweeps=sweeps, n_exact=sweep["n_exact"],
                     coarse=sweep["coarse"], **kern)
            row["flat_" + tag] = f
            row["components_" + tag] = c
            row["greedy_" + tag] = g
        out["t_%g" % t] = row
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
