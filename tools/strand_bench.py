"""Both-strand identity search (mc2_identity_pairs_both_strands) on the cfg3 shape: 100 k x 1 kb, k = 5, uint8, upper
triangle, cutoff 0.9, the regression model of tests/test_integrated_fastcar.py.

Times, with CUDA events and the L2 overwritten before every timed call (the 100 MB set otherwise sits in the 126 MB L2):
  - one-strand (mc2_identity_pairs) against both-strand search at t = 0.9 and t = 0.5, with the survivors of the forward
    strand, of the reverse strand alone (the reverse-complement set as the query set) and of the union;
  - the reverse-complement kernel (revcomp_kernel, from torch.profiler CUDA activity) on cfg3's 100 MB set and on cfg4's
    shape (5 000 x 65 536 uint16 bins, 655 MB), as GB/s (bytes read + written) against the HBM bandwidth of a 1 GiB
    device-to-device copy measured in the same run.
Prints one JSON line, with the card name, power limit and maximum SM clock read by nvidia-smi in the same run.

    python tools/strand_bench.py [--warmup 5] [--steps 10] [--out FILE]
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


def hbm_copy_gbs(torch, reps=20):
    """bytes read + written per second of a 1 GiB device-to-device copy"""
    a = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del a, b
    return 2 * (1 << 30) / (ms * 1e-3) / 1e9


def revcomp_kernel_ms(torch, hs, warmup, steps):
    """mean duration of revcomp_kernel over `steps` calls of reverse_complement() (allocation of the new set excluded)"""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(warmup):
        hs.reverse_complement().free()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            hs.reverse_complement().free()
        torch.cuda.synchronize()
    us = [e.time_range.elapsed_us() for e in prof.events() if "revcomp_kernel" in e.name]
    if len(us) != steps:
        raise RuntimeError("expected %d revcomp_kernel launches in the trace, found %d" % (steps, len(us)))
    return float(np.mean(us)) / 1e3


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
    bufs = (np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT))
    strand = np.zeros(MAX_OUT, dtype=np.int8)
    for b in bufs + (strand,):
        capi.host_register(b)
    hr = hs.reverse_complement()

    def one(t, query=hs):
        def call():
            r = ctx.identity_pairs(reg, query, hs, t, CUTOFF, upper_only=True, max_out=MAX_OUT, out=bufs)
            return r["n_out"], r["n_scored"]
        return call

    def both(t):
        def call():
            r = ctx.identity_pairs_both_strands(reg, hs, hs, t, CUTOFF, upper_only=True, max_out=MAX_OUT, out=bufs + (strand,))
            return r["n_out"], r["n_scored"]
        return call

    out = dict(tool="strand_bench", shape="cfg3: %d x 1 kb, k=%d, uint%d, upper triangle, cutoff %.1f, L2 flushed per call"
               % (n, k, 8 * eb, CUTOFF), gpu=info, warmup=a.warmup, steps=a.steps, max_out=MAX_OUT)
    for t in (0.9, 0.5):
        o = timed(ctx, one(t), a.warmup, a.steps)
        b = timed(ctx, both(t), a.warmup, a.steps)
        sweep = ctx.last_sweep()
        rev_only = one(t, hr)()[0]
        out["t_%g" % t] = dict(one_strand=o, both_strands=b, survivors_forward=o["n_out"], survivors_reverse=int(rev_only),
                               survivors_union=b["n_out"], both_over_one=round(b["ms_per_step"] / o["ms_per_step"], 4),
                               both_n_exact=sweep["n_exact"], both_coarse=sweep["coarse"])
    peak = hbm_copy_gbs(torch)
    out["hbm_copy_GBps"] = round(peak, 1)
    rc = {}
    for name, h in (("cfg3", hs), ("cfg4", None)):
        if h is None:
            h = ctx.hset_alloc(5000, 8, 2)
        ms = revcomp_kernel_ms(torch, h, a.warmup, a.steps)
        nbytes = 2 * len(h) * 4 ** h.k * h.elem_bytes
        gbs = nbytes / (ms * 1e-3) / 1e9
        rc[name] = dict(rows=len(h), k=h.k, elem_bytes=h.elem_bytes, kernel_ms=round(ms, 4), GBps=round(gbs, 1),
                        of_hbm_copy=round(gbs / peak, 3))
        if name == "cfg4":
            h.free()
    out["reverse_complement"] = rc
    for b in bufs + (strand,):
        capi.host_unregister(b)
    hr.free()
    hs.free()
    ctx.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
