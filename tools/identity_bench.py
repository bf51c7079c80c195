"""Identity search (mc2_identity_pairs) on the cfg3 shape: 100 k x 1 kb, k = 5, uint8, upper triangle, cutoff 0.9.

Times, with CUDA events and the L2 overwritten before every timed step (the 100 MB set otherwise sits in the 126 MB L2):
  - the identity sweep of the regression model of tests/test_integrated_fastcar.py (normalized vectors, Euclidean, EMD^2)
    at t = the smallest positive double (fastcar's `sim > 0`), 0.5 and 0.9, with survivor counts;
  - the classifier sweep (mc2_all_pairs) of weights_cfg1_id90 on the same set, the reference point;
  - the identity sweep at t = 0.9 on the first 20 k rows, on the tile form and forced onto the row-streaming form
    (MC2_SWEEP_LEGACY=1, read per call).
Prints one JSON line, with the card name, power limit and maximum SM clock read by nvidia-smi in the same run.

    python tools/identity_bench.py [--warmup 5] [--steps 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from meshclust2_b200 import capi, synth  # noqa: E402
from test_integrated_fastcar import REGRESSION_SECTION  # noqa: E402

WEIGHTS = os.path.join(ROOT, "tests", "golden", "weights_cfg1_id90.txt")
MAX_OUT = 1 << 24       # survivors written per call; n_out still counts them all
CUTOFF = 0.9


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, power, clock = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def timed(ctx, call, warmup, steps):
    """ms per step (mean, min, max) of call() with the L2 overwritten before each step; call() returns (n_out, n_scored)"""
    for _ in range(warmup):
        ctx.flush_l2(256 << 20)
        res = call()
    ms = []
    for _ in range(steps):
        ctx.flush_l2(256 << 20)
        ctx.sync()
        ctx.timer_start()
        res = call()
        ms.append(ctx.timer_stop())
    n_out, n_scored = res
    mean = float(np.mean(ms))
    return dict(ms_per_step=round(mean, 3), ms_min=round(min(ms), 3), ms_max=round(max(ms), 3), n_out=int(n_out),
                n_scored=int(n_scored), pairs_per_s=float("%.4g" % (n_scored / (mean * 1e-3))),
                survivor_fraction=float("%.4g" % (n_out / max(1, n_scored))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--n", type=int, default=None, help="rows (default: cfg3's 100 k)")
    ap.add_argument("--subset", type=int, default=20000, help="rows of the row-streaming comparison")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if a.steps < 10:
        ap.error("--steps must be >= 10")
    info = gpu_info()
    seqs, _, k, eb = synth.make_config("cfg3", n=a.n)
    n = len(seqs)
    ctx = capi.Context(0)
    enc = capi.encode_batch(seqs)
    sq = ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"])
    hs = ctx.count_kmers(sq, k, eb)
    with tempfile.TemporaryDirectory() as tmp:
        w3 = os.path.join(tmp, "w3.txt")
        with open(w3, "w") as f:
            f.write(open(WEIGHTS).read().replace("mode: 1", "mode: 3").rstrip("\n") + "\n\n" + REGRESSION_SECTION)
        reg = ctx.model_from_file(w3, which=1)
    cls = ctx.model_from_file(WEIGHTS)
    bufs = (np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT, dtype=np.uint64), np.zeros(MAX_OUT))
    for b in bufs:
        capi.host_register(b)

    def ident(t, rows=None):
        rng = (0, rows) if rows else None

        def call():
            r = ctx.identity_pairs(reg, hs, hs, t, CUTOFF, q_range=rng, d_range=rng, upper_only=True, max_out=MAX_OUT, out=bufs)
            return r["n_out"], r["n_scored"]
        return call

    def classifier():
        r = ctx.all_pairs(cls, hs, hs, CUTOFF, upper_only=True, max_out=MAX_OUT, out=bufs)
        return r["n_out"], r["n_scored"]

    out = dict(tool="identity_bench", shape="cfg3: %d x 1 kb, k=%d, uint%d, upper triangle, cutoff %.1f, L2 flushed per step"
               % (n, k, 8 * eb, CUTOFF), gpu=info, warmup=a.warmup, steps=a.steps, max_out=MAX_OUT)
    tiny = float(np.nextafter(0.0, 1.0))
    out["classifier_cfg1_id90"] = timed(ctx, classifier, a.warmup, a.steps)
    out["identity"] = {}
    for name, t in (("t_min_positive", tiny), ("t_0.5", 0.5), ("t_0.9", 0.9)):
        out["identity"][name] = dict(min_identity=t, **timed(ctx, ident(t), a.warmup, a.steps))
    sub = min(a.subset, n)
    out["subset_rows"] = sub
    out["subset_identity_t_0.9_tile"] = timed(ctx, ident(0.9, sub), a.warmup, a.steps)
    os.environ["MC2_SWEEP_LEGACY"] = "1"
    try:
        out["subset_identity_t_0.9_row_streaming"] = timed(ctx, ident(0.9, sub), a.warmup, a.steps)
    finally:
        os.environ.pop("MC2_SWEEP_LEGACY", None)
    c, i9 = out["classifier_cfg1_id90"]["ms_per_step"], out["identity"]["t_0.9"]["ms_per_step"]
    out["identity_t_0.9_over_classifier"] = round(i9 / c, 4)
    for b in bufs:
        capi.host_unregister(b)
    ctx.close()
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
