"""Sharded greedy clustering (dist.all_pairs_step(..., greedy=True)) on the cfg3 shape: 100 k x 1 kb, k = 5, uint8, cutoff
0.9, upper triangle, the regression model of the identity benches (tools/identity_bench.py), t = 0.9 and 0.5, one and
both strands.  Run under torch.distributed.run with one process per GPU (or plain python for one GPU):

    python -m torch.distributed.run --nproc-per-node N tools/greedy_dist_bench.py [--warmup 2] [--steps 4] [--out FILE]

Every rank counts the whole set itself, so only the clustering is timed.  Per configuration, alternating in one session
with the L2 overwritten before every timed call (the 100 MB set otherwise sits in the 126 MB L2):
  - at world 1: the staged loop (the block loop of all_pairs_step(greedy=True)) and the single call
    mc2_identity_greedy_clusters;
  - at every world: the greedy loop and the components form (each rank labels its triangle_row_blocks share, the labels
    are all-gathered and joined, as all_pairs_step(components=True) does).
Phases of the greedy loop, summed over its blocks: begin (the object's allocation), the sweep, the count gather, the edge
gather, add_block and end (outputs and release), max over ranks, host clocks around calls that end in a device
synchronise.  --cfg5 adds a 10^6 x 1 kb set at t = 0.9 on one strand.  Rank 0 prints
one JSON line with the card name, power limit and maximum SM clock read by nvidia-smi in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from identity_bench import CUTOFF, WEIGHTS, gpu_info  # noqa: E402
from meshclust2_b200 import capi, dist as mdist, synth  # noqa: E402
from test_integrated_fastcar import REGRESSION_SECTION  # noqa: E402


class Timed:
    """an engine / comm wrapper that adds the host time of each named call (each ends in a device synchronise) to `ms`"""

    def __init__(self, inner, ms, names):
        self._inner, self._ms, self._names = inner, ms, names

    def __getattr__(self, name):
        f = getattr(self._inner, name)
        if name not in self._names or not callable(f):
            return f
        tag = self._names[name]

        def call(*a, **kw):
            t0 = time.perf_counter()
            r = f(*a, **kw)
            self._ms[tag] = self._ms.get(tag, 0.0) + (time.perf_counter() - t0) * 1e3
            return r
        return call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--n", type=int, default=None, help="rows of the cfg3 shape (default 100 k)")
    ap.add_argument("--cfg5", action="store_true", help="also the 10^6-row set")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    import tempfile

    import torch
    tdist = None
    if world > 1:
        import torch.distributed as td
        torch.cuda.set_device(local_rank)
        td.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        tdist = td
    comm = mdist.Comm(tdist)
    ctx = capi.Context(local_rank)
    with tempfile.TemporaryDirectory() as tmp:
        w3 = os.path.join(tmp, "w3.txt")
        with open(w3, "w") as f:
            f.write(open(WEIGHTS).read().replace("mode: 1", "mode: 3").rstrip("\n") + "\n\n" + REGRESSION_SECTION)
        reg = ctx.model_from_file(w3, which=1)

    def load(cfg, n=None):
        seqs, _, k, eb = synth.make_config(cfg, n=n)
        enc = capi.encode_batch(seqs)
        hs = ctx.count_kmers(ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"]), k, eb)
        eng = mdist.GpuEngine(capi, ctx, torch, reg, k, eb, local_rank)
        eng.full, eng.n_total = hs, len(seqs)
        return eng, hs, k, eb

    def barrier():
        torch.cuda.synchronize()
        comm.barrier()

    def run_timed(fn, warmup, steps):
        """ms per step over ranks (max of each step), with the L2 overwritten before each step"""
        for _ in range(warmup):
            ctx.flush_l2(256 << 20)
            barrier()
            res = fn()
        ms = []
        for _ in range(steps):
            ctx.flush_l2(256 << 20)
            barrier()
            t0 = time.perf_counter()
            res = fn()
            barrier()
            ms.append(comm.all_reduce_max((time.perf_counter() - t0) * 1e3, torch, torch.device("cuda", local_rank)))
        return dict(ms_per_step=round(float(np.mean(ms)), 3), ms_min=round(min(ms), 3), ms_max=round(max(ms), 3)), res

    def greedy_fn(eng, t, both, phases=None):
        def fn():
            ms = {}
            e = Timed(eng, ms, dict(greedy_begin="begin", greedy_sweep_part="sweep", greedy_gather="edge_gather",
                                    greedy_add_block="add_block", greedy_end="end"))
            c = Timed(comm, ms, dict(all_reduce_sum="count_gather"))
            r = mdist._greedy_blocks(e, c, torch, eng.n_total, CUTOFF, (reg, t, both))
            if phases is not None:
                phases.append((ms, len(r[1])))
            return r
        return fn

    def components_fn(eng, t, both):
        def fn():
            parts = [eng.components(q0, q1, CUTOFF, (reg, t, both)) for q0, q1 in
                     mdist.triangle_row_blocks(eng.n_total, world, rank)]
            comp = parts[0] if parts else dict(label=np.arange(eng.n_total, dtype=np.uint64))
            if tdist is not None:
                local = torch.as_tensor(np.asarray(comp["label"], dtype=np.int64), device=eng.device)
                comp = eng.merge_components(comm.all_gather_rows(local, torch).cpu().numpy().reshape(world, eng.n_total))
            return comp
        return fn

    def single_fn(eng, t, both):
        return lambda: ctx.identity_greedy_clusters(reg, eng.full, t, CUTOFF, both_strands=both)

    def phase_summary(phases, most_of):
        """per-phase ms per call: each rank's, then the max over ranks (the sweep is where the ranks wait for each other)"""
        keys = ("begin", "sweep", "count_gather", "edge_gather", "add_block", "end")
        timed_calls = phases[-a.steps:]            # the last timed calls, no warm-up
        mean = [float(np.mean([p[0].get(k, 0.0) for p in timed_calls])) for k in keys]
        top = [most_of(v) for v in mean]
        return dict({k + "_ms": round(v, 3) for k, v in zip(keys, top)}, blocks=phases[-1][1])

    dev = torch.device("cuda", local_rank)
    most_of = lambda v: comm.all_reduce_max(v, torch, dev)  # noqa: E731
    out = dict(tool="greedy_dist_bench", world=world, gpu=gpu_info() if rank == 0 else None, warmup=a.warmup, steps=a.steps,
               protocol="every rank counts the whole set; host clocks around the clustering only, max over ranks per step, "
                        "L2 overwritten before every timed call, variants alternated in one session")
    eng, hs, k, eb = load("cfg3", a.n)
    out["shape"] = "cfg3: %d x 1 kb, k=%d, uint%d, upper triangle, cutoff %.1f" % (eng.n_total, k, 8 * eb, CUTOFF)
    for t in (0.9, 0.5):
        for both in (False, True):
            tag = "t_%g_%s" % (t, "both_strands" if both else "one_strand")
            row = {}
            gr, cc, sg, phases = [], [], [], []
            for _ in range(2):
                gr.append(run_timed(greedy_fn(eng, t, both, phases), a.warmup, a.steps))
                cc.append(run_timed(components_fn(eng, t, both), a.warmup, a.steps))
                if world == 1:
                    sg.append(run_timed(single_fn(eng, t, both), a.warmup, a.steps))
            mean = lambda rs: round(float(np.mean([r[0]["ms_per_step"] for r in rs])), 3)  # noqa: E731
            res = gr[-1][1][0]
            row["greedy_ms"] = mean(gr)
            row["components_ms"] = mean(cc)
            row["greedy_over_components"] = round(row["greedy_ms"] / row["components_ms"], 4)
            row["n_clusters"] = int(res["n_clusters"])
            row["n_edges"] = int(gr[-1][1][3])
            row.update(phase_summary(phases, most_of))
            if world == 1:
                row["single_call_ms"] = mean(sg)
                row["staged_over_single"] = round(row["greedy_ms"] / row["single_call_ms"], 4)
                s = sg[-1][1]
                row["same_as_single"] = bool(np.array_equal(s["rep"], res["rep"]) and s["n_clusters"] == res["n_clusters"]
                                             and np.array_equal(s["identity"].view(np.uint64), res["identity"].view(np.uint64)))
            out[tag] = row
    hs.free()
    if a.cfg5:
        eng, hs, k, eb = load("cfg5")
        phases = []
        r, res = run_timed(greedy_fn(eng, 0.9, False, phases), 1, 2)
        out["cfg5_t_0.9_one_strand"] = dict(r, shape="cfg5: %d x 1 kb, k=%d, uint%d" % (eng.n_total, k, 8 * eb),
                                             n_clusters=int(res[0]["n_clusters"]), n_edges=int(res[3]),
                                             **phase_summary(phases, most_of))
        hs.free()
    if rank == 0:
        line = json.dumps(out)
        print(line, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(line + "\n")
    ctx.close()
    if tdist is not None:
        tdist.destroy_process_group()


if __name__ == "__main__":
    main()
