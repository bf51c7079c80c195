#!/usr/bin/env python3
"""Multi-rank check of the sharded greedy clustering on real GPUs: all_pairs_step(..., greedy=True) (every rank sweeps an
equal-cost share of each query-row block, the part slots are all-gathered over NCCL and every rank adds the block) must
equal, on every rank, mc2_identity_greedy_clusters over the gathered set on that rank: rep, the bits of identity, strand,
n_clusters and n_scored.  At t = 0.9, 0.5 and the smallest positive double (most pairs are edges: several blocks), on one
and on both strands.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
      tests/multi_gpu_greedy_check.py [--n-seqs 3000]
  python tests/multi_gpu_greedy_check.py            # world size 1, same code path without a process group

Prints " OK " and exits 0 only if every rank agrees."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-seqs", type=int, default=3000)
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    import torch
    from helpers import to_desc
    from meshclust2_b200 import capi, dist as mdist, synth
    from oracle import port
    tdist = None
    if world > 1:
        import torch.distributed as td
        torch.cuda.set_device(local_rank)
        td.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        tdist = td
    comm = mdist.Comm(tdist)
    n_total = args.n_seqs
    k, eb, cutoff = 5, 1, 0.9
    per, bounds = mdist.shard_bounds(n_total, world)
    lo, hi = bounds[rank]
    seqs, _ = synth.make_range(n_total, 1000, 40, 0.1, seed=4242, lo=lo, hi=hi)
    ctx = capi.Context(local_rank)
    om = port.Model.from_text(open(os.path.join(ROOT, "tests", "golden", "weights_cfg1_id90.txt")).read())
    om.weights[0] = 0.0         # without the intercept the identities of this set spread over about [0.1, 3]
    model = ctx.model(to_desc(capi, om, regression=1))
    eng = mdist.GpuEngine(capi, ctx, torch, model, k, eb, local_rank)
    enc = capi.encode_batch(seqs)
    eng.set_local_sequences(ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"]), hi - lo, per)

    bad = 0
    notes = []
    for t in (0.9, 0.5, float(np.nextafter(0.0, 1.0))):
        for both in (False, True):
            res = mdist.all_pairs_step(eng, comm, torch, n_total, cutoff, identity=(model, t, both), greedy=True)
            got = res["greedy"]
            want = ctx.identity_greedy_clusters(model, eng.full, t, cutoff, both_strands=both, range=(0, n_total))
            same = (np.array_equal(got["rep"], want["rep"])
                    and np.array_equal(got["identity"].view(np.uint64), want["identity"].view(np.uint64))
                    and np.array_equal(got["strand"], want["strand"]) and got["n_clusters"] == want["n_clusters"]
                    and res["n_scored"] == want["n_scored"])
            if not same:
                bad += 1
                print("[rank %d] t=%r both=%d MISMATCH: %d vs %d clusters, scored %d vs %d" % (
                    rank, t, both, got["n_clusters"], want["n_clusters"], res["n_scored"], want["n_scored"]), flush=True)
            notes.append("t=%.3g%s: %d clusters, %d edges, %d blocks" % (t, " both" if both else "", got["n_clusters"],
                                                                       res["n_close"], len(res["blocks"])))
    tot_bad = comm.all_reduce_sum([bad], torch, eng.device)[0]
    if rank == 0:
        print("multi_gpu_greedy_check world=%d n=%d: %s (%s)" % (world, n_total, "OK" if tot_bad == 0 else "FAILED",
                                                                 "; ".join(notes)), flush=True)
    if tdist is not None:
        tdist.destroy_process_group()
    sys.exit(0 if tot_bad == 0 else 1)


if __name__ == "__main__":
    main()
