"""CPU, world_size 2, gloo: all_pairs_step(..., identity=(model, t)) -- the identity search sharded over ranks by the same
row ranges and gathers as the classifier sweep -- equals the same step in one process.  The engine is a stand-in built
on the oracle (predicted identity = Predictor<T>::similarity, the GLM sum clamped to [0, 1])."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as tdist
import torch.multiprocessing as mp

from conftest import weights_text
from meshclust2_b200 import dist as mdist
from meshclust2_b200 import synth
from oracle import port

T = 0.45


class IdentityEngine:
    """K1 and the identity sweep through the oracle"""

    def __init__(self, seqs, per):
        self.seqs, self.per = seqs, per
        self.device = torch.device("cpu")

    def count(self):
        pts = [port.get_point(s, 5, 1) for s in self.seqs]
        self.H = np.stack([p["hist"] for p in pts]) if pts else np.zeros((0, 1024), dtype=np.uint8)
        self.ln = np.array([p["len"] for p in pts], dtype=np.int64)
        self.mag = np.array([p["mag"] for p in pts], dtype=np.int64)

    def use_local_as_full(self):
        self.full = (self.H, self.ln, self.mag)

    def export_local(self):
        bins = torch.ones((self.per, 1024), dtype=torch.uint8)
        ln = torch.zeros((self.per,), dtype=torch.int64)
        mag = torch.zeros((self.per,), dtype=torch.int64)
        n = len(self.seqs)
        bins[:n] = torch.from_numpy(self.H)
        ln[:n] = torch.from_numpy(self.ln)
        mag[:n] = torch.from_numpy(self.mag)
        return bins, ln, mag

    def install_full(self, bins, length, mag, n_total):
        assert bins.shape[0] == n_total
        self.full = (bins.numpy(), length.numpy(), mag.numpy())

    def sweep(self, q0, q1, upper_only, cutoff, max_out, identity=None):
        model, t = identity
        H, ln, mag = self.full
        q, d, s = [], [], []
        for r in range(q0, q1):
            lo, hi = int(float(ln[r]) * cutoff), int(float(ln[r]) / cutoff)
            for c in range(r + 1 if upper_only else 0, H.shape[0]):
                if lo <= ln[c] <= hi:
                    v = port.predict_pair(model, H[c], H[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                    q.append(r), d.append(c), s.append(v)
        s = np.array(s)
        keep = s >= t
        return int(keep.sum()), len(s), (np.array(q, dtype=np.uint64)[keep], np.array(d, dtype=np.uint64)[keep], s[keep])


def _model():
    m = port.Model.from_text(weights_text("weights_cfg1_id90"))
    m.weights[0] = 0.0          # without the intercept the sums of this set spread over about [0.1, 3]
    return m


def _worker(rank, world, port_no, n_total, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_no)
    tdist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        per, bounds = mdist.shard_bounds(n_total, world)
        lo, hi = bounds[rank]
        seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31, lo=lo, hi=hi)
        eng = IdentityEngine(seqs, per)
        res = mdist.all_pairs_step(eng, mdist.Comm(tdist), torch, n_total, 0.9, upper_only=True, blocks_per_rank=2,
                                   identity=(_model(), T))
        surv = res["survivors"]
        gathered = [None] * world
        tdist.all_gather_object(gathered, list(zip(map(tuple, surv.tolist()), surv.scores().tolist())))
        if rank == 0:
            out.put((res["n_scored"], res["n_close"], sorted(sum(gathered, []))))
    finally:
        tdist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.timeout(300)
def test_two_ranks_identity_step_equals_one_rank():
    n_total = 61      # odd: the tail shard is padded for the all-gather
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    pno = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, pno, n_total, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    seqs, _ = synth.make_range(n_total, 1000, 9, 0.1, seed=31)
    eng = IdentityEngine(seqs, n_total)
    res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n_total, 0.9, upper_only=True, blocks_per_rank=2,
                               identity=(_model(), T))
    surv = res["survivors"]
    want = (res["n_scored"], res["n_close"], sorted(zip(map(tuple, surv.tolist()), surv.scores().tolist())))
    assert got == want
    assert 0 < want[1] < want[0]
    assert any(0 < s < 1 for _, s in want[2])
