"""CPU, world_size 2, gloo: all_pairs_step(..., identity=(model, t, True)) -- the both-strand identity search sharded over
ranks -- equals the same step in one process, strands included.  The engine is a stand-in built on the oracle: each rank
reverse-complements the gathered histograms itself (bin j of the other strand is bin rc(j), big-endian base-4 k-mers) and
keeps the better strand of each pair, ties going to the forward one."""
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


class BothStrandEngine:
    """K1 and the both-strand identity sweep through the oracle"""

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
        model, t, both = identity
        assert both
        H, ln, mag = self.full
        R = np.empty_like(H)
        R[:, _rc_perm(5)] = H                   # the other strand of every gathered row, built on this rank
        q, d, s, st = [], [], [], []
        for r in range(q0, q1):
            lo, hi = int(float(ln[r]) * cutoff), int(float(ln[r]) / cutoff)
            for c in range(r + 1 if upper_only else 0, H.shape[0]):
                if lo <= ln[c] <= hi:
                    f = port.predict_pair(model, H[c], H[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                    v = port.predict_pair(model, H[c], R[r], int(mag[c]), int(mag[r]), int(ln[c]), int(ln[r]))
                    q.append(r), d.append(c), s.append(max(f, v)), st.append(1 if v > f else 0)
        s = np.array(s)
        keep = s >= t
        return int(keep.sum()), len(s), (np.array(q, dtype=np.uint64)[keep], np.array(d, dtype=np.uint64)[keep], s[keep],
                                         np.array(st, dtype=np.int8)[keep])


def _rc_perm(k):
    j = np.arange(4 ** k, dtype=np.int64)
    r = np.zeros_like(j)
    for p in range(k):
        r = r * 4 + (3 - ((j >> (2 * p)) & 3))
    return r


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
        eng = BothStrandEngine(seqs, per)
        res = mdist.all_pairs_step(eng, mdist.Comm(tdist), torch, n_total, 0.9, upper_only=True, blocks_per_rank=2,
                                   identity=(_model(), T, True))
        surv = res["survivors"]
        gathered = [None] * world
        tdist.all_gather_object(gathered, list(zip(map(tuple, surv.tolist()), surv.scores().tolist(), surv.strands().tolist())))
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
def test_two_ranks_both_strand_step_equals_one_rank():
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
    eng = BothStrandEngine(seqs, n_total)
    res = mdist.all_pairs_step(eng, mdist.Comm(None), torch, n_total, 0.9, upper_only=True, blocks_per_rank=2,
                               identity=(_model(), T, True))
    surv = res["survivors"]
    want = (res["n_scored"], res["n_close"], sorted(zip(map(tuple, surv.tolist()), surv.scores().tolist(), surv.strands().tolist())))
    assert got == want
    assert 0 < want[1] < want[0]
    assert any(0 < s < 1 for _, s, _ in want[2])
    assert {st for _, _, st in want[2]} == {0, 1}
