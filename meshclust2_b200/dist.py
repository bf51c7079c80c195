"""Multi-GPU plumbing for the sharded hot path: one process per GPU, torch.distributed for the exchange step.

north_star's partition (SURVEY.md section 8e): sequences are split contiguously by rank for k-mer counting (K1);
the per-rank histogram shards are ALL-GATHERED so every GPU holds the full n x 4^k set; the all-pairs sweep (K2) is
split by query-row blocks.  No floating-point value ever crosses ranks, so results are bitwise independent of the
number of GPUs.  Everything here is host logic over an `engine` object, so the same code runs under gloo on CPU in
the tests (engine = a stand-in) and under NCCL on GPUs (engine = GpuEngine over the C ABI).
"""
import numpy as np


def shard_bounds(n, world):
    """Contiguous, equal-size (padded) shards: every rank owns `per` rows, the tail ranks may own fewer real rows."""
    per = (n + world - 1) // world
    return per, [(min(r * per, n), min((r + 1) * per, n)) for r in range(world)]


def folded_row_blocks(n, world, rank, blocks_per_rank=8):
    """Query-row blocks of an upper-triangular sweep for `rank`, balanced by folding: block b and block B-1-b together
    hold a constant number of pairs, so each fold goes to one rank (cyclic over folds)."""
    B = 2 * world * blocks_per_rank
    B = min(B, max(2, n - n % 2))
    edges = np.linspace(0, n, B + 1).astype(np.int64)
    out = []
    for fold in range((B + 1) // 2):
        if fold % world != rank:
            continue
        for b in {fold, B - 1 - fold}:
            q0, q1 = int(edges[b]), int(edges[b + 1])
            if q1 > q0:
                out.append((q0, q1))
    return sorted(out)


def triangle_row_blocks(n, world, rank, blocks_per_rank=1, row_overhead=160):
    """Query-row blocks of an upper-triangular sweep for `rank`: CONTIGUOUS row ranges of equal cost (so they get longer
    towards the end of the set), `blocks_per_rank` of them per rank.  Row q costs its n - 1 - q pairs plus `row_overhead`
    pair slots: the tile kernel pays whole 64 x 256 tiles along the diagonal (about half a tile width + half a tile height
    of unused slots per query row), which would otherwise make the last rank, whose range is mostly diagonal, the slowest.
    One range per rank means one sweep launch per rank and step: every launch pays a tail of up to one tile per SM."""
    B = max(1, world * blocks_per_rank)

    def cost(x):                                    # rows [0, x)
        return x * (n - 1) - x * (x - 1) // 2 + row_overhead * x

    total = cost(n)
    edges = [0]
    for j in range(1, B):
        target = total * j // B
        lo, hi = edges[-1], n
        while lo < hi:                              # smallest x with cost(rows < x) >= target
            mid = (lo + hi) // 2
            if cost(mid) >= target:
                hi = mid
            else:
                lo = mid + 1
        edges.append(lo)
    edges.append(n)
    out = []
    for b in range(rank * blocks_per_rank, (rank + 1) * blocks_per_rank):
        q0, q1 = edges[b], edges[b + 1]
        if q1 > q0:
            out.append((q0, q1))
    return out


def rect_row_blocks(n, world, rank):
    """Query-row blocks of a rectangular (query set x database) sweep: plain contiguous split."""
    _, b = shard_bounds(n, world)
    lo, hi = b[rank]
    return [(lo, hi)] if hi > lo else []


class Survivors:
    """This rank's survivor pairs of one step, block by block, WITHOUT copying them together: an engine may hand back views
    of its own (page-locked, per-block) buffers, valid until its next step.  tolist() / array() build the [m, 2] form;
    scores() the pairs' scores in the same order, where the engine reported them; strands() the strand of each pair's
    identity (0 forward, 1 reverse) after a both-strand identity search."""

    def __init__(self):
        self.parts = []

    def add(self, pairs):
        if isinstance(pairs, tuple):
            self.parts.append(tuple(np.asarray(p) for p in pairs))
        else:
            pairs = np.asarray(pairs).reshape(-1, 2)
            self.parts.append((pairs[:, 0], pairs[:, 1]))

    def __len__(self):
        return int(sum(len(p[0]) for p in self.parts))

    def array(self):
        if not self.parts:
            return np.zeros((0, 2), dtype=np.uint64)
        return np.stack([np.concatenate([p[0] for p in self.parts]), np.concatenate([p[1] for p in self.parts])], axis=1)

    def scores(self):
        if not self.parts:
            return np.zeros(0)
        return np.concatenate([p[2] for p in self.parts])

    def strands(self):
        if not self.parts:
            return np.zeros(0, dtype=np.int8)
        return np.concatenate([p[3] for p in self.parts])

    def tolist(self):
        return self.array().tolist()


class Comm:
    """Thin wrapper so single-process runs need no process group."""

    def __init__(self, dist=None):
        self.dist = dist
        self.rank = dist.get_rank() if dist is not None else 0
        self.world = dist.get_world_size() if dist is not None else 1

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def all_gather_rows(self, local, torch):
        """local: torch tensor [per, ...] on the engine's device -> [world*per, ...] (rank-major)."""
        if self.dist is None:
            return local
        out = torch.empty((self.world * local.shape[0],) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        local = local.contiguous()
        if local.dtype in (getattr(torch, "uint16", None), getattr(torch, "uint32", None), getattr(torch, "uint64", None)):
            # NCCL has no unsigned 16 / 32 / 64-bit types: a gather moves bytes
            self.dist.all_gather_into_tensor(out.view(torch.uint8), local.view(torch.uint8))
        else:
            self.dist.all_gather_into_tensor(out, local)
        return out

    def all_reduce_sum(self, values, torch, device):
        t = torch.tensor(values, dtype=torch.int64, device=device)
        if self.dist is not None:
            self.dist.all_reduce(t)
        return [int(v) for v in t.tolist()]

    def all_reduce_max(self, value, torch, device):
        t = torch.tensor([value], dtype=torch.float64, device=device)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def all_pairs_step(engine, comm, torch, n_total, cutoff, upper_only=True, blocks_per_rank=1, max_out=1 << 20, identity=None,
                   top_k=None):
    """One pass of the hot path over a batch: local K1 -> all-gather -> row-block K2 sweep.

    identity: None sweeps with the engine's classifier; (regression model, min_identity) makes it an identity search
    (survivors = pairs whose predicted identity is >= min_identity, Survivors.scores() = those identities);
    (regression model, min_identity, True) searches both strands of each query (identity = the better strand's,
    Survivors.strands() = which strand).  Each rank reverse-complements the gathered set itself: no extra collective, and no
    floating-point value is reduced across ranks.
    top_k: with a one-strand identity search, keep each query's top_k best hits instead of the survivor list: `topk` is
    this rank's [(q0, q1, table)] with table = dict(d [q1-q0, top_k], identity [q1-q0, top_k], count, n_hits) as
    engine.topk returns it.  A query lives in exactly one block of one rank, so the tables are complete per query and
    nothing but the counters is reduced; n_close is the total hit count.

    engine.count()                  K1 over this rank's shard
    engine.export_local()           -> (bins [per, N] tensor, length [per] int64 tensor, mag [per] int64 tensor) padded
    engine.install_full(bins, length, mag, n_total)   make the gathered set the sweep's database
    engine.use_local_as_full()      single rank: the counted shard is the database (no copy, no collective)
    engine.sweep(q0, q1, upper_only, cutoff, max_out[, identity=(model, min_identity[, both_strands])])
                                    -> (n_survivors, n_scored, survivors: array [m,2], (q[m], d[m]), (q[m], d[m], score[m])
                                        or, both strands, (q[m], d[m], identity[m], strand[m]))
    engine.topk(q0, q1, upper_only, cutoff, (model, min_identity), top_k) -> (n_hits, n_scored, table)
    Returns dict(n_scored, n_close, survivors (this rank's), topk (this rank's, [] without top_k), blocks)."""
    if top_k is not None and (identity is None or (len(identity) > 2 and identity[2])):
        raise ValueError("top_k needs a one-strand identity search: identity=(regression model, min_identity)")
    if comm.world > 1 and hasattr(engine, "count_and_gather_in_place"):
        # the product engine: K1 writes this rank's rows straight into the full set, the all-gathers run in place on it
        engine.count_and_gather_in_place(comm, n_total)
    elif comm.world == 1:
        engine.count()
        engine.use_local_as_full()
    else:
        engine.count()
        bins, length, mag = engine.export_local()
        bins = comm.all_gather_rows(bins, torch)
        length = comm.all_gather_rows(length, torch)
        mag = comm.all_gather_rows(mag, torch)
        per = bins.shape[0] // comm.world
        if per * comm.world != n_total:
            # drop the padding rows of the tail shards: rows are rank-major, real rows are a prefix of each shard
            _, bounds = shard_bounds(n_total, comm.world)
            keep = np.concatenate([np.arange(r * per, r * per + (hi - lo)) for r, (lo, hi) in enumerate(bounds)])
            idx = torch.as_tensor(keep, device=bins.device)
            bins, length, mag = bins[idx].contiguous(), length[idx].contiguous(), mag[idx].contiguous()
        engine.install_full(bins, length, mag, n_total)
    blocks = (triangle_row_blocks(n_total, comm.world, comm.rank, blocks_per_rank) if upper_only
              else rect_row_blocks(n_total, comm.world, comm.rank))
    n_scored = n_close = 0
    surv = Survivors()
    tables = []
    for q0, q1 in blocks:
        if top_k is not None:
            ns, sc, table = engine.topk(q0, q1, upper_only, cutoff, identity, top_k)
            tables.append((q0, q1, table))
            n_close += ns
            n_scored += sc
            continue
        if identity is None:
            ns, sc, pairs = engine.sweep(q0, q1, upper_only, cutoff, max_out)
        else:
            ns, sc, pairs = engine.sweep(q0, q1, upper_only, cutoff, max_out, identity=identity)
        n_close += ns
        n_scored += sc
        surv.add(pairs)
    tot_scored, tot_close = comm.all_reduce_sum([n_scored, n_close], torch, engine.device)
    return dict(n_scored=tot_scored, n_close=tot_close, local_scored=n_scored, local_close=n_close, survivors=surv, topk=tables,
                blocks=blocks)


def candidate_scan(engine, comm, torch, q_global, n_total, cutoff):
    """Trainer<T>::get_close with the candidate set RANGE-PARTITIONED over ranks (SURVEY.md section 8e, third bullet;
    BASELINE configs[4] shape): the histograms stay sharded where K1 produced them, only the query row (1 KiB + side-band) is
    broadcast from its owner, every rank scans its own shard, and the (max dist, first index) pair is combined from an
    all-gather of one (dist, index, any-close) triple per rank.  Marks stay on the rank that owns the candidate.

    engine.local_query(row_local)      -> (bins[1,N], length[1], mag[1]) tensors of a local row
    engine.scan_local(bins, length, mag, cutoff) -> (best_local_pos or -1, best_dist, is_min, marks[local_n])
    Returns dict(best=global row or -1, best_dist, is_min, marks_local, shard=(lo, hi)); marks_local may be a view of a
    buffer the engine reuses: it is valid until the next scan."""
    per, bounds = shard_bounds(n_total, comm.world)
    owner = min(q_global // per, comm.world - 1) if per else 0
    lo, hi = bounds[comm.rank]
    if comm.dist is None and hasattr(engine, "scan_row"):
        # one rank: the query row already sits in the set being scanned
        best, bd, is_min, marks = engine.scan_row(q_global - lo, cutoff)
    else:
        if comm.rank == owner:
            bins, length, mag = engine.local_query(q_global - bounds[owner][0])
        else:
            bins, length, mag = engine.empty_query()
        if comm.dist is not None:
            pack = engine.query_pack() if hasattr(engine, "query_pack") else None
            if pack is not None:                    # the three tensors are views of one buffer: one broadcast
                comm.dist.broadcast(pack, src=owner)
            else:
                for t in (bins, length, mag):
                    comm.dist.broadcast(t, src=owner)
        best, bd, is_min, marks = engine.scan_local(bins, length, mag, cutoff)
    # combine: larger dist wins, ties go to the smaller global index (the sequential first maximum)
    triple = [bd if best >= 0 else -1.0, float(lo + best if best >= 0 else -1), 0.0 if is_min else 1.0]
    if comm.dist is not None:
        mine = torch.tensor(triple, dtype=torch.float64, device=engine.device)
        allv = torch.empty((comm.world * 3,), dtype=torch.float64, device=engine.device)
        comm.dist.all_gather_into_tensor(allv, mine)
        allv = allv.cpu().numpy().reshape(comm.world, 3)
    else:
        allv = np.array([triple])
    gbest, gdist = -1, -1.0
    for dist_r, idx_r, _ in allv:
        if idx_r >= 0 and (gbest < 0 or dist_r > gdist or (dist_r == gdist and idx_r < gbest)):
            gbest, gdist = int(idx_r), float(dist_r)
    return dict(best=gbest, best_dist=gdist, is_min=not bool(allv[:, 2].any()), marks_local=marks, shard=(lo, hi))


def balanced_ranges(weights, world):
    """Contiguous ranges of items for `world` ranks with about equal total weight (prefix-sum split); every item lands in
    exactly one range, ranges may be empty."""
    w = np.asarray(weights, dtype=np.float64)
    n = len(w)
    if n == 0:
        return [(0, 0)] * world
    cum = np.concatenate([[0.0], np.cumsum(w + 1.0)])      # + 1: an item costs something even with no members
    cuts = [int(np.searchsorted(cum, cum[-1] * r / world, side="left")) for r in range(world + 1)]
    cuts[0], cuts[-1] = 0, n
    cuts = np.maximum.accumulate(np.minimum(cuts, n))
    return [(int(cuts[r]), int(cuts[r + 1])) for r in range(world)]


def _gather_ranges(values, ranges, comm, torch, device, fill):
    """values: this rank's int64 results for its range -> the full array in range order on every rank."""
    total = ranges[-1][1]
    if comm.dist is None:
        return np.asarray(values, dtype=np.int64)
    width = max(1, max(hi - lo for lo, hi in ranges))
    mine = torch.full((width,), fill, dtype=torch.int64, device=device)
    if len(values):
        mine[:len(values)] = torch.as_tensor(np.asarray(values, dtype=np.int64), device=device)
    allv = torch.empty((comm.world * width,), dtype=torch.int64, device=device)
    comm.dist.all_gather_into_tensor(allv, mine)
    allv = allv.cpu().numpy().reshape(comm.world, width)
    out = np.full(total, fill, dtype=np.int64)
    for r, (lo, hi) in enumerate(ranges):
        out[lo:hi] = allv[r, :hi - lo]
    return out


def update_pass(engine, comm, torch, center_rows, center_mag, center_len, member_off, members, cutoff):
    """One pass of the update loop (ClusterFactory.cpp:639-642: mean_shift_update for every center) over the replicated point
    set, centers split over ranks by member count.  center_rows[c] = row of the point center c carries, center_mag / center_len
    = what the host center object reports (quirk Q4); members[member_off[c]:member_off[c+1]] = rows of the candidate members.

    engine.update_centers(rows, mag, length, off, members, cutoff) -> (next positions int64[m], survivors uint64[m])
    Returns (next[n_centers] position in the center's member list or -1, n_good[n_centers]) on every rank."""
    member_off = np.asarray(member_off, dtype=np.uint64)
    nc = len(center_rows)
    ranges = balanced_ranges(np.diff(member_off.astype(np.int64)), comm.world)
    lo, hi = ranges[comm.rank]
    if hi > lo:
        off = member_off[lo:hi + 1] - member_off[lo]
        nxt, ng = engine.update_centers(center_rows[lo:hi], center_mag[lo:hi], center_len[lo:hi], off,
                                        members[int(member_off[lo]):int(member_off[hi])], cutoff)
    else:
        nxt, ng = np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    nxt = _gather_ranges(nxt, ranges, comm, torch, engine.device, -1)
    ng = _gather_ranges(np.asarray(ng, dtype=np.int64), ranges, comm, torch, engine.device, 0)
    assert len(nxt) == nc
    return nxt, ng


def merge_pass(engine, comm, torch, center_rows, center_mag, center_len, delta, cutoff):
    """One call of merge() (ClusterFactory.cpp:382-401: Trainer::merge of center c against centers c+1 .. c+delta), centers
    split contiguously over ranks; a rank stages its range plus the `delta` centers after it.

    engine.merge_centers(rows, mag, length, delta, cutoff) -> chosen index per staged center (0 = none), staged-relative
    Returns out[n_centers] (global center index, 0 = none) on every rank."""
    nc = len(center_rows)
    ranges = balanced_ranges(np.ones(nc), comm.world)
    lo, hi = ranges[comm.rank]
    if hi > lo:
        end = min(nc, hi + delta)
        rel = np.asarray(engine.merge_centers(center_rows[lo:end], center_mag[lo:end], center_len[lo:end], delta, cutoff),
                         dtype=np.int64)[:hi - lo]
        mine = np.where(rel > 0, rel + lo, 0)
    else:
        mine = np.zeros(0, dtype=np.int64)
    return _gather_ranges(mine, ranges, comm, torch, engine.device, 0)


class GpuEngine:
    """The product engine: K1 / K2 through the C ABI on this rank's GPU; torch only carries device memory for NCCL."""

    def __init__(self, capi, ctx, torch, model, k, elem_bytes, device_index):
        self.capi, self.ctx, self.torch, self.model = capi, ctx, torch, model
        self.k, self.eb = k, elem_bytes
        self.N = 4 ** k
        self.device = torch.device("cuda", device_index)
        self.seqs = None       # resident packed sequences of this rank's shard
        self.per = 0           # padded shard size
        self.n_local = 0
        self.full = None
        self._dt = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[elem_bytes]

    def set_local_sequences(self, seqs_handle, n_local, per):
        self.seqs, self.n_local, self.per = seqs_handle, n_local, per

    def upload_local(self, enc):
        self.seqs = self.ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"])
        return self.seqs

    def _local(self):
        """(set, first row, rows) of this rank's shard: its own set after count(), a window of the full set after
        count_and_gather_in_place()"""
        base = getattr(self, "_local_in_full", None)
        if base is not None:
            return self.full, base, self.n_local
        return self.local_hset, 0, len(self.local_hset)

    def count(self):
        self._slot = 0          # a new step: the per-block survivor buffers are free again
        self._local_in_full = None
        # steady state: recount into the same device allocation (cudaMalloc / cudaFree stall the device)
        hs = getattr(self, "local_hset", None)
        if hs is not None and len(hs) == len(self.seqs):
            self.ctx.count_kmers_into(self.seqs, hs)
        else:
            if hs is not None and hs is not self.full:
                hs.free()
            self.local_hset = self.ctx.count_kmers(self.seqs, self.k, self.eb)

    class _DevArray:
        """a raw device allocation as a __cuda_array_interface__ object (torch.as_tensor wraps it without a copy)"""

        def __init__(self, ptr, shape, typestr):
            self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}

    def count_and_gather_in_place(self, comm, n_total):
        """K1 for this rank's shard into rows [rank * per, ...) of the full set, then ONE in-place all-gather each for the
        bins, the lengths and the magnitudes (NCCL reads every rank's own slice of the output buffer): no export copy, no
        install copy, no compaction -- the padding rows of the tail shard sit past n_total and are never swept."""
        torch = self.torch
        self._slot = 0
        rows = self.per * comm.world
        full = getattr(self, "_gfull", None)
        if full is None or len(full) != rows:
            if full is not None:
                full.free()
            full = self._gfull = self.ctx.hset_alloc(rows, self.k, self.eb)
            # the bins as bytes whatever their width: the gather moves bytes, and NCCL has no unsigned 16-bit type
            self._gt = (torch.as_tensor(self._DevArray(full.device_bins(), (rows, self.N * self.eb), "|u1"), device=self.device),
                        torch.as_tensor(self._DevArray(full.device_sideband(1), (rows,), "<i8"), device=self.device),
                        torch.as_tensor(self._DevArray(full.device_sideband(0), (rows,), "<i8"), device=self.device))
        self.ctx.count_kmers_into_rows(self.seqs, full, comm.rank * self.per)    # synchronises the ctx stream
        lo = comm.rank * self.per
        for t in self._gt:
            comm.dist.all_gather_into_tensor(t, t[lo:lo + self.per])
        torch.cuda.synchronize(self.device)
        full.refresh(set_mag=False)
        self.full = full
        self.n_total = n_total
        self._local_in_full = comm.rank * self.per      # this rank's shard lives inside the full set

    def use_local_as_full(self):
        if self.full is not None and self.full is not self.local_hset and self.full is not getattr(self, "_gfull", None):
            self.full.free()
        self.full = self.local_hset
        self.n_total = None

    def export_local(self):
        torch = self.torch
        hs = self.local_hset
        if getattr(self, "_exp", None) is None:
            self._exp = (torch.ones((self.per, self.N), dtype=self._dt, device=self.device),
                         torch.zeros((self.per,), dtype=torch.int64, device=self.device),
                         torch.zeros((self.per,), dtype=torch.int64, device=self.device))
        bins, length, mag = self._exp           # padding rows (if any) keep their initial all-ones / zero contents
        torch.cuda.synchronize(self.device)     # the fills above run on torch's stream
        if self.n_local:
            hs.copy_to_device(bins.data_ptr(), mag.data_ptr(), length.data_ptr(), 0, self.n_local)
        return bins, length, mag

    def install_full(self, bins, length, mag, n_total):
        self.torch.cuda.synchronize(self.device)
        self.n_total = None
        if self.full is not None and self.full is not self.local_hset and len(self.full) == n_total:
            self.full.update_from_device(bins.data_ptr(), length.data_ptr(), mag.data_ptr())
            return
        if self.full is not None and self.full is not self.local_hset:
            self.full.free()
        self.full = self.ctx.hset_from_device(bins.data_ptr(), n_total, self.k, self.eb, length.data_ptr(),
                                              mag.data_ptr())

    # ---- sharded candidate scan (candidate_scan) ----
    def query_pack(self):
        """the query message of a distributed scan: length (8 bytes) | magnitude (8) | bins, ONE device buffer kept for the
        engine's life, so a scan costs one broadcast and no allocation"""
        if getattr(self, "_qpack", None) is None:
            self._qpack = self.torch.zeros((16 + self.N * self.eb,), dtype=self.torch.uint8, device=self.device)
        return self._qpack

    def empty_query(self):
        torch, pack = self.torch, self.query_pack()
        return pack[16:].view(self._dt).view(1, self.N), pack[0:8].view(torch.int64), pack[8:16].view(torch.int64)

    def local_query(self, row_local):
        bins, length, mag = self.empty_query()
        hs, base, _ = self._local()
        hs.copy_to_device(bins.data_ptr(), mag.data_ptr(), length.data_ptr(), base + row_local, 1)
        self.ctx.sync()                                 # the copy ran on the context's stream; the broadcast runs on torch's
        return bins, length, mag

    def _marks(self, n):
        """page-locked mark buffer reused by every scan (a fresh pageable array costs page faults and a staged copy per call)"""
        buf = getattr(self, "_marks_buf", None)
        if buf is None or len(buf) < n:
            if buf is not None and self._marks_pinned:
                self.capi.host_unregister(buf)
            buf = self._marks_buf = np.zeros(max(n, 1 << 16), dtype=np.uint8)
            try:
                self.capi.host_register(buf)
                self._marks_pinned = True
            except self.capi.Mc2Error:          # locked-memory limit: a pageable buffer still works
                self._marks_pinned = False
        return buf

    def scan_local(self, bins, length, mag, cutoff):
        self.torch.cuda.synchronize(self.device)
        if getattr(self, "_qset", None) is None:
            self._qset = self.ctx.hset_from_device(bins.data_ptr(), 1, self.k, self.eb, length.data_ptr(), mag.data_ptr())
        else:
            self._qset.update_from_device(bins.data_ptr(), length.data_ptr(), mag.data_ptr())
        hs, base, n = self._local()
        if n == 0:
            return -1, -1.0, True, np.zeros(0, dtype=np.uint8)
        return self.ctx.get_close(self.model, self._qset, 0, hs, cand_begin=base, n_cand=n, cutoff=cutoff, marks=self._marks(n))

    def scan_row(self, row_local, cutoff):
        """get_close of a row of the local shard against the whole shard (what a scan is with one rank)"""
        hs, base, n = self._local()
        return self.ctx.get_close(self.model, hs, base + row_local, hs, cand_begin=base, n_cand=n, cutoff=cutoff, marks=self._marks(n))

    # ---- update stage (update_pass / merge_pass) over the replicated set self.full ----
    def _stage_centers(self, rows, mag, length):
        n = len(rows)
        sc = getattr(self, "_centers", None)
        if sc is None or len(sc) < n:
            if sc is not None:
                sc.free()
            cap = max(n, 64)
            sc = self._centers = self.ctx.hset_from_host(np.ones((cap, self.N), dtype=self.capi.DTYPES[self.eb]), self.k,
                                                         length=np.ones(cap, dtype=np.uint64))
        sc.assign_rows(np.arange(n, dtype=np.uint64), self.full, rows, mag=mag, length=length)
        return sc

    def update_centers(self, rows, mag, length, off, members, cutoff):
        sc = self._stage_centers(rows, mag, length)
        return self.ctx.update_centers(self.model, sc, len(rows), self.full, off, members, cutoff)

    def merge_centers(self, rows, mag, length, delta, cutoff):
        sc = self._stage_centers(rows, mag, length)
        return self.ctx.merge_centers(self.model, sc, len(rows), delta, cutoff)

    def topk(self, q0, q1, upper_only, cutoff, identity, top_k):
        """each query's top_k best identity hits (Context.identity_topk) -> (total hits, n_scored, table)"""
        model, t = identity[:2]
        nd = min(len(self.full), getattr(self, "n_total", None) or len(self.full))   # rows past n_total are shard padding
        r = self.ctx.identity_topk(model, self.full, self.full, t, top_k, cutoff, q_range=(q0, q1), d_range=(0, nd),
                                   upper_only=upper_only)
        return int(r["n_hits"].sum()), r["n_scored"], r

    def sweep(self, q0, q1, upper_only, cutoff, max_out, identity=None):
        """identity: None = the engine's classifier (all_pairs), else (regression model, min_identity) (identity_pairs) or
        (regression model, min_identity, both_strands) (identity_pairs_both_strands when both_strands is true)"""
        # survivor buffers: one page-locked triple per block of a step, allocated once and reused by every step (fresh
        # pageable arrays cost page faults + a staged copy per call; a shared triple would force a host copy per block)
        slots = getattr(self, "_surv_slots", None)
        if slots is None:
            slots = self._surv_slots = []
        slot = getattr(self, "_slot", 0)
        self._slot = slot + 1
        while len(slots) <= slot:
            slots.append(None)
        if slots[slot] is None or len(slots[slot][0]) < max_out:
            if slots[slot] is not None:
                for old in slots[slot][3]:
                    self.capi.host_unregister(old)
            bufs = (np.zeros(max_out, dtype=np.uint64), np.zeros(max_out, dtype=np.uint64), np.zeros(max_out, dtype=np.float64))
            pinned = []
            for b in bufs:
                try:
                    self.capi.host_register(b)
                    pinned.append(b)
                except self.capi.Mc2Error:      # locked-memory limit: pageable buffers still work
                    pass
            slots[slot] = bufs + (pinned,)
        nd = min(len(self.full), getattr(self, "n_total", None) or len(self.full))   # rows past n_total are shard padding
        if identity is not None and len(identity) > 2 and identity[2]:
            model, t = identity[:2]
            strand = getattr(self, "_strand_slots", {})
            self._strand_slots = strand
            if slot not in strand or len(strand[slot]) < max_out:
                strand[slot] = np.zeros(max_out, dtype=np.int8)
            r = self.ctx.identity_pairs_both_strands(model, self.full, self.full, t, cutoff, q_range=(q0, q1), d_range=(0, nd),
                                                     upper_only=upper_only, max_out=max_out,
                                                     out=slots[slot][:3] + (strand[slot],))
            return r["n_out"], r["n_scored"], (r["q"], r["d"], r["identity"], r["strand"])
        if identity is not None:
            model, t = identity[:2]
            r = self.ctx.identity_pairs(model, self.full, self.full, t, cutoff, q_range=(q0, q1), d_range=(0, nd),
                                        upper_only=upper_only, max_out=max_out, out=slots[slot][:3])
            return r["n_out"], r["n_scored"], (r["q"], r["d"], r["identity"])
        r = self.ctx.all_pairs(self.model, self.full, self.full, cutoff, q_range=(q0, q1), d_range=(0, nd),
                               upper_only=upper_only, max_out=max_out, out=slots[slot][:3])
        return r["n_out"], r["n_scored"], (r["q"], r["d"], r["score"])
