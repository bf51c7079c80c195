#!/usr/bin/env python
"""bench.py — one JSON line for the MeShClust2 hot path on B200 (DESIGN.md §Measurement).

A step = one pass of the hot path over one batch of synthetic mutated-template DNA:
    K1  k-mer histograms of every sequence (Loader<T>::get_point), then
    K2  the all-pairs feature + GLM + cutoff sweep with the reference's length prefilter (fastcar work() /
        the candidate scans of Trainer::get_close) -> survivor list.
`value` = pairs scored per second over the whole step with the packed sequences already resident in HBM;
`e2e`   = the same metric through the C ABI from HOST buffers (codes + segments in, survivors out), copies timed.
N > 1: one process per GPU (torchrun); sequences sharded for K1, histogram shards all-gathered over NCCL, the sweep
split by folded query-row blocks; total work fixed ("strong" scaling).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg4|cfg5] [--n-seqs N]
                  [--dump-outputs DIR]

--workload cfg4 / cfg5 print the same kind of line for BASELINE configs[3] (long records, k=8, uint16) and configs[4]
(1M x 1 kb candidate scans + one update / merge pass, sharded over the ranks); the default cfg3 run carries both as
`also_cfg4` / `also_cfg5` blocks so that the default run times them.
--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (dump_outputs; cfg5: dump_scan_outputs), so
that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sequence pairs scored/sec (features+GLM)"
UNIT = "pairs/s"
WEIGHTS = os.path.join(ROOT, "tests", "golden", "weights_cfg1_id90.txt")
WORKLOADS = {
    # BASELINE.json configs[2]: 100k sequences 1 kb, k=5, uint8, all-pairs feature+GLM sweep at 1/2/4/8 B200
    "cfg3": dict(synth="cfg3", desc="BASELINE configs[2]: 100k x 1 kb, k=5, uint8, all-pairs feature+GLM sweep (id 0.9)"),
    # BASELINE.json configs[1] shape: 10k 16S-like 1.5 kb (hot-path content of the train+cluster run: K1 + candidate scans)
    "cfg2": dict(synth="cfg2", desc="BASELINE configs[1] shape: 10k x 1.5 kb 16S-like, k=5, uint8, K1 + all-pairs candidate sweep (id 0.9)"),
    # BASELINE.json configs[3]: 5k long records (5 contigs x 10 kb joined by 50 N, --single-file), k=8, uint16 (128 KiB rows)
    "cfg4": dict(synth=None, desc="BASELINE configs[3]: 5k x 50 kb --single-file records, k=8, uint16 (65,536-bin rows), K1 + all-pairs sweep (id 0.9)"),
    # BASELINE.json configs[4]: 1M x 1 kb, candidate scans of the mean-shift accumulate stage + update / merge passes at --delta 5
    "cfg5": dict(synth=None, desc="BASELINE configs[4]: 1M x 1 kb, k=5, uint8, Trainer::get_close candidate scans sharded over the ranks + one update / merge pass (--delta 5)"),
}
N_DEFAULT = {"cfg3": 100000, "cfg2": 10000, "cfg4": 5000, "cfg5": 1000000}


def workload_config(name, n_total, k, eb):
    """The `config` object: identical in both arms (the driver compares them key by key)."""
    return {"workload": WORKLOADS[name]["desc"], "n_sequences": int(n_total), "k": int(k), "elem_bytes": int(eb),
            "pairs_per_step": int(n_total) * (int(n_total) - 1) // 2, "model": os.path.basename(WEIGHTS), "cutoff": 0.9}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def profile_entry(key):
    """per-kernel figures read off the committed ncu --set full captures (profiles/r2_traffic.json, then r1_traffic.json):
    dram_bytes_per_pair, warp_instr_per_pair, tensor_pipe_pct, source"""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            for k, v in d.items():
                if k.startswith(key):
                    return v
        except Exception:
            pass
    return {}


def traffic_per_pair(key):
    v = profile_entry(key)
    return (float(v["dram_bytes_per_pair"]), v.get("source")) if "dram_bytes_per_pair" in v else (None, None)


def instr_per_pair(key):
    v = profile_entry(key)
    return (float(v["warp_instr_per_pair"]), v.get("source")) if "warp_instr_per_pair" in v else (None, None)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, sampled in-process through NVML every 200 ms
    (the B200_PROFILING.md clocks line without spawning nvidia-smi, whose polling loop perturbs short steps)."""

    def __init__(self, device, interval=0.5):
        self.device, self.rows, self.stop_flag, self.t, self.interval = device, [], False, None, interval
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(device))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(device):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[device])
            except Exception:
                pass
        return device

    def _loop(self):
        nv = self.nv
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                # two light NVML reads per sample; NVML queries serialise with CUDA calls in the driver, so keep them sparse
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), mx, reasons(self.h)))
            except Exception:
                pass
            for _ in range(int(self.interval / 0.05)):
                if self.stop_flag:
                    break
                time.sleep(0.05)

    def start(self):
        if self.nv is None:
            return
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def stop(self):
        if self.nv is None or self.t is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.t.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        sm = [r[0] for r in self.rows]
        smax = self.rows[-1][1] if self.rows else None
        reasons = sorted(k for k, bit in names.items() if any(r[2] & bit for r in self.rows))
        busy = [x for x in sm if smax and x > 0.3 * smax] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": float(smax) if smax else None,
                "reasons": reasons, "samples": len(sm)}


def load_workload(name, n_override, lo, hi):
    from meshclust2_b200 import synth
    t0 = time.time()
    if name == "cfg4":
        n = n_override or N_DEFAULT["cfg4"]
        seqs = synth.make_single_file(n, 5, 10000, seed=4)[lo:hi]
        k, eb = 8, 2
    else:
        seqs, _, k, eb = synth.make_config_range(WORKLOADS[name]["synth"] or name, lo=lo, hi=hi, n=n_override)
    log("[bench] generated %d synthetic sequences [%d,%d) in %.1fs" % (len(seqs), lo, hi, time.time() - t0))
    return seqs, k, eb


def host_bytes(enc):
    return int(enc["codes"].nbytes + enc["seq_off"].nbytes + enc["segs"].nbytes + enc["seg_off"].nbytes)


# ---------------------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the reference's own implementation compiled in place (oracle/_ref), else the C port
# ---------------------------------------------------------------------------------------------------------------
def cpu_leg(seqs, k, eb, n_total, n_scored_total, cutoff, hist_sample, pair_sample, seed=0):
    """Times Loader<T>::get_point (omp over sequences) and Predictor<T>::close (omp over pairs) on all host cores on a
    bounded sample of the workload; returns dict with the workload-equivalent pairs/s."""
    from oracle import port, ref
    threads = os.cpu_count() or 1
    rng = np.random.default_rng(seed)
    model_txt = open(WEIGHTS).read()
    hs = min(hist_sample, len(seqs))
    sample = [seqs[i] for i in rng.choice(len(seqs), hs, replace=False)] if hs < len(seqs) else list(seqs)
    if ref.available():
        kind = "reference"
        H, t_hist = ref.count_batch(sample, k, eb, threads=threads, want_hist=True)
        ln = np.array([len(s) for s in sample], dtype=np.uint64)   # synthetic ACGT: effective size == length
    else:
        kind = "port"
        encs = [port.encode(s) for s in sample]
        codes = np.concatenate([e[0] for e in encs])
        seq_off = np.concatenate([[0], np.cumsum([len(e[0]) for e in encs])])
        segs = np.concatenate([e[1].reshape(-1, 2) for e in encs])
        seg_off = np.concatenate([[0], np.cumsum([len(e[1].reshape(-1, 2)) for e in encs])])
        H, t_hist = port.count_batch(codes, seq_off, segs, seg_off, k, eb, threads=threads)
        ln = np.array([e[2] for e in encs], dtype=np.uint64)
    hist_rate = hs / t_hist
    # pairs inside the length window, as the sweep scores them
    order = np.argsort(ln, kind="stable")
    ia = rng.integers(0, hs, pair_sample * 2)
    ib = rng.integers(0, hs, pair_sample * 2)
    lo = (ln[ib].astype(np.float64) * cutoff).astype(np.uint64)
    hi = (ln[ib].astype(np.float64) / cutoff).astype(np.uint64)
    ok = (ln[ia] >= lo) & (ln[ia] <= hi)
    ia, ib = ia[ok][:pair_sample], ib[ok][:pair_sample]
    if kind == "reference":
        rm = ref.RefModel(model_txt, eb, cutoff)
        r = rm.score_pairs(H, None, ln, ia, ib, mode=1, threads=threads)      # Predictor<T>::close
        t_pairs, n_close = r["seconds"], int(r["close"].sum())
    else:
        m = port.Model.from_text(model_txt)
        mag = H.sum(axis=1, dtype=np.uint64)
        r = port.score_pairs(m, H, mag, ln, ia, ib, threads=threads, want_cache=False)
        t_pairs, n_close = r["seconds"], int(r["close"].sum())
    pair_rate = len(ia) / t_pairs
    t_step = n_total / hist_rate + n_scored_total / pair_rate
    del order
    return dict(value=n_scored_total / t_step, unit=UNIT, cores=threads, kind=kind,
                sample="%d sequences through Loader<T>::get_point (%.2fs) + %d in-window pairs through Predictor<T>::close "
                       "(%.2fs), %d OpenMP threads; extrapolated to the step's %d histograms + %d pairs; the pairs are drawn "
                       "at random over the sample (worse cache locality than fastcar's query-major loop)" % (
                           hs, t_hist, len(ia), t_pairs, threads, n_total, n_scored_total),
                hist_per_s=hist_rate, pairs_per_s_kernel=pair_rate, seconds=t_hist + t_pairs, n_close_sample=n_close)


def run_reference(args, rank, world):
    if rank != 0:
        return
    n_total = args.n or N_DEFAULT[args.workload]
    nsamp = min(n_total, args.cpu_hist_sample if args.workload != "cfg4" else 256)
    seqs, k, eb = load_workload(args.workload, args.n if args.workload != "cfg4" else nsamp, 0, nsamp)
    n_scored_total = n_total * (n_total - 1) // 2          # synthetic lengths are within the 0.9 window (L +/- 5 %)
    pair_sample = args.cpu_pair_sample if args.workload != "cfg4" else 200000
    vals, secs = [], []
    leg = None
    for s in range(args.warmup + args.steps):
        leg = cpu_leg(seqs, k, eb, n_total, n_scored_total, 0.9, nsamp, pair_sample, seed=s)
        if s >= args.warmup:
            vals.append(leg["value"])
            secs.append(leg["seconds"])
    v = float(np.mean(vals))
    line = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": float(np.mean(secs)) * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8" if eb == 1 else "u16", "data": "synthetic", "impl": "reference",
            "config": workload_config(args.workload, n_total, k, eb),
            "notes": {"sampling": "each step is a bounded sample; value is the workload-equivalent rate"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": leg["cores"], "kind": leg["kind"], "sample": leg["sample"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    from meshclust2_b200 import capi, dist as mdist
    import torch
    tdist = None
    if world > 1:
        import torch.distributed as tdist_mod
        torch.cuda.set_device(local_rank)
        tdist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        tdist = tdist_mod
    comm = mdist.Comm(tdist)
    n_total = args.n or N_DEFAULT[args.workload]
    if args.workload == "cfg5":
        # the candidate-scan form: a step = 16 Trainer::get_close scans over the whole sharded set
        ctx = capi.Context(local_rank)
        model = ctx.model_from_file(WEIGHTS)
        peak, peak_src = peaks()
        dump = {} if args.dump_outputs else None
        blk = cfg5_block(ctx, capi, mdist, torch, comm, model, model.meta["id"], local_rank, peak, n_total=n_total,
                         n_queries=16 * args.steps, dump=dump)
        if dump is not None:
            dump_scan_outputs(args.dump_outputs, dump, comm)
        cs = blk["candidate_scan"]
        line = {"metric": METRIC, "value": cs["pairs_per_s"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": 4,
                "ms_per_step": cs["ms_per_query"] * 16, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic (histograms generated directly)", "config": workload_config("cfg5", n_total, 5, 1),
                "notes": {"step": "16 get_close scans over all candidates; 4 warm-up scans"},
                "e2e": {"value": cs["pairs_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 16 * (n_total // world + 64),
                        "from": "mc2_get_close through the C ABI: marks and the arg-max come back to the host every scan"},
                "gpu_launches": int(ctx.launches),
                "roofline": {"bound": "hbm", "achieved": cs["achieved_gbs"], "peak": peak * world, "unit": "GB/s",
                             "frac": cs["frac_of_hbm_per_gpu"], "traffic": None, "kernel": "pair_fast_kernel<u8> (one query vs shard)",
                             "algorithmic_bytes_per_unit": 1057, "peak_source": peak_src},
                "cfg5": blk}
        if rank == 0:
            emit(line)
        ctx.close()
        if tdist is not None:
            tdist.destroy_process_group()
        return
    per, bounds = mdist.shard_bounds(n_total, world)
    lo, hi = bounds[rank]
    seqs, k, eb = load_workload(args.workload, args.n, lo, hi)
    t0 = time.time()
    enc = capi.encode_batch(seqs)
    log("[bench] rank %d host encode %.2fs" % (rank, time.time() - t0))
    ctx = capi.Context(local_rank)
    pin_inputs(capi, enc)
    model = ctx.model_from_file(WEIGHTS)
    cutoff = model.meta["id"]
    eng = mdist.GpuEngine(capi, ctx, torch, model, k, eb, local_rank)
    eng.set_local_sequences(ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"]), hi - lo, per)
    max_out = 1 << 22

    def step_resident():
        ctx.flush_l2(256 << 20)
        return mdist.all_pairs_step(eng, comm, torch, n_total, cutoff, upper_only=True, blocks_per_rank=args.blocks_per_rank,
                                    max_out=max_out)

    # end to end starts from RAW sequence text in page-locked host memory: H2D, N-run segmentation, letter coding and
    # packing (mc2_seqs_from_text_into), K1, exchange, sweep, D2H of the survivors are all inside the timed region
    text = np.frombuffer(bytearray(b"".join(seqs)), dtype=np.uint8) if seqs else np.zeros(1, dtype=np.uint8)
    text_off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    text_off[1:] = np.cumsum([len(s) for s in seqs])
    for arr in (text, text_off):
        try:
            capi.host_register(arr)
        except capi.Mc2Error as e:
            log("[bench] could not page-lock the text: %s" % e)

    def step_e2e():
        ctx.flush_l2(256 << 20)
        ctx.seqs_from_text_into(eng.seqs, text, text_off)
        return mdist.all_pairs_step(eng, comm, torch, n_total, cutoff, upper_only=True, blocks_per_rank=args.blocks_per_rank,
                                    max_out=max_out)

    def timed(fn, steps, sample_clocks=False):
        sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()          # before the barrier: rank 0 must not enter the timed region later than the others
        comm.barrier()
        torch.cuda.synchronize()
        ctx.sync()
        l0 = ctx.launches
        ctx.profile(True)
        ctx.timer_start()
        res = None
        for _ in range(steps):
            res = fn()
        ms = ctx.timer_stop()
        comm.barrier()
        torch.cuda.synchronize()
        ktime = {kind: ctx.kernel_time(kind) for kind in range(6)}
        ctx.profile(False)
        clocks = sampler.stop() if sampler else None
        ms = comm.all_reduce_max(ms, torch, eng.device)
        return ms, res, ctx.launches - l0, ktime, clocks

    for _ in range(args.warmup):
        res = step_resident()
    ms, res, launches, ktime, clocks = timed(step_resident, args.steps, sample_clocks=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res, eng, n_total, comm)
    n_scored = res["n_scored"]
    value = n_scored * args.steps / (ms * 1e-3)
    log("[bench] rank %d per-kind device ms per step: %s" % (rank, {kk: round(v[0] / args.steps, 3) for kk, v in ktime.items()}))
    log("[bench] rank %d resident: %.1f ms/step, %d pairs scored, %d close, %d launches" % (
        rank, ms / args.steps, n_scored, res["n_close"], launches))
    # end to end from host buffers
    log("[bench] rank %d e2e phase" % rank)
    for _ in range(min(args.warmup, 3)):
        step_e2e()
    e2e_steps = max(1, min(args.steps, 3))
    ms_e, res_e, _, _, _ = timed(step_e2e, e2e_steps)
    e2e_value = res_e["n_scored"] * e2e_steps / (ms_e * 1e-3)
    log("[bench] rank %d e2e: %.1f ms/step" % (rank, ms_e / e2e_steps))
    h2d = int(text.nbytes + text_off.nbytes)
    d2h = int(len(res_e["survivors"]) * 24 + 16 * len(res_e["blocks"]))

    # roofline of the dominant kernel (the sweep).  SURVEY.md 8(d), all-pairs tile sweep row: "not HBM -- CUDA-core integer
    # issue rate for sum-min and sum|cum diff|, tensor pipe for sum p*q".  Algorithmic CUDA-core work of the benchmarked model
    # (Gram term + EMD): the EMD's N bins at the densest instructions the ISA has for 16-bit cumulative values, 2 bins per
    # VIMNMX.U16x2 and 2 per IDP.2A -> N lane-instructions = N/32 warp-instructions per pair; the Gram term's 2N integer
    # ops per pair run on the tensor pipe.  Peak = the same instruction pair measured in this process (mc2_bench_issue_rate).
    N = 4 ** k
    sweep_ms, sweep_n = ktime[3]
    count_ms, count_n = ktime[1]
    peak, peak_src = peaks()
    local_pairs = res["local_scored"] * args.steps
    tile = eb in (1, 2) and 5 <= k <= 8          # the synthetic sets fit the tile form (counts below 256, sums in 16 bits)
    kernel_name = "tile_sweep_kernel<NEED_DOT|NEED_EMD> (TMA ring + tcgen05 u8 MMA + VIMNMX.U16x2/IDP.2A EMD), %d slab%s per row" % (
        N // 1024, "" if k == 5 else "s") if tile else "sweep_wide_kernel<u16,NEED_DOT|NEED_EMD>"
    if tile:
        prof = profile_entry("tile_sweep_kernel") if k == 5 else (profile_entry("tile_sweep_kernel<NEED_DOT|NEED_EMD>, 64 slabs") if k == 8 else {})
    else:
        prof = profile_entry("sweep_wide_kernel")
    pairs_per_s_kernel = local_pairs / (sweep_ms * 1e-3) if sweep_ms > 0 else 0.0
    try:
        probe = ctx.issue_rate()
    except Exception as e:
        log("[bench] issue-rate probe failed: %r" % (e,))
        probe = None
    # tile sweep: N/32; wide rows (u16 bins, no cumulative rows): Gram term on CUDA cores as well, N/2 IDP.2A more
    alg_wi = N / 32.0 if tile else (N + N / 2) / 32.0
    ach = pairs_per_s_kernel * alg_wi
    tpp = prof.get("dram_bytes_per_pair")
    roofline = {"bound": "alu", "achieved": ach / 1e9, "peak": probe / 1e9 if probe else None, "unit": "Gwarp-instr/s",
                "frac": ach / probe if probe else None,
                "traffic": tpp * local_pairs / max(1, sweep_n) if tpp else None, "traffic_source": prof.get("source"),
                "kernel": kernel_name,
                "algorithmic_ops_per_unit": alg_wi, "algorithmic_ops_unit": "warp-instructions per pair",
                "algorithmic_ops_note": "EMD over N=4^k bins on 16-bit cumulative values: N/2 VIMNMX.U16x2 + N/2 IDP.2A lane-"
                                        "instructions (2 bins each)" + ("" if tile else " + N/2 IDP.2A for the Gram term") +
                                        "; SURVEY 8(d) counts the same work as N byte-ops per reduction at 4 bins per SIMD op "
                                        "(N/4 lane-instructions + accumulation), which no sm_100a instruction offers for 16-bit data",
                "units_per_launch": local_pairs / max(1, sweep_n),
                "avg_launch_ms": sweep_ms / max(1, sweep_n), "launches": sweep_n,
                "kernel_share_of_step": sweep_ms / ms if ms > 0 else None,
                "peak_source": "mc2_bench_issue_rate: VIMNMX.U16x2 + IDP.2A, register operands, 32 warps / SM, measured in this process",
                "pairs_per_s": pairs_per_s_kernel,
                "hbm": {"achieved_gbs": (tpp * pairs_per_s_kernel / 1e9) if tpp else None, "peak_gbs": peak, "peak_source": peak_src,
                        "frac": (tpp * pairs_per_s_kernel / 1e9 / peak) if tpp else None,
                        "note": "measured DRAM bytes per pair (ncu) x live pairs/s: the sweep is not HBM bound"},
                "tensor": {"int_ops_per_pair": 2 * N if tile else 0, "achieved_tops": pairs_per_s_kernel * 2 * N / 1e12 if tile else 0.0,
                           "pipe_active_pct": prof.get("tensor_pipe_pct"),
                           "note": "Gram term sum p*q: tcgen05.mma kind::i8 (u8 x u8 -> s32, exact) into TMEM; it is ~1 % of the "
                                   "tensor pipe because the CUDA-core EMD term paces the tile"}}
    ipp = prof.get("warp_instr_per_pair")
    sm_mhz = (clocks or {}).get("sm_mhz")
    if ipp and sm_mhz:
        issue_peak = ctx.sm_count * 4 * sm_mhz * 1e6
        roofline["issue"] = {"executed_warp_instr_per_pair": ipp, "achieved": pairs_per_s_kernel * ipp / 1e9, "peak": issue_peak / 1e9,
                             "unit": "Gwarp-instr/s", "frac": pairs_per_s_kernel * ipp / issue_peak,
                             "note": "slot occupancy (counts overhead as work): executed instructions per pair from the committed "
                                     "ncu capture x live pairs/s over 4 schedulers x SMs x sampled clock"}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u8" if eb == 1 else "u16", "data": "synthetic",
            "config": workload_config(args.workload, n_total, k, eb),
            "notes": {"pairs_scored_per_step": n_scored, "pairs_close_per_step": res["n_close"],
                      "parallelism": "equal-pair-count query-row ranges x%d (one sweep launch per rank), in-place NCCL all-gather of histograms" % world,
                      "l2": "L2 flushed between steps (256 MB memset inside the timed region)",
                      "e2e_steps": e2e_steps},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                    "ms_per_step": ms_e / e2e_steps, "steps": e2e_steps,
                    "from": "raw sequence text in page-locked host memory (mc2_seqs_from_text_into -> mc2_count_kmers_into -> "
                            "mc2_all_pairs; survivors copied back)"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "k1": {"hist_per_s": (hi - lo) * args.steps / (count_ms * 1e-3) if count_ms > 0 else None,
                   "avg_launch_ms": count_ms / max(1, count_n),
                   "achieved_gbs": (hi - lo) * args.steps * (np.mean([len(x) for x in seqs]) / 4 + N * eb + 40) / (count_ms * 1e-3) / 1e9 if count_ms > 0 and seqs else None}}
    if line["k1"]["achieved_gbs"]:
        line["k1"]["frac_of_hbm"] = line["k1"]["achieved_gbs"] / peak
    if not args.no_extras:
        if world == 1 and k == 5 and eb == 1:
            line["roofline_candidates"] = candidates_roofline(ctx, capi, model, k, eb, peak, peak_src)
            try:
                line["gram_term"] = gram_term_block(ctx, capi, eng.full, n_total, cutoff)
            except Exception as e:
                log("[bench] gram-term extra failed: %r" % (e,))
            try:
                line["slow_singles"] = slow_singles_block(ctx, capi, peak)
            except Exception as e:
                log("[bench] slow-singles extra failed: %r" % (e,))
        if world == 1 and args.workload == "cfg3":
            line["also_cfg2"] = small_workload(ctx, capi, mdist, torch, model, cutoff)
            if rank == 0:
                try:
                    line["also_cfg2"]["e2e_cluster"] = e2e_cluster_block()
                except Exception as e:
                    log("[bench] e2e_cluster extra failed: %r" % (e,))
                try:
                    line["also_cfg2"]["e2e_fastcar"] = e2e_fastcar_block()
                except Exception as e:
                    log("[bench] e2e_fastcar extra failed: %r" % (e,))
        if args.workload == "cfg3":
            try:
                if world == 1:
                    line["also_cfg4"] = cfg4_block(ctx, capi, model, cutoff, peak, probe)
                line["also_cfg5"] = cfg5_block(ctx, capi, mdist, torch, comm, model, cutoff, local_rank, peak)
            except Exception as e:                      # an extra, never the reason a bench line is lost
                log("[bench] cfg4 / cfg5 extra failed: %r" % (e,))
    if rank == 0 and world == 1 and not args.no_cpu:
        t0 = time.time()
        cb = cpu_leg(seqs, k, eb, n_total, n_scored, cutoff, args.cpu_hist_sample, args.cpu_pair_sample)
        log("[bench] cpu baseline leg %.1fs" % (time.time() - t0))
        line["cpu_baseline"] = {kk: cb[kk] for kk in ("value", "unit", "cores", "kind", "sample")}
    if rank == 0:
        emit(line)
    ctx.close()
    if tdist is not None:
        tdist.destroy_process_group()


def pin_inputs(capi, enc):
    """page-lock the step's host inputs (the encoded batch) so the timed H2D copies are DMA transfers from pinned memory"""
    done = []
    for key in ("codes", "seq_off", "segs", "seg_off"):
        enc[key] = np.ascontiguousarray(enc[key])
        if enc[key].nbytes:
            try:
                capi.host_register(enc[key])
                done.append(enc[key])
            except capi.Mc2Error as e:          # e.g. a locked-memory limit: the copies still work, just through pageable memory
                log("[bench] could not page-lock %s: %s" % (key, e))
    return done


DUMP_MAX_SURVIVORS = 1 << 21        # three float64 arrays: 48 MiB
DUMP_HIST_BYTES = 8 << 20           # the float32 histogram sample


def _pair_sample(a, b, cap):
    """The pairs (a[i], b[i]) in (a, b) order: all of them up to cap, above it a fixed sample, the pairs whose splitmix64
    hash has its top `shift` bits clear, with the smallest shift that brings the expected count to 3/4 of cap.  Whether a
    pair is kept depends on the pair alone, so two builds that differ in one pair differ in that pair only (unless their
    pair counts fall on two sides of cap or of a halving step).  Returns (indices into a / b, shift)."""
    shift = 0
    while len(a) > cap and (len(a) >> shift) > cap * 3 // 4:
        shift += 1
    keep = np.arange(len(a))
    if shift:
        with np.errstate(over="ignore"):
            h = a.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15) ^ b.astype(np.uint64)
            h ^= h >> np.uint64(30)
            h *= np.uint64(0xBF58476D1CE4E5B9)
            h ^= h >> np.uint64(27)
            h *= np.uint64(0x94D049BB133111EB)
            h ^= h >> np.uint64(31)
        keep = np.flatnonzero((h >> np.uint64(64 - shift)) == 0)
    return keep[np.lexsort((b[keep], a[keep]))], shift


def _save_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32 if name == "hist" else np.float64))


def dump_outputs(out_dir, res, eng, n_total, comm):
    """--dump-outputs, all-pairs workloads: what the last timed step computed, as out_dir/<name>.npy, float64 unless noted
    (56 MiB at most):
      survivor_q, survivor_d, survivor_score   the survivor pairs of every rank and their scores, in (q, d) order; above
                                               DUMP_MAX_SURVIVORS pairs the fixed hash sample of _pair_sample
      counts                                   [pairs scored, pairs close, survivors returned, sample shift]
      hist_rows, hist (float32), hist_mag, hist_len
                                               32 fixed seeded runs of consecutive k-mer histogram rows of the step, with
                                               the rows' magnitudes and lengths
    Runs before the next step: the survivors are views of buffers the engine reuses."""
    surv = res["survivors"]
    qd = surv.array()
    q, d, score = qd[:, 0], qd[:, 1], surv.scores()
    if comm.dist is not None:
        parts = [None] * comm.world
        comm.dist.all_gather_object(parts, (q, d, score))
        q, d, score = (np.concatenate([p[i] for p in parts]) for i in range(3))
    if comm.rank != 0:
        return
    order, shift = _pair_sample(q, d, DUMP_MAX_SURVIVORS)
    want = min(n_total, max(1, DUMP_HIST_BYTES // (4 * eng.N)))
    run = max(1, want // 32)
    starts = np.sort(np.random.default_rng(1).choice(n_total // run, want // run, replace=False)) * run
    got = [eng.full.download(int(a), run) for a in starts]
    _save_outputs(out_dir, {"survivor_q": q[order], "survivor_d": d[order], "survivor_score": score[order],
                            "counts": [res["n_scored"], res["n_close"], len(q), shift],
                            "hist_rows": np.concatenate([np.arange(a, a + run) for a in starts]),
                            "hist": np.concatenate([g["hist"] for g in got]),
                            "hist_mag": np.concatenate([g["mag"] for g in got]),
                            "hist_len": np.concatenate([g["len"] for g in got])})
    log("[bench] last step's outputs written to %s (%d of %d survivors, %d histogram rows)" % (
        out_dir, len(order), len(q), len(starts) * run))


def dump_scan_outputs(out_dir, dump, comm):
    """--dump-outputs, cfg5: what the last timed step computed, as out_dir/<name>.npy, all float64 (48 MiB at most):
      scan_q, scan_best, scan_best_dist, scan_is_min   the step's 16 get_close scans: query row, arg-max row (-1: none), its
                                                       distance, whether no candidate was close
      mark_q, mark_candidate                           the (query, candidate) pairs the scans marked close, every rank's, in
                                                       that order; above DUMP_MAX_SURVIVORS the hash sample of
                                                       _pair_sample
      counts                                           [pairs marked, sample shift]
      update_next, update_n_good, merge_choice         the timed update + merge pass (-1 / 0: none)"""
    mq, mc = dump.pop("marks")
    if comm.dist is not None:
        parts = [None] * comm.world
        comm.dist.all_gather_object(parts, (mq, mc))
        mq, mc = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
    if comm.rank != 0:
        return
    order, shift = _pair_sample(mq, mc, DUMP_MAX_SURVIVORS)
    dump.update(mark_q=mq[order], mark_candidate=mc[order], counts=[len(mq), shift])
    _save_outputs(out_dir, dump)
    log("[bench] last step's outputs written to %s (%d of %d marks)" % (out_dir, len(order), len(mq)))


def small_workload(ctx, capi, mdist, torch, model, cutoff, steps=20):
    """The BASELINE configs[1] shape in the same run (10k x 1.5 kb 16S-like, k=5, uint8): K1 + all-pairs candidate sweep,
    resident and end to end; the whole histogram set (10 MB) is L2-resident, steps are ~15 ms."""
    from meshclust2_b200 import synth
    seqs, _, k, eb = synth.make_config_range("cfg2", 0, None)
    enc = capi.encode_batch(seqs)
    pinned = pin_inputs(capi, enc)
    eng = mdist.GpuEngine(capi, ctx, torch, model, k, eb, 0)
    n = len(seqs)
    eng.set_local_sequences(ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"]), n, n)
    comm = mdist.Comm(None)
    text = np.frombuffer(bytearray(b"".join(seqs)), dtype=np.uint8)
    text_off = np.zeros(n + 1, dtype=np.uint64)
    text_off[1:] = np.cumsum([len(s) for s in seqs])
    for arr in (text, text_off):
        try:
            capi.host_register(arr)
            pinned.append(arr)
        except capi.Mc2Error:
            pass
    out = {}
    for name in ("resident", "e2e"):
        def step():
            ctx.flush_l2(256 << 20)
            if name == "e2e":
                ctx.seqs_from_text_into(eng.seqs, text, text_off)
            return mdist.all_pairs_step(eng, comm, torch, n, cutoff, upper_only=True, blocks_per_rank=1, max_out=1 << 22)
        for _ in range(3):
            res = step()
        ctx.sync()
        ctx.timer_start()
        for _ in range(steps):
            res = step()
        ms = ctx.timer_stop() / steps
        out[name] = {"value": res["n_scored"] / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms}
    try:
        out["update_stage"] = update_stage(ctx, capi, model, eng.full, cutoff)
    except Exception as e:                              # an extra, never the reason a bench line is lost
        log("[bench] update-stage extra failed: %r" % (e,))
    ctx.sync()
    for arr in pinned:       # a page-locked range must be released before its memory goes back to the allocator: a later
        try:                 # array landing on the same addresses would make its copies fail
            capi.host_unregister(arr)
        except capi.Mc2Error:
            pass
    out["workload"] = WORKLOADS["cfg2"]["desc"]
    out["pairs_scored_per_step"] = res["n_scored"]
    out["pairs_close_per_step"] = res["n_close"]
    out["hist_per_step"] = n
    return out


def update_stage(ctx, capi, model, hs, cutoff, delta=5, per_cluster=5, passes=5):
    """One pass of the mean-shift update stage (ClusterFactory.cpp:636-653) over the configs[1]-shaped point set: clusters of
    5 consecutive points (the synthetic set keeps a template's variants together), center = the cluster's first point,
    members of center j = the points of clusters j-delta..j+delta, merge candidates = the next delta centers.  Batched
    (mc2_update_centers + mc2_merge_centers: one device call each per pass) next to what the reference's per-center loops
    issue through the same C ABI (mc2_filter_as + mc2_mean_closest + mc2_merge per center).  Host wall clock, since the
    difference IS the per-call overhead; both forms return the same choices."""
    n = len(hs)
    got = hs.download()
    mag, ln = got["mag"].astype(np.uint64), got["len"].astype(np.uint64)
    nc = n // per_cluster
    rows = np.arange(nc, dtype=np.uint64) * per_cluster
    off = np.zeros(nc + 1, dtype=np.uint64)
    mem = []
    for j in range(nc):
        lo, hi = max(0, j - delta) * per_cluster, min(nc, j + delta + 1) * per_cluster
        mem.append(np.arange(lo, hi, dtype=np.uint64))
        off[j + 1] = off[j] + np.uint64(hi - lo)
    members = np.concatenate(mem)
    sc = ctx.hset_from_host(np.ones((nc, 4 ** hs.k), dtype=np.uint8), hs.k, length=np.ones(nc, dtype=np.uint64))
    idx = np.arange(nc, dtype=np.uint64)

    def batched():
        sc.assign_rows(idx, hs, rows, mag=mag[rows], length=ln[rows])
        nxt, ng = ctx.update_centers(model, sc, nc, hs, off, members, cutoff)
        mg = ctx.merge_centers(model, sc, nc, delta, cutoff)
        return nxt, mg

    def per_center(limit):
        nxt = np.full(limit, -1, dtype=np.int64)
        mg = np.zeros(limit, dtype=np.int64)
        sc.assign_rows(idx, hs, rows, mag=mag[rows], length=ln[rows])
        for j in range(limit):
            keep = ctx.filter_as(model, hs, int(rows[j]), int(mag[rows[j]]), int(ln[rows[j]]), hs, mem[j], cutoff).astype(bool)
            if keep.any():
                nxt[j] = np.flatnonzero(keep)[ctx.mean_closest(hs, mem[j][keep])[0]]
            mg[j] = ctx.merge(model, sc, idx, j, j + 1, min(nc - 1, j + delta), cutoff)
        return nxt, mg

    batched()
    ctx.sync()
    t0 = time.perf_counter()
    for _ in range(passes):
        b = batched()
    ctx.sync()
    t_b = (time.perf_counter() - t0) / passes
    limit = min(nc, 500)                                 # a bounded sample of the per-center form, scaled to the pass
    per_center(8)
    t0 = time.perf_counter()
    p = per_center(limit)
    ctx.sync()
    t_p = (time.perf_counter() - t0) * nc / limit
    same = bool(np.array_equal(b[0][:limit], p[0]) and np.array_equal(b[1][:limit], p[1]))
    sc.free()
    return {"centers": nc, "member_pairs_per_pass": int(off[-1]), "batched_ms_per_pass": t_b * 1e3,
            "per_center_calls_ms_per_pass": t_p * 1e3, "speedup": t_p / t_b, "same_choices": same,
            "sample": "per-center form timed on the first %d centers and scaled to %d" % (limit, nc)}


def cfg4_block(ctx, capi, model, cutoff, peak, probe=None, n=5000):
    """BASELINE configs[3] in the same run: 5k --single-file records (5 contigs x 10 kb joined by 50 N), k = 8, uint16
    histograms (65,536 bins = 128 KiB rows): K1 rate and the all-pairs sweep (tile form, and the row-streaming form beside it),
    device-timed."""
    from meshclust2_b200 import synth
    t0 = time.time()
    seqs = synth.make_single_file(n, 5, 10000, seed=4)
    enc = capi.encode_batch(seqs)
    log("[bench] cfg4: %d records generated + encoded in %.1fs" % (n, time.time() - t0))
    sq = ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"])
    L = float(np.mean([len(x) for x in seqs]))
    for _ in range(2):
        k1_ms = ctx.bench_count_kmers(sq, 8, 2, iters=3, flush_l2=True)
    hs, largest, eb = ctx.count_kmers_auto(sq, 8)
    if eb != 2:
        hs.free()
        hs = ctx.count_kmers(sq, 8, 2)
    out = {"workload": WORKLOADS["cfg4"]["desc"], "n_records": n, "mean_length": L, "largest_count": int(largest),
           "detected_elem_bytes": int(eb)}
    k1_bytes = n * (L / 4 + 65536 * 2 + 40)
    out["k1"] = {"ms": k1_ms, "hist_per_s": n / (k1_ms * 1e-3), "achieved_gbs": k1_bytes / (k1_ms * 1e-3) / 1e9,
                 "frac_of_hbm": k1_bytes / (k1_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_hist": k1_bytes / n}
    # first call: builds the tile sweep's operands for the set (u16 cumulative rows of bin - 1, the byte plane: 983 MB)
    ctx.timer_start()
    r = ctx.all_pairs(model, hs, hs, cutoff, upper_only=True, max_out=1 << 22)
    ms_first = ctx.timer_stop()
    ms_best = None
    for _ in range(3):
        ctx.flush_l2(256 << 20)
        ctx.timer_start()
        r = ctx.all_pairs(model, hs, hs, cutoff, upper_only=True, max_out=1 << 22)
        ms = ctx.timer_stop()
        ms_best = ms if ms_best is None else min(ms_best, ms)
    pps = r["n_scored"] / (ms_best * 1e-3)
    os.environ["MC2_SWEEP_LEGACY"] = "1"        # the row-streaming form (round 1), for the record
    try:
        ctx.timer_start()
        r1 = ctx.all_pairs(model, hs, hs, cutoff, upper_only=True, max_out=1 << 22)
        ms_legacy = ctx.timer_stop()
    finally:
        os.environ.pop("MC2_SWEEP_LEGACY", None)
    out["sweep"] = {"ms": ms_best, "ms_first_call_with_operand_build": ms_first, "pairs_scored": r["n_scored"], "pairs_close": r["n_out"],
                    "pairs_per_s": pps,
                    "kernel": "tile_sweep_kernel<NEED_DOT|NEED_EMD>, 64 slabs per row (u16 cumulative rows of bin - pseudo-count, "
                              "uint16 bins as a byte plane for tcgen05 kind::i8)",
                    "alu": {"algorithmic_warp_instr_per_pair": 65536 / 32.0, "achieved": pps * 65536 / 32.0 / 1e9,
                            "peak": probe / 1e9 if probe else None, "unit": "Gwarp-instr/s",
                            "frac": pps * 65536 / 32.0 / probe if probe else None},
                    "row_streaming_form": {"ms": ms_legacy, "pairs_per_s": r1["n_scored"] / (ms_legacy * 1e-3),
                                           "kernel": "sweep_wide_kernel<u16>", "same_counts": bool(r1["n_scored"] == r["n_scored"] and r1["n_out"] == r["n_out"])}}
    hs.free()
    sq.free()
    return out


def cfg5_block(ctx, capi, mdist, torch, comm, model, cutoff, local_rank, peak, n_total=1000000, n_queries=64, delta=5, dump=None):
    """BASELINE configs[4] in the same run: 1M x 1 kb (k = 5, uint8) histograms RANGE-PARTITIONED over the ranks (1 GiB in
    all), Trainer::get_close candidate scans of the accumulate stage (the query row broadcast from its owner, every rank
    scanning its shard with mc2_get_close, one triple per rank combined) and one update + merge pass of the update stage at
    --delta 5 over the replicated set (mc2_update_centers / mc2_merge_centers, centers split over the ranks).
    Histograms are generated directly (template rows + noise), bypassing FASTA, as SURVEY 8(d) allows for pair kernels.
    dump: a dict to receive the results of the last 16 scans and of the update pass (dump_scan_outputs)."""
    world, rank = comm.world, comm.rank
    per, bounds = mdist.shard_bounds(n_total, world)
    lo, hi = bounds[rank]
    N = 1024
    rng = np.random.default_rng([55, rank])
    trng = np.random.default_rng(55)
    base = trng.integers(1, 6, size=(10000, N), dtype=np.uint8)            # 10,000 templates x 100 variants
    tid = (np.arange(lo, hi) % 10000)
    H = base[tid]
    flip = rng.random(H.shape) < 0.02
    H = np.where(flip, np.clip(H.astype(np.int16) + rng.integers(-1, 2, size=H.shape), 1, 255).astype(np.uint8), H)
    ln = (950 + (tid * 7919) % 100).astype(np.uint64)
    eng = mdist.GpuEngine(capi, ctx, torch, model, 5, 1, local_rank)
    eng.local_hset = ctx.hset_from_host(H, 5, length=ln)
    eng.n_local, eng.per = hi - lo, per
    del H
    out = {"workload": WORKLOADS["cfg5"]["desc"], "n_sequences": n_total, "ranks": world}
    # accumulate-stage scans: n_queries get_close calls, each over all 1M candidates
    qs = [(q * 15485863) % n_total for q in range(n_queries)]
    for q in qs[:4]:
        mdist.candidate_scan(eng, comm, torch, q, n_total, cutoff)
    comm.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n_close = 0
    timed_best = []
    for q in qs:
        r = mdist.candidate_scan(eng, comm, torch, q, n_total, cutoff)
        n_close += int(np.count_nonzero(r["marks_local"]))
        if dump is not None:
            timed_best.append((r["best"], r["best_dist"], r["is_min"]))
    torch.cuda.synchronize()
    comm.barrier()
    dt = comm.all_reduce_max(time.perf_counter() - t0, torch, eng.device)
    if dump is not None:
        # a scan reuses its mark buffer, so the marks of the last step's scans come from scanning those queries again,
        # untimed; each repeat must return what the timed scan returned
        last = qs[-16:]
        mq, mc = [], []
        for t, q in enumerate(last):
            r = mdist.candidate_scan(eng, comm, torch, q, n_total, cutoff)
            assert (r["best"], r["best_dist"], r["is_min"]) == timed_best[len(qs) - len(last) + t], "get_close scan not repeatable"
            c = np.flatnonzero(r["marks_local"]) + lo
            mq.append(np.full(len(c), q))
            mc.append(c)
        got = timed_best[len(qs) - len(last):]
        dump.update(scan_q=last, scan_best=[g[0] for g in got], scan_best_dist=[g[1] for g in got],
                    scan_is_min=[g[2] for g in got], marks=(np.concatenate(mq), np.concatenate(mc)))
    out["candidate_scan"] = {"queries": n_queries, "candidates_per_query": n_total, "ms_per_query": dt / n_queries * 1e3,
                             "pairs_per_s": n_queries * n_total / dt, "achieved_gbs": n_queries * n_total * 1057 / dt / 1e9,
                             "frac_of_hbm_per_gpu": n_queries * n_total * 1057 / dt / 1e9 / (peak * world),
                             "timing": "host wall clock around the whole distributed call (broadcast + scan + combine), max over ranks",
                             "close_marks_rank0": n_close}
    # update stage: one pass over centers = every 100th point, members = the 2*delta+1 neighbouring clusters' points
    try:
        if world > 1:
            eng.full = None
            bins, length, mag = eng.export_local()
            bins = comm.all_gather_rows(bins, torch); length = comm.all_gather_rows(length, torch); mag = comm.all_gather_rows(mag, torch)
            eng.install_full(bins, length, mag, per * world)
            del bins
        else:
            eng.use_local_as_full()
        nfull = len(eng.full)
        per_cluster = 5
        nc = min(nfull // per_cluster, 20000)
        rows = np.arange(nc, dtype=np.uint64) * per_cluster
        off = np.zeros(nc + 1, dtype=np.uint64)
        mem = []
        for j in range(nc):
            a, b = max(0, j - delta) * per_cluster, min(nc, j + delta + 1) * per_cluster
            mem.append(np.arange(a, b, dtype=np.uint64))
            off[j + 1] = off[j] + np.uint64(b - a)
        members = np.concatenate(mem)
        side = eng.full.download(0, nc * per_cluster)                   # the centers' own magnitudes and lengths
        cm = side["mag"][::per_cluster].astype(np.uint64)
        cl = side["len"][::per_cluster].astype(np.uint64)
        del side
        mdist.update_pass(eng, comm, torch, rows, cm, cl, off, members, cutoff)
        comm.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        nxt, ng = mdist.update_pass(eng, comm, torch, rows, cm, cl, off, members, cutoff)
        mg = mdist.merge_pass(eng, comm, torch, rows, cm, cl, delta, cutoff)
        torch.cuda.synchronize(); comm.barrier()
        dtu = comm.all_reduce_max(time.perf_counter() - t0, torch, eng.device)
        if dump is not None:
            dump.update(update_next=nxt, update_n_good=ng, merge_choice=mg)
        out["update_stage"] = {"centers": int(nc), "delta": delta, "member_pairs": int(off[-1]), "merge_pairs": int(nc * delta),
                               "ms_per_pass": dtu * 1e3, "pairs_per_s": (int(off[-1]) + nc * delta) / dtu,
                               "moved": int(np.count_nonzero(nxt >= 0)), "merged": int(np.count_nonzero(mg > 0))}
    except Exception as e:
        log("[bench] cfg5 update stage failed: %r" % (e,))
    try:
        if eng.full is not None and eng.full is not eng.local_hset:
            eng.full.free()
        eng.local_hset.free()
    except Exception:
        pass
    return out


def gram_term_block(ctx, capi, hs, n_total, cutoff, nq=10000):
    """The Gram term sum p*q on the tensor pipe next to the CUDA-core form: a model over the three singles that need only
    that reduction (euclidean Feature.cpp:1112-1124, normalized_vectors :1170-1184, pearson :794-811) sweeps the first nq
    query rows of the bench's own histogram set twice -- tile_sweep_kernel (TMA + tcgen05.mma kind::i8 into TMEM) and, with
    MC2_SWEEP_LEGACY set for the call, sweep_kernel (IDP.4A from registers) -- device-timed, survivors compared."""
    singles = [(1 << 3, 0.0, 60.0), (1 << 5, 0.0, 1.0), (1 << 9, 0.0, 1.0)]        # Feature.h FEAT_TYPE bits of the three
    combos = [(0, [0]), (0, [1]), (0, [2])]
    nq = min(nq, n_total)
    # threshold: the 99.9th percentile of the summed normalised singles over a random pair sample (about 1 pair in 1000 close)
    rng = np.random.default_rng(9)
    probe = ctx.model(capi.make_desc(singles, combos, [0.0, 1.0, 1.0, 1.0]))
    ia = rng.integers(0, nq, 50000).astype(np.uint64)
    ib = rng.integers(0, n_total, 50000).astype(np.uint64)
    cache = ctx.score_pairs(probe, hs, hs, ia=ia, ib=ib, want=("cache",))["cache"]
    thr = float(np.quantile(cache.sum(axis=1), 0.999))
    gm = ctx.model(capi.make_desc(singles, combos, [-8.0 * thr, 8.0, 8.0, 8.0]))
    out = {"model": "euclidean + normalized_vectors + pearson (needs only sum p*q and the per-row side band)", "query_rows": nq,
           "database_rows": n_total}
    keep = {}
    for name, env in (("tensor_core_tile_sweep", None), ("cuda_core_sweep", "1")):
        if env:
            os.environ["MC2_SWEEP_LEGACY"] = env
        try:
            best = None
            for _ in range(3):
                ctx.timer_start()
                r = ctx.all_pairs(gm, hs, hs, cutoff, q_range=(0, nq), d_range=(0, n_total), upper_only=True, max_out=1 << 22)
                ms = ctx.timer_stop()
                best = ms if best is None else min(best, ms)
        finally:
            os.environ.pop("MC2_SWEEP_LEGACY", None)
        keep[name] = r
        out[name] = {"ms": best, "pairs_per_s": r["n_scored"] / (best * 1e-3), "pairs_scored": int(r["n_scored"]), "pairs_close": int(r["n_out"]),
                     "gram_int_ops_per_s": r["n_scored"] * 2 * 1024 / (best * 1e-3)}
    a, b = keep["tensor_core_tile_sweep"], keep["cuda_core_sweep"]
    sa = set(zip(a["q"].tolist(), a["d"].tolist()))
    sb = set(zip(b["q"].tolist(), b["d"].tolist()))
    out["same_survivors"] = bool(sa == sb and a["n_scored"] == b["n_scored"])
    out["speedup"] = out["cuda_core_sweep"]["ms"] / out["tensor_core_tile_sweep"]["ms"]
    return out


def slow_singles_block(ctx, capi, peak, n=1 << 18):
    """SURVEY 8 a8: the two "slow" singles (jefferey_divergence, jensen_shannon: per-bin fp64 logarithms, Feature.cpp:1230-1263,
    :983-1009) run pair_generic_kernel; one query vs 2^18 candidate rows, device-timed."""
    rng = np.random.default_rng(2)
    base = rng.integers(1, 7, size=(4096, 1024), dtype=np.uint8)
    H = base[rng.integers(0, 4096, n)]
    ln = rng.integers(950, 1050, n).astype(np.uint64)
    hs = ctx.hset_from_host(H, 5, length=ln)
    del H
    out = {}
    for name, flags in (("jefferey_divergence", [128]), ("jensen_shannon", [536870912]), ("both", [128, 536870912])):
        singles = [(f, 0.0, 1.0) for f in flags]
        combos = [(0, [i]) for i in range(len(flags))]
        gm = ctx.model(capi.make_desc(singles, combos, [0.5] + [-1.0] * len(flags)))
        for _ in range(2):
            ms, _nc = ctx.bench_score_pairs(gm, hs, hs, n_pairs=n, a_begin=0, b_begin=3, b_bc=1, iters=5, flush_l2=False)
        out[name] = {"ms": ms, "pairs_per_s": n / (ms * 1e-3), "log_evals_per_s": n * 1024 * (1 if name != "both" else 2) * (1 if name == "jefferey_divergence" else 2 if name == "jensen_shannon" else 1.5) / (ms * 1e-3),
                     "hbm_frac": n * 1057 / (ms * 1e-3) / 1e9 / peak}
    hs.free()
    out["kernel"] = "pair_generic_kernel<u8> (fp64 log per bin; bound by the fp64 / special-function pipes, not HBM)"
    out["candidates"] = n
    return out


def e2e_fastcar_block(n_query=500):
    """The second consumer of the path as the job it is: the reference's fastcar binary (oracle/_ref/fastcar) next to the
    same binary with ONE call added to work() (oracle/_ref/fastcar_b200, INTEGRATION.md section 3b): n_query sequences of
    the configs[1] set (10k x 1.5 kb) against all of it, classifier read from weights_cfg1_id90.txt (--recover), every host
    thread; wall clock of the whole process, output lines compared as sorted lists."""
    import tempfile
    from meshclust2_b200 import synth
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "fastcar")
    our_bin = os.path.join(ROOT, "oracle", "_ref", "fastcar_b200")
    if not (os.path.exists(ref_bin) and os.path.exists(our_bin)):
        return {"unavailable": "oracle/_ref fastcar binaries not built on this box"}
    seqs, tids, _, _ = synth.make_config_range("cfg2", 0, None)
    tmp = tempfile.mkdtemp()
    db, q = os.path.join(tmp, "db.fa"), os.path.join(tmp, "q.fa")
    open(db, "w").write(synth.to_fasta(seqs, tids))
    open(q, "w").write(synth.to_fasta(seqs[:n_query], tids[:n_query]))
    weights = os.path.join(ROOT, "tests", "golden", "weights_cfg1_id90.txt")
    threads = os.cpu_count() or 1
    res = {"workload": "fastcar: %d queries x %d database sequences of 1.5 kb, --id 0.9, --recover weights_cfg1_id90.txt, --threads %d; "
                       "whole process wall clock" % (n_query, len(seqs), threads)}
    lines = {}
    for name, binary in (("reference", ref_bin), ("b200", our_bin)):
        wd = os.path.join(tmp, name)
        os.makedirs(wd, exist_ok=True)
        t0 = time.time()
        r = subprocess.run([binary, db, "--query", q, "--id", "0.9", "--threads", str(threads), "--output", os.path.join(wd, "out"),
                            "--recover", weights], cwd=wd, capture_output=True, text=True, timeout=900)
        res[name + "_s"] = time.time() - t0
        res[name + "_rc"] = r.returncode
        if r.returncode != 0:
            res[name + "_tail"] = (r.stdout + r.stderr)[-300:]
            return res
        lines[name] = sorted(open(os.path.join(wd, "out0")).read().splitlines())
    res["output_lines"] = len(lines["reference"])
    res["identical_output"] = bool(lines["reference"] == lines["b200"])
    res["speedup"] = res["reference_s"] / res["b200_s"] if res["b200_s"] > 0 else None
    return res


def e2e_cluster_block(threads_list=None):
    """BASELINE configs[1] as the full job it names: the reference's own meshclust2 binary (oracle/_ref/meshclust2) next to
    the same binary relinked against this library (oracle/_ref/meshclust2_b200, INTEGRATION.md) on the 10k x 1.5 kb
    synthetic 16S-like FASTA at --id 0.9; wall clock of the whole process, clusters compared as sets."""
    import re
    import tempfile
    from meshclust2_b200 import synth
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "meshclust2")
    our_bin = os.path.join(ROOT, "oracle", "_ref", "meshclust2_b200")
    if not (os.path.exists(ref_bin) and os.path.exists(our_bin)):
        return {"unavailable": "oracle/_ref binaries not built on this box"}
    seqs, tids, _, _ = synth.make_config_range("cfg2", 0, None)
    tmp = tempfile.mkdtemp()
    fasta = os.path.join(tmp, "in.fa")
    open(fasta, "w").write(synth.to_fasta(seqs, tids))

    def clusters(path):
        out, cur = [], None
        for ln_ in open(path):
            if ln_.startswith(">Cluster"):
                cur = set()
                out.append(cur)
            else:
                m = re.search(r">(\S+)", ln_)
                if m:
                    cur.add(m.group(1).rstrip("."))
        return {frozenset(c) for c in out if c}

    res = {"workload": "meshclust2 --id 0.9 on 10k x 1.5 kb (BASELINE configs[1]), whole process wall clock", "runs": []}
    for threads in (threads_list or [os.cpu_count() or 1, 1]):
        got = {}
        for name, binary in (("reference", ref_bin), ("b200", our_bin)):
            wd = os.path.join(tmp, "%s_%d" % (name, threads))
            os.makedirs(wd, exist_ok=True)
            outp = os.path.join(wd, "out.clstr")
            t0 = time.time()
            r = subprocess.run([binary, "--id", "0.9", "--threads", str(threads), fasta, "--output", outp], cwd=wd,
                               capture_output=True, text=True, timeout=600)
            got[name] = (time.time() - t0, r.returncode, clusters(outp) if r.returncode == 0 else None)
        same = got["reference"][2] is not None and got["reference"][2] == got["b200"][2]
        res["runs"].append({"threads": threads, "reference_s": got["reference"][0], "b200_s": got["b200"][0],
                            "rc": [got["reference"][1], got["b200"][1]],
                            "clusters": len(got["reference"][2]) if got["reference"][2] is not None else None,
                            "identical_clusters": bool(same),
                            "note": None if threads == 1 else "the reference's OpenMP training is not reproducible run to run "
                                                              "(SURVEY section 4): identical clusters are asserted at --threads 1"})
    return res


def candidates_roofline(ctx, capi, model, k, eb, peak, peak_src, n=1 << 20):
    """The HBM-streaming form (Trainer::get_close over a long candidate range, BASELINE configs[4] shape):
    one query vs 2^20 candidate histograms (1 GiB > L2), device-timed per launch."""
    rng = np.random.default_rng(1)
    N = 4 ** k
    base = rng.integers(1, 7, size=(4096, N), dtype=np.uint8)
    H = base[rng.integers(0, 4096, n)]
    ln = rng.integers(950, 1050, n).astype(np.uint64)
    hs = ctx.hset_from_host(H, k, length=ln)
    del H
    ms, nclose = ctx.bench_score_pairs(model, hs, hs, n_pairs=n, a_begin=0, b_begin=3, b_bc=1, iters=20, flush_l2=False,
                                       len_filter=1, anchor_is_b=1, cutoff=0.9)
    ms, nclose = ctx.bench_score_pairs(model, hs, hs, n_pairs=n, a_begin=0, b_begin=3, b_bc=1, iters=20, flush_l2=False,
                                       len_filter=1, anchor_is_b=1, cutoff=0.9)
    hs.free()
    bpp = N * eb + 24 + 9
    ach = n * bpp / (ms * 1e-3) / 1e9
    tpp, tsrc = traffic_per_pair("pair_fast_kernel")
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "traffic": tpp * n if tpp else None, "traffic_source": tsrc,
            "kernel": "pair_fast_kernel<u8> one query vs 2^20 candidates (1 GiB streamed, > L2)",
            "algorithmic_bytes_per_unit": bpp, "units_per_launch": n, "avg_launch_ms": ms, "pairs_per_s": n / (ms * 1e-3),
            "peak_source": peak_src}


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else libraries print to fd 1 (e.g. NCCL's version banner)
    has been redirected to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--n-seqs", dest="n", type=int, default=None, help="override the number of sequences (smoke runs)")
    ap.add_argument("--blocks-per-rank", type=int, default=1, help="contiguous equal-pair-count query-row ranges (= sweep launches) per rank and step")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--cpu-hist-sample", type=int, default=100000)
    ap.add_argument("--cpu-pair-sample", type=int, default=20000000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs covers the timed device path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3 and args.impl == "ours":
        log("[bench] note: W >= 3 warm-up steps are required for a valid number")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
