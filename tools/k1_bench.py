"""K1 timings (development aid): cfg3-shaped short reads and cfg4-shaped long multi-segment records."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from meshclust2_b200 import capi, synth
ctx = capi.Context(0)
def run(name, seqs, k, eb, iters=10):
    enc = capi.encode_batch(seqs)
    sq = ctx.upload_seqs(enc["codes"], enc["seq_off"], enc["segs"], enc["seg_off"])
    L = sum(len(s) for s in seqs) / len(seqs)
    ms = ctx.bench_count_kmers(sq, k, eb, iters=iters, flush_l2=True)
    ms = ctx.bench_count_kmers(sq, k, eb, iters=iters, flush_l2=True)
    byts = len(seqs) * (L / 4 + 4 ** k * eb + 40)
    print("%-28s n=%d L=%.0f k=%d eb=%d: %.3f ms  %.3e hist/s  %.3e kmers/s  %.0f GB/s (%.1f%% of 6540)" % (
        name, len(seqs), L, k, eb, ms, len(seqs) / ms * 1e3, len(seqs) * L / ms * 1e3, byts / ms / 1e6, byts / ms / 1e6 / 65.4))
seqs, _, k, eb = synth.make_config_range("cfg3", 0, int(os.environ.get("K1_N", 100000)))
for legacy in (False, True):
    if legacy:
        os.environ["MC2_K1_LEGACY"] = "1"   # count_kernel (the generic form) instead of count_warp_kernel
    else:
        os.environ.pop("MC2_K1_LEGACY", None)
    tag = " [generic kernel]" if legacy else ""
    run("cfg3 short reads" + tag, seqs, 5, 1)
    run("cfg3 short reads u16" + tag, seqs, 5, 2)
    run("cfg3 short reads k=6" + tag, seqs, 6, 1)
os.environ.pop("MC2_K1_LEGACY", None)
if os.environ.get("K1_SHORT"):
    sys.exit(0)
long_ = synth.make_single_file(int(os.environ.get("K1_LONG_N", 500)), 5, 10000, seed=4)
run("cfg4 long records", long_, 8, 2, iters=3)
run("long records k=7", long_, 7, 2, iters=3)
run("long records k=5", long_, 5, 1, iters=3)
if os.environ.get("K1_NO_INGEST"):
    sys.exit(0)
# input contract on the device (mc2_seqs_from_text) vs host encode + upload, cfg3 shape
import time
blob = b"".join(seqs)
off = np.zeros(len(seqs) + 1, dtype=np.uint64); off[1:] = np.cumsum([len(s) for s in seqs])
buf = capi.host_register(np.frombuffer(bytearray(blob), dtype=np.uint8))
for name, fn in (("device ingest (text -> packed + segments)", lambda: ctx.seqs_from_text((buf, off)).free()),
                 ("host encode (16 threads) + upload", lambda: (lambda e: ctx.upload_seqs(e["codes"], e["seq_off"], e["segs"], e["seg_off"]).free())(capi.encode_batch(seqs, threads=16)))):
    fn(); fn()
    t0 = time.perf_counter()
    for _ in range(5):
        fn()
    ctx.sync()
    dt = (time.perf_counter() - t0) / 5
    print("%-45s %.2f ms for %d sequences, %.1f Mbases -> %.2f Gbases/s" % (name, dt * 1e3, len(seqs), len(blob) / 1e6, len(blob) / dt / 1e9))
