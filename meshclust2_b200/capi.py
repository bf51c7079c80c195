"""ctypes binding of the C ABI in include/meshclust2_b200.h (lib/libmeshclust2_b200.so).

This is the Python face of the drop-in boundary: thin wrappers, numpy in / numpy out, no compute.
There is no CPU fallback — if the CUDA library is missing or no sm_100 device is present every
entry point raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MC2_LIB") or os.path.join(_HERE, "lib", "libmeshclust2_b200.so")   # MC2_LIB: tuning variants

MAX_SINGLES, MAX_COMBOS, MAX_COMBO_IDX = 16, 16, 4
DTYPES = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}

FEAT_MANHATTAN = 1 << 2
FEAT_EUCLIDEAN = 1 << 3
FEAT_NORMALIZED_VECTORS = 1 << 5
FEAT_JEFFEREY_DIV = 1 << 7
FEAT_PEARSON_COEFF = 1 << 9
FEAT_INTERSECTION = 1 << 13
FEAT_EMD = 1 << 18
FEAT_LENGTHD = 1 << 21
FEAT_KULCZYNSKI2 = 1 << 27
FEAT_SIMRATIO = 1 << 28
FEAT_JENSEN_SHANNON = 1 << 29
PRED_FEAT_FAST = (FEAT_EUCLIDEAN | FEAT_MANHATTAN | FEAT_INTERSECTION | FEAT_KULCZYNSKI2 | FEAT_SIMRATIO |
                  FEAT_NORMALIZED_VECTORS | FEAT_PEARSON_COEFF | FEAT_EMD | FEAT_LENGTHD)
PRED_FEAT_DIV = FEAT_JEFFEREY_DIV | FEAT_JENSEN_SHANNON

# every symbol include/meshclust2_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "mc2_abi_version", "mc2_last_error", "mc2_device_count", "mc2_ctx_create", "mc2_ctx_destroy", "mc2_ctx_sync",
    "mc2_ctx_device", "mc2_ctx_sm_count", "mc2_ctx_stream", "mc2_timer_start", "mc2_timer_stop",
    "mc2_ctx_launch_count", "mc2_ctx_profile", "mc2_ctx_kernel_time", "mc2_ctx_flush_l2", "mc2_seqs_upload", "mc2_seqs_upload_into", "mc2_seqs_from_text", "mc2_seqs_from_text_into", "mc2_seqs_download_segments", "mc2_seqs_total_segments", "mc2_host_register", "mc2_host_unregister", "mc2_seqs_free", "mc2_seqs_count",
    "mc2_seqs_total_bases", "mc2_count_kmers", "mc2_count_kmers_into", "mc2_count_kmers_auto", "mc2_hset_largest_count", "mc2_hset_alloc", "mc2_count_kmers_into_rows", "mc2_hset_refresh", "mc2_width_for_count", "mc2_kmer_table_increment", "mc2_hset_from_host", "mc2_hset_from_device", "mc2_hset_update_from_device", "mc2_hset_device_sideband", "mc2_hset_free",
    "mc2_hset_count", "mc2_hset_k", "mc2_hset_elem_bytes", "mc2_hset_device_bins", "mc2_hset_download", "mc2_hset_copy_to_device",
    "mc2_hset_set_sideband", "mc2_hset_set_row", "mc2_hset_assign_rows", "mc2_hset_reverse_complement", "mc2_model_create", "mc2_model_free", "mc2_model_desc_from_file",
    "mc2_score_pairs", "mc2_get_close", "mc2_get_close_as", "mc2_filter", "mc2_filter_as", "mc2_merge", "mc2_all_pairs", "mc2_identity_pairs", "mc2_identity_pairs_both_strands", "mc2_identity_topk", "mc2_debug_tile_reductions", "mc2_debug_last_sweep", "mc2_distance", "mc2_mean_closest", "mc2_closest",
    "mc2_update_centers", "mc2_merge_centers",
    "mc2_bench_score_pairs", "mc2_bench_count_kmers", "mc2_bench_issue_rate", "mc2_encode_dna", "mc2_encode_dna_batch",
]


class Mc2Error(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("mc2 status %d: %s" % (status, msg))
        self.status = status


class ModelDesc(C.Structure):
    _fields_ = [
        ("n_singles", C.c_int32),
        ("single_flag", C.c_uint64 * MAX_SINGLES),
        ("single_min", C.c_double * MAX_SINGLES),
        ("single_max", C.c_double * MAX_SINGLES),
        ("n_combos", C.c_int32),
        ("combo_kind", C.c_int32 * MAX_COMBOS),
        ("combo_nidx", C.c_int32 * MAX_COMBOS),
        ("combo_idx", (C.c_int32 * MAX_COMBO_IDX) * MAX_COMBOS),
        ("weight", C.c_double * (MAX_COMBOS + 1)),
        ("bias", C.c_double),
        ("regression", C.c_int32),
    ]


class Pairs(C.Structure):
    _fields_ = [
        ("set_a", C.c_void_p), ("set_b", C.c_void_p), ("n_pairs", C.c_uint64),
        ("ia", C.c_void_p), ("ib", C.c_void_p),
        ("a_begin", C.c_uint64), ("b_begin", C.c_uint64),
        ("a_broadcast", C.c_int32), ("b_broadcast", C.c_int32),
        ("len_filter", C.c_int32), ("anchor_is_b", C.c_int32),
        ("cutoff", C.c_double),
        ("bc_override", C.c_int32), ("reserved_", C.c_int32), ("bc_mag", C.c_uint64), ("bc_len", C.c_uint64),
    ]


_lib = None


def lib():
    """Load the CUDA library; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(meshclust2_b200 has no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.mc2_last_error.restype = C.c_char_p
        L.mc2_ctx_stream.restype = C.c_void_p
        L.mc2_ctx_launch_count.restype = C.c_uint64
        L.mc2_seqs_count.restype = C.c_uint64
        L.mc2_seqs_total_bases.restype = C.c_uint64
        L.mc2_seqs_total_segments.restype = C.c_uint64
        L.mc2_hset_count.restype = C.c_uint64
        L.mc2_hset_device_bins.restype = C.c_void_p
        L.mc2_hset_device_sideband.restype = C.c_void_p
        L.mc2_ctx_flush_l2.argtypes = [C.c_void_p, C.c_size_t]
        L.mc2_identity_pairs.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                                         C.c_uint64, C.c_uint64, C.c_int32, C.c_double, C.c_uint64, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
        L.mc2_identity_pairs_both_strands.argtypes = (L.mc2_identity_pairs.argtypes[:15] + [C.c_void_p]
                                                      + L.mc2_identity_pairs.argtypes[15:])
        L.mc2_identity_topk.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint64,
                                        C.c_void_p, C.c_uint64, C.c_uint64, C.c_int32, C.c_int32, C.c_double, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise Mc2Error(rc, lib().mc2_last_error().decode(errors="replace"))


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _u64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.uint64)


def device_count():
    return lib().mc2_device_count()


class Context:
    def __init__(self, device=0):
        self.h = C.c_void_p()
        _check(lib().mc2_ctx_create(device, C.byref(self.h)))

    def close(self):
        if self.h:
            lib().mc2_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        _check(lib().mc2_ctx_sync(self.h))

    @property
    def sm_count(self):
        return lib().mc2_ctx_sm_count(self.h)

    @property
    def launches(self):
        return lib().mc2_ctx_launch_count(self.h)

    def stream(self):
        return lib().mc2_ctx_stream(self.h)

    def timer_start(self):
        _check(lib().mc2_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        _check(lib().mc2_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def profile(self, enable=True):
        _check(lib().mc2_ctx_profile(self.h, int(enable)))

    def kernel_time(self, kind):
        """kind: 0 pack, 1 count, 2 pair score, 3 sweep, 4 argmax, 5 side-band -> (total_ms, launches)"""
        ms, n = C.c_double(), C.c_uint64()
        _check(lib().mc2_ctx_kernel_time(self.h, kind, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def flush_l2(self, nbytes=256 << 20):
        _check(lib().mc2_ctx_flush_l2(self.h, nbytes))

    # ---- K1 ----
    def upload_seqs(self, codes, seq_off, segs, seg_off):
        """codes: int8/uint8 concatenated; seq_off uint64[n+1]; segs int32[total,2] sequence-relative inclusive;
        seg_off uint64[n+1]."""
        codes = np.ascontiguousarray(codes).view(np.int8)
        seq_off = _u64(seq_off)
        seg_off = _u64(seg_off)
        segs = np.ascontiguousarray(segs, dtype=np.int32)
        out = C.c_void_p()
        _check(lib().mc2_seqs_upload(self.h, _p(codes), _p(seq_off), C.c_uint64(len(seq_off) - 1), _p(segs),
                                     _p(seg_off), C.byref(out)))
        return Seqs(self, out)

    def seqs_from_text(self, seqs):
        """raw nucleotide text (list of bytes, or (blob, offsets)) -> Seqs, segmentation + encoding + packing on the device"""
        if isinstance(seqs, tuple):
            blob, off = seqs
            off = _u64(off)
        else:
            off = np.zeros(len(seqs) + 1, dtype=np.uint64)
            off[1:] = np.cumsum([len(s) for s in seqs])
            blob = b"".join(seqs)
        buf = np.frombuffer(blob, dtype=np.uint8) if len(blob) else np.zeros(1, dtype=np.uint8)
        out = C.c_void_p()
        _check(lib().mc2_seqs_from_text(self.h, _p(buf), _p(off), C.c_uint64(len(off) - 1), C.byref(out)))
        return Seqs(self, out)

    def seqs_from_text_into(self, dst, blob, off):
        """refill `dst` from raw text: blob = uint8 array (may be page-locked), off = uint64[n+1]"""
        off = _u64(off)
        _check(lib().mc2_seqs_from_text_into(self.h, dst.h, _p(blob), _p(off), C.c_uint64(len(off) - 1)))
        return dst

    def upload_seqs_into(self, dst, codes, seq_off, segs, seg_off):
        """refill `dst` (a Seqs of this context) with another batch, reusing its device arrays"""
        codes = np.ascontiguousarray(codes).view(np.int8)
        seq_off = _u64(seq_off)
        seg_off = _u64(seg_off)
        segs = np.ascontiguousarray(segs, dtype=np.int32)
        _check(lib().mc2_seqs_upload_into(self.h, dst.h, _p(codes), _p(seq_off), C.c_uint64(len(seq_off) - 1), _p(segs),
                                          _p(seg_off)))
        return dst

    def count_kmers_auto(self, seqs, k):
        """width detection fused with counting -> (HistSet, largest_count, elem_bytes)"""
        out = C.c_void_p()
        largest, eb = C.c_uint64(), C.c_int()
        _check(lib().mc2_count_kmers_auto(self.h, seqs.h, k, C.byref(largest), C.byref(eb), C.byref(out)))
        return HistSet(self, out), largest.value, eb.value

    def count_kmers(self, seqs, k, elem_bytes):
        out = C.c_void_p()
        _check(lib().mc2_count_kmers(self.h, seqs.h, k, elem_bytes, C.byref(out)))
        return HistSet(self, out)

    def count_kmers_into(self, seqs, hset):
        _check(lib().mc2_count_kmers_into(self.h, seqs.h, hset.h))
        return hset

    def kmer_table_increment(self, codes, first, last, k, elem_bytes, init=1):
        codes = np.ascontiguousarray(codes).view(np.int8)
        vals = np.zeros(4 ** k, dtype=DTYPES[elem_bytes])
        ret = C.c_int32()
        _check(lib().mc2_kmer_table_increment(self.h, _p(codes), first, last, k, elem_bytes, C.c_uint64(init),
                                              _p(vals), C.byref(ret)))
        return vals, ret.value

    def hset_from_host(self, bins, k, mag=None, length=None):
        bins = np.ascontiguousarray(bins)
        n = bins.shape[0]
        assert bins.ndim == 2 and bins.shape[1] == 4 ** k
        length = _u64(length if length is not None else np.ones(n))
        mag = _u64(mag)
        out = C.c_void_p()
        _check(lib().mc2_hset_from_host(self.h, _p(bins), C.c_uint64(n), k, bins.dtype.itemsize, _p(mag), _p(length),
                                        C.byref(out)))
        return HistSet(self, out)

    def hset_alloc(self, n, k, elem_bytes):
        """an n-row set with zeroed rows, to be filled by count_kmers_into_rows / a collective + refresh()"""
        out = C.c_void_p()
        _check(lib().mc2_hset_alloc(self.h, C.c_uint64(n), k, elem_bytes, C.byref(out)))
        return HistSet(self, out)

    def count_kmers_into_rows(self, seqs, hset, first_row):
        _check(lib().mc2_count_kmers_into_rows(self.h, seqs.h, hset.h, C.c_uint64(first_row)))

    def hset_from_device(self, d_bins, n, k, elem_bytes, d_len, d_mag=None):
        """d_bins / d_len / d_mag: raw device pointers (ints), e.g. torch_tensor.data_ptr()"""
        out = C.c_void_p()
        _check(lib().mc2_hset_from_device(self.h, C.c_void_p(d_bins), C.c_uint64(n), k, elem_bytes,
                                          C.c_void_p(d_mag) if d_mag else None, C.c_void_p(d_len), C.byref(out)))
        return HistSet(self, out)

    def model(self, desc):
        out = C.c_void_p()
        _check(lib().mc2_model_create(self.h, C.byref(desc), C.byref(out)))
        return Model(self, out, desc)

    def model_from_file(self, path, which=0):
        desc, meta = model_desc_from_file(path, which)
        m = self.model(desc)
        m.meta = meta
        return m

    # ---- K2 ----
    def _pairs(self, set_a, set_b, ia, ib, n_pairs, a_begin=0, b_begin=0, a_bc=0, b_bc=0, len_filter=0,
               anchor_is_b=0, cutoff=0.0):
        ia = _u64(ia)
        ib = _u64(ib)
        p = Pairs(set_a.h.value, set_b.h.value, n_pairs, ia.ctypes.data if ia is not None else None,
                  ib.ctypes.data if ib is not None else None, a_begin, b_begin, a_bc, b_bc, len_filter, anchor_is_b,
                  cutoff)
        p._keep = (ia, ib)
        return p

    def score_pairs(self, model, set_a, set_b, ia=None, ib=None, n_pairs=None, a_begin=0, b_begin=0, a_bc=0, b_bc=0,
                    len_filter=0, anchor_is_b=0, cutoff=0.0, want=("score", "dist", "close", "cache", "raw", "skipped")):
        if n_pairs is None:
            n_pairs = len(ia) if ia is not None else len(ib)
        p = self._pairs(set_a, set_b, ia, ib, n_pairs, a_begin, b_begin, a_bc, b_bc, len_filter, anchor_is_b, cutoff)
        S = model.desc.n_singles
        out = {}
        out["score"] = np.zeros(n_pairs) if "score" in want else None
        out["dist"] = np.zeros(n_pairs) if "dist" in want else None
        out["close"] = np.zeros(n_pairs, dtype=np.uint8) if "close" in want else None
        out["cache"] = np.zeros((n_pairs, S)) if "cache" in want else None
        out["raw"] = np.zeros((n_pairs, S)) if "raw" in want else None
        out["skipped"] = np.zeros(n_pairs, dtype=np.uint8) if "skipped" in want else None
        _check(lib().mc2_score_pairs(self.h, model.h, C.byref(p), _p(out["score"]), _p(out["dist"]), _p(out["close"]),
                                     _p(out["cache"]), _p(out["raw"]), _p(out["skipped"])))
        return out

    def get_close(self, model, set_q, q, set_c, cand=None, cand_begin=0, n_cand=None, cutoff=0.9, marks=None):
        """marks: optional uint8 buffer of >= n_cand bytes to fill (e.g. page-locked and reused across calls); its first n_cand
        bytes are returned"""
        cand = _u64(cand)
        if n_cand is None:
            n_cand = len(cand)
        best, bd, ismin = C.c_int64(), C.c_double(), C.c_int32()
        if marks is None:
            marks = np.zeros(n_cand, dtype=np.uint8)
        else:
            assert marks.dtype == np.uint8 and marks.flags.c_contiguous and len(marks) >= n_cand
            marks = marks[:n_cand]
        _check(lib().mc2_get_close(self.h, model.h, set_q.h, C.c_uint64(q), set_c.h, _p(cand), C.c_uint64(cand_begin),
                                   C.c_uint64(n_cand), C.c_double(cutoff), C.byref(best), C.byref(bd), C.byref(ismin),
                                   _p(marks)))
        return best.value, bd.value, bool(ismin.value), marks

    def get_close_as(self, model, set_q, q, q_mag, q_len, set_c, cand=None, cand_begin=0, n_cand=None, cutoff=0.9):
        """get_close for a center = row q of set_q reporting (q_mag, q_len) as its side-band"""
        cand = _u64(cand)
        if n_cand is None:
            n_cand = len(cand)
        best, bd, ismin = C.c_int64(), C.c_double(), C.c_int32()
        marks = np.zeros(n_cand, dtype=np.uint8)
        _check(lib().mc2_get_close_as(self.h, model.h, set_q.h, C.c_uint64(q), C.c_uint64(q_mag), C.c_uint64(q_len), set_c.h,
                                      _p(cand), C.c_uint64(cand_begin), C.c_uint64(n_cand), C.c_double(cutoff), C.byref(best),
                                      C.byref(bd), C.byref(ismin), _p(marks)))
        return best.value, bd.value, bool(ismin.value), marks

    def filter_as(self, model, set_c, center, c_mag, c_len, set_m, members, ident):
        members = _u64(members)
        keep = np.zeros(len(members), dtype=np.uint8)
        _check(lib().mc2_filter_as(self.h, model.h, set_c.h, C.c_uint64(center), C.c_uint64(c_mag), C.c_uint64(c_len), set_m.h,
                                   _p(members), C.c_uint64(len(members)), C.c_double(ident), _p(keep)))
        return keep

    def filter(self, model, set_c, center, set_m, members, ident):
        members = _u64(members)
        keep = np.zeros(len(members), dtype=np.uint8)
        _check(lib().mc2_filter(self.h, model.h, set_c.h, C.c_uint64(center), set_m.h, _p(members),
                                C.c_uint64(len(members)), C.c_double(ident), _p(keep)))
        return keep

    def merge(self, model, centers, rows, cur, begin, last, ident):
        rows = _u64(rows)
        out = C.c_int64()
        _check(lib().mc2_merge(self.h, model.h, centers.h, _p(rows), C.c_int64(cur), C.c_int64(begin), C.c_int64(last),
                               C.c_double(ident), C.byref(out)))
        return out.value

    def all_pairs(self, model, set_q, set_d, cutoff, q_range=None, d_range=None, upper_only=False, max_out=1 << 20, out=None):
        """out: optional (q uint64[max_out], d uint64[max_out], score float64[max_out]) buffers to fill (e.g. page-locked and
        reused across calls); the returned arrays are then views of them"""
        q0, q1 = q_range if q_range else (0, len(set_q))
        d0, d1 = d_range if d_range else (0, len(set_d))
        if out is not None:
            oq, od, osc = out
            assert len(oq) >= max_out and len(od) >= max_out and len(osc) >= max_out
        else:
            oq = np.empty(max_out, dtype=np.uint64)
            od = np.empty(max_out, dtype=np.uint64)
            osc = np.empty(max_out)
        n_out, n_scored = C.c_uint64(), C.c_uint64()
        _check(lib().mc2_all_pairs(self.h, model.h, set_q.h, C.c_uint64(q0), C.c_uint64(q1), set_d.h, C.c_uint64(d0),
                                   C.c_uint64(d1), int(upper_only), C.c_double(cutoff), C.c_uint64(max_out), _p(oq),
                                   _p(od), _p(osc), C.byref(n_out), C.byref(n_scored)))
        got = min(n_out.value, max_out)
        return dict(q=oq[:got], d=od[:got], score=osc[:got], n_out=n_out.value, n_scored=n_scored.value)

    def identity_pairs(self, model, set_q, set_d, min_identity, cutoff, q_range=None, d_range=None, upper_only=False,
                       max_out=1 << 20, out=None):
        """Identity search with a regression model: the in-window pairs of all_pairs whose predicted identity (the GLM sum
        clamped to [0, 1]) is >= min_identity, with that identity.  out: optional (q, d, identity) buffers as in all_pairs."""
        q0, q1 = q_range if q_range else (0, len(set_q))
        d0, d1 = d_range if d_range else (0, len(set_d))
        if out is not None:
            oq, od, oid = out
            assert len(oq) >= max_out and len(od) >= max_out and len(oid) >= max_out
        else:
            oq = np.empty(max_out, dtype=np.uint64)
            od = np.empty(max_out, dtype=np.uint64)
            oid = np.empty(max_out)
        n_out, n_scored = C.c_uint64(), C.c_uint64()
        _check(lib().mc2_identity_pairs(self.h, model.h, min_identity, set_q.h, q0, q1, set_d.h, d0, d1, int(upper_only), cutoff,
                                        max_out, _p(oq), _p(od), _p(oid), C.byref(n_out), C.byref(n_scored)))
        got = min(n_out.value, max_out)
        return dict(q=oq[:got], d=od[:got], identity=oid[:got], n_out=n_out.value, n_scored=n_scored.value)

    def identity_pairs_both_strands(self, model, set_q, set_d, min_identity, cutoff, q_range=None, d_range=None,
                                    upper_only=False, max_out=1 << 20, out=None):
        """identity_pairs on both strands of each query: a pair survives when the larger of its forward identity and its
        identity against the query's reverse complement is >= min_identity.  Returns identity_pairs' dict plus `strand`
        (int8: 0 forward, 1 reverse; ties go to forward).  out: optional (q, d, identity, strand) buffers."""
        q0, q1 = q_range if q_range else (0, len(set_q))
        d0, d1 = d_range if d_range else (0, len(set_d))
        if out is not None:
            oq, od, oid, ostr = out
            assert min(len(oq), len(od), len(oid), len(ostr)) >= max_out
        else:
            oq = np.empty(max_out, dtype=np.uint64)
            od = np.empty(max_out, dtype=np.uint64)
            oid = np.empty(max_out)
            ostr = np.empty(max_out, dtype=np.int8)
        n_out, n_scored = C.c_uint64(), C.c_uint64()
        _check(lib().mc2_identity_pairs_both_strands(self.h, model.h, min_identity, set_q.h, q0, q1, set_d.h, d0, d1,
                                                     int(upper_only), cutoff, max_out, _p(oq), _p(od), _p(oid), _p(ostr),
                                                     C.byref(n_out), C.byref(n_scored)))
        got = min(n_out.value, max_out)
        return dict(q=oq[:got], d=od[:got], identity=oid[:got], strand=ostr[:got], n_out=n_out.value,
                    n_scored=n_scored.value)

    def identity_topk(self, model, set_q, set_d, min_identity, k_best, cutoff, q_range=None, d_range=None, upper_only=False,
                      exclude_self=False, out=None):
        """Each query's k_best best identity_pairs hits, ordered by identity descending then database row ascending.
        exclude_self also drops the pair (r, r) (set_q must be set_d).  Returns dict(d=uint64[nq, K], identity=[nq, K],
        count=uint32[nq], n_hits=uint64[nq], n_scored); unused slots hold d = 2^64 - 1 and identity -1.0.
        out: optional (d, identity, count, n_hits) arrays of those shapes to fill (e.g. page-locked and reused)."""
        q0, q1 = q_range if q_range else (0, len(set_q))
        d0, d1 = d_range if d_range else (0, len(set_d))
        nq = max(q1 - q0, 0)
        if out is not None:
            od, oid, cnt, hits = out
            assert od.shape == oid.shape == (nq, k_best) and cnt.shape == hits.shape == (nq,)
            assert od.dtype == np.uint64 and oid.dtype == np.float64 and cnt.dtype == np.uint32 and hits.dtype == np.uint64
        else:
            od = np.empty((nq, k_best), dtype=np.uint64)
            oid = np.empty((nq, k_best))
            cnt = np.empty(nq, dtype=np.uint32)
            hits = np.empty(nq, dtype=np.uint64)
        n_scored = C.c_uint64()
        _check(lib().mc2_identity_topk(self.h, model.h, min_identity, k_best, set_q.h, q0, q1, set_d.h, d0, d1, int(upper_only),
                                       int(exclude_self), cutoff, _p(od), _p(oid), _p(cnt), _p(hits), C.byref(n_scored)))
        return dict(d=od, identity=oid, count=cnt, n_hits=hits, n_scored=n_scored.value)

    def issue_rate(self, iters=100000):
        """measured warp-instructions / s of the VIMNMX.U16x2 + IDP.2A pair (roofline denominator of the tile sweep)"""
        out = C.c_double()
        _check(lib().mc2_bench_issue_rate(self.h, int(iters), C.byref(out)))
        return out.value

    def tile_reductions(self, set_q, set_d, need, q_range=None, d_range=None):
        """Diagnostic: dense uint32 matrices {sad, dot, emd} (those in `need`: 1 | 2 | 4) of the tile sweep's reductions"""
        q0, q1 = q_range if q_range else (0, len(set_q))
        d0, d1 = d_range if d_range else (0, len(set_d))
        shape = (q1 - q0, d1 - d0)
        out = {k: np.zeros(shape, dtype=np.uint32) for k, bit in (("sad", 1), ("dot", 2), ("emd", 4)) if need & bit}
        _check(lib().mc2_debug_tile_reductions(self.h, set_q.h, C.c_uint64(q0), C.c_uint64(q1), set_d.h, C.c_uint64(d0),
                                               C.c_uint64(d1), int(need), _p(out["dot"]) if "dot" in out else None,
                                               _p(out["emd"]) if "emd" in out else None, _p(out["sad"]) if "sad" in out else None))
        return out

    def last_sweep(self):
        """Diagnostic: {n_exact, coarse} of the last all_pairs / identity_pairs call -- the pairs the tile sweep sent
        through the exact epilogue, and whether it took the coarse form"""
        n, c = C.c_uint64(), C.c_int32()
        _check(lib().mc2_debug_last_sweep(self.h, C.byref(n), C.byref(c)))
        return dict(n_exact=n.value, coarse=bool(c.value))

    def distance(self, set_a, set_b, ia, ib):
        p = self._pairs(set_a, set_b, ia, ib, len(ia))
        out = np.zeros(len(ia), dtype=np.uint64)
        _check(lib().mc2_distance(self.h, C.byref(p), _p(out)))
        return out

    def mean_closest(self, hset, members):
        """K3: (best position in members, its distance_d, mean[4^k], dist[n])"""
        members = _u64(members)
        best, bd = C.c_int64(), C.c_double()
        mean = np.zeros(4 ** hset.k)
        dist = np.zeros(len(members))
        _check(lib().mc2_mean_closest(self.h, hset.h, _p(members), C.c_uint64(len(members)), C.byref(best), C.byref(bd),
                                      _p(mean), _p(dist)))
        return best.value, bd.value, mean, dist

    def update_centers(self, model, centers, n_centers, set_m, member_off, members, ident):
        """Batched mean_shift_update: (next position per center or -1, survivors per center)"""
        member_off, members = _u64(member_off), _u64(members)
        nxt = np.zeros(n_centers, dtype=np.int64)
        ng = np.zeros(n_centers, dtype=np.uint64)
        _check(lib().mc2_update_centers(self.h, model.h, centers.h, C.c_uint64(n_centers), set_m.h, _p(member_off), _p(members),
                                        C.c_double(ident), _p(nxt), _p(ng)))
        return nxt, ng

    def merge_centers(self, model, centers, n_centers, delta, ident):
        """Batched Trainer::merge: chosen center index per center, 0 when none is close"""
        out = np.zeros(n_centers, dtype=np.int64)
        _check(lib().mc2_merge_centers(self.h, model.h, centers.h, C.c_uint64(n_centers), C.c_int64(delta), C.c_double(ident),
                                       _p(out)))
        return out

    def closest(self, hset, members, mean):
        """Trainer::closest: (best position, distance, dist[n]) against a caller-supplied double mean"""
        members = _u64(members)
        mean = np.ascontiguousarray(mean, dtype=np.float64)
        best, bd = C.c_int64(), C.c_double()
        dist = np.zeros(len(members))
        _check(lib().mc2_closest(self.h, hset.h, _p(members), C.c_uint64(len(members)), _p(mean), C.byref(best), C.byref(bd),
                                 _p(dist)))
        return best.value, bd.value, dist

    def bench_score_pairs(self, model, set_a, set_b, ia=None, ib=None, n_pairs=None, iters=10, flush_l2=True, **kw):
        if n_pairs is None:
            n_pairs = len(ia) if ia is not None else len(ib)
        p = self._pairs(set_a, set_b, ia, ib, n_pairs, **kw)
        ms, nc = C.c_float(), C.c_uint64()
        _check(lib().mc2_bench_score_pairs(self.h, model.h, C.byref(p), iters, int(flush_l2), C.byref(ms), C.byref(nc)))
        return ms.value, nc.value

    def bench_count_kmers(self, seqs, k, elem_bytes, iters=10, flush_l2=True):
        ms = C.c_float()
        _check(lib().mc2_bench_count_kmers(self.h, seqs.h, k, elem_bytes, iters, int(flush_l2), C.byref(ms)))
        return ms.value


def host_register(arr):
    """page-lock a numpy array's memory so uploads from it are asynchronous DMA copies; returns the array"""
    _check(lib().mc2_host_register(_p(arr), C.c_uint64(arr.nbytes)))
    return arr


def host_unregister(arr):
    _check(lib().mc2_host_unregister(_p(arr)))


def width_for_count(largest):
    return lib().mc2_width_for_count(C.c_uint64(largest))


class Seqs:
    def __init__(self, ctx, h):
        self.ctx, self.h = ctx, h

    def __len__(self):
        return lib().mc2_seqs_count(self.h)

    @property
    def total_bases(self):
        return lib().mc2_seqs_total_bases(self.h)

    def segments(self):
        """(segs int32[total,2], seg_off uint64[n+1], lengths uint64[n]) as held on the device"""
        n = len(self)
        tot = lib().mc2_seqs_total_segments(self.h)
        segs = np.zeros((tot, 2), dtype=np.int32)
        off = np.zeros(n + 1, dtype=np.uint64)
        ln = np.zeros(n, dtype=np.uint64)
        _check(lib().mc2_seqs_download_segments(self.ctx.h, self.h, _p(segs) if tot else None, _p(off), _p(ln) if n else None))
        return segs, off, ln

    def free(self):
        if self.h:
            lib().mc2_seqs_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class HistSet:
    def __init__(self, ctx, h):
        self.ctx, self.h = ctx, h

    def __len__(self):
        return lib().mc2_hset_count(self.h)

    @property
    def k(self):
        return lib().mc2_hset_k(self.h)

    @property
    def elem_bytes(self):
        return lib().mc2_hset_elem_bytes(self.h)

    def largest_count(self):
        """Runner::run's "Largest count" (1 + largest k-mer multiplicity); only for sets produced by count_kmers*"""
        out = C.c_uint64()
        _check(lib().mc2_hset_largest_count(self.h, C.byref(out)))
        return out.value

    def device_bins(self):
        return lib().mc2_hset_device_bins(self.h)

    def update_from_device(self, d_bins, d_len, d_mag=None):
        _check(lib().mc2_hset_update_from_device(self.ctx.h, self.h, C.c_void_p(d_bins), C.c_void_p(d_mag) if d_mag else None,
                                                 C.c_void_p(d_len)))

    def refresh(self, set_mag=False):
        """after external writes through the device pointers: recompute the true sums, drop the derived caches"""
        _check(lib().mc2_hset_refresh(self.ctx.h, self.h, int(set_mag)))

    def device_sideband(self, which):
        """0 mag, 1 len, 2 sum, 3 sumsq -> raw device pointer"""
        return lib().mc2_hset_device_sideband(self.h, which)

    def download(self, first=0, count=None):
        n = len(self)
        count = n - first if count is None else count
        N = 4 ** self.k
        out = dict(
            hist=np.zeros((count, N), dtype=DTYPES[self.elem_bytes]),
            mag=np.zeros(count, dtype=np.uint64), len=np.zeros(count, dtype=np.uint64),
            mers1=np.zeros((count, 4), dtype=np.uint64), stddev=np.zeros(count),
            n_overflow=np.zeros(count, dtype=np.int32), max_count=np.zeros(count, dtype=np.uint32))
        _check(lib().mc2_hset_download(self.ctx.h, self.h, C.c_uint64(first), C.c_uint64(count), _p(out["hist"]),
                                       _p(out["mag"]), _p(out["len"]), _p(out["mers1"]), _p(out["stddev"]),
                                       _p(out["n_overflow"]), _p(out["max_count"])))
        return out

    def copy_to_device(self, d_bins=None, d_mag=None, d_len=None, first=0, count=None):
        """D2D copy of rows into caller-owned device buffers given as raw pointers (torch_tensor.data_ptr())"""
        count = len(self) - first if count is None else count
        _check(lib().mc2_hset_copy_to_device(self.ctx.h, self.h, C.c_uint64(first), C.c_uint64(count),
                                             C.c_void_p(d_bins) if d_bins else None, C.c_void_p(d_mag) if d_mag else None,
                                             C.c_void_p(d_len) if d_len else None))

    def set_sideband(self, rows, mag=None, length=None):
        rows = _u64(rows)
        _check(lib().mc2_hset_set_sideband(self.ctx.h, self.h, C.c_uint64(len(rows)), _p(rows), _p(_u64(mag)),
                                           _p(_u64(length))))

    def set_row(self, dst_row, src, src_row):
        _check(lib().mc2_hset_set_row(self.ctx.h, self.h, C.c_uint64(dst_row), src.h, C.c_uint64(src_row)))

    def assign_rows(self, dst_rows, src, src_rows, mag=None, length=None):
        dst_rows, src_rows = _u64(dst_rows), _u64(src_rows)
        _check(lib().mc2_hset_assign_rows(self.ctx.h, self.h, C.c_uint64(len(dst_rows)), _p(dst_rows), src.h, _p(src_rows),
                                          _p(_u64(mag)), _p(_u64(length))))

    def reverse_complement(self):
        """a new set whose row i is the histogram of the other strand of the sequence row i counted"""
        h = C.c_void_p()
        _check(lib().mc2_hset_reverse_complement(self.ctx.h, self.h, C.byref(h)))
        return HistSet(self.ctx, h)

    def free(self):
        if self.h:
            lib().mc2_hset_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Model:
    def __init__(self, ctx, h, desc):
        self.ctx, self.h, self.desc = ctx, h, desc
        self.meta = {}

    def free(self):
        if self.h:
            lib().mc2_model_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def encode_dna(text):
    """raw DNA text (bytes) -> (codes int8[len], segs int32[nseg,2], effective_size); host-only (input contract a1)."""
    n = len(text)
    codes = np.zeros(max(n, 1), dtype=np.int8)
    max_segs = n // 2 + 2
    segs = np.zeros((max_segs, 2), dtype=np.int32)
    nseg, eff = C.c_uint64(), C.c_uint64()
    _check(lib().mc2_encode_dna(text, C.c_uint64(n), _p(codes), _p(segs), C.c_uint64(max_segs), C.byref(nseg),
                                C.byref(eff)))
    return codes[:n], segs[:nseg.value].copy(), eff.value


def encode_batch(texts, threads=0):
    """list of raw DNA bytes -> dict(codes, seq_off, segs, seg_off, eff) ready for Context.upload_seqs."""
    n = len(texts)
    off = np.zeros(n + 1, dtype=np.uint64)
    if n:
        off[1:] = np.cumsum([len(t) for t in texts])
    blob = b"".join(texts)
    total = int(off[n])
    codes = np.zeros(max(total, 1), dtype=np.int8)
    max_segs = total // 20 + 2 * n + 16
    segs = np.zeros((max_segs, 2), dtype=np.int32)
    seg_off = np.zeros(n + 1, dtype=np.uint64)
    eff = np.zeros(max(n, 1), dtype=np.uint64)
    if threads <= 0:
        threads = os.cpu_count() or 1
    _check(lib().mc2_encode_dna_batch(blob, _p(off), C.c_uint64(n), _p(codes), _p(segs), C.c_uint64(max_segs),
                                      _p(seg_off), _p(eff), threads))
    return dict(codes=codes[:total], seq_off=off, segs=segs[:int(seg_off[n])].copy(), seg_off=seg_off, eff=eff[:n])


def model_desc_from_file(path, which=0):
    """Parse a reference weights.txt (Predictor::save format). Pure host parsing inside the C library; needs no GPU."""
    d = ModelDesc()
    k, ident, eb, mode = C.c_int(), C.c_double(), C.c_int(), C.c_int()
    _check(lib().mc2_model_desc_from_file(os.fsencode(path), which, C.byref(d), C.byref(k), C.byref(ident), C.byref(eb),
                                          C.byref(mode)))
    return d, dict(k=k.value, id=ident.value, elem_bytes=eb.value, mode=mode.value)


def make_desc(singles, combos, weights, bias=0.0, regression=0):
    """singles: [(flag, min, max)], combos: [(kind_code, [single indices])], weights: C+1 doubles."""
    d = ModelDesc()
    d.n_singles = len(singles)
    for i, (f, lo, hi) in enumerate(singles):
        d.single_flag[i], d.single_min[i], d.single_max[i] = f, lo, hi
    d.n_combos = len(combos)
    for c, (kind, idx) in enumerate(combos):
        d.combo_kind[c] = kind
        d.combo_nidx[c] = len(idx)
        for j, ix in enumerate(idx):
            d.combo_idx[c][j] = ix
    for i, w in enumerate(weights):
        d.weight[i] = w
    d.bias = bias
    d.regression = regression
    return d
