/* meshclust2_b200.h — C ABI of the B200-native MeShClust2 hot path.
 *
 * The reference (BioinformaticsToolsmith/MeShClust2 2.3.0) has no FFI layer: its boundary for this
 * path is a C++ template API linked statically (SURVEY.md §8b).  This header is what a cgo/JNI/ctypes
 * style binding — or the C++ shim classes in meshclust2_b200/host/ that keep the reference's own class
 * names — binds instead.  Each entry point cites the reference interface it replaces (paths relative to
 * the reference root).
 *
 * Conventions: plain C types only; every function returns MC2_OK (0) or a negative mc2_status;
 * mc2_last_error() gives a thread-local message; no C++ exception ever crosses this boundary;
 * outputs are caller-allocated.  One mc2_ctx per GPU; a ctx and the objects made from it may be used
 * from one host thread at a time (create one ctx per thread for concurrent use).
 * There is NO CPU fallback: every compute entry point fails with MC2_ERR_CUDA when no sm_100 device
 * is usable.
 */
#ifndef MESHCLUST2_B200_H
#define MESHCLUST2_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MC2_ABI_VERSION 1

typedef enum {
	MC2_OK = 0,
	MC2_ERR_ARG = -1,        /* bad argument (k, elem_bytes, NULL, index out of range ...) */
	MC2_ERR_CUDA = -2,       /* CUDA runtime / no device / wrong architecture */
	MC2_ERR_INPUT = -3,      /* the reference would throw InvalidInputException (code outside 0..3 in a segment) */
	MC2_ERR_FEATURE = -4,    /* the reference would throw while scoring (length 0 for length_difference, NaN after normalise) */
	MC2_ERR_UNSUPPORTED = -5,/* feature flag / combination outside the hot-path scope (SURVEY.md §8 a9) */
	MC2_ERR_IO = -6          /* weights file unreadable / malformed */
} mc2_status;

/* single-feature flags: src/predict/Feature.h:31-64 (same bit values) */
#define MC2_FEAT_MANHATTAN           (1ULL << 2)
#define MC2_FEAT_EUCLIDEAN           (1ULL << 3)
#define MC2_FEAT_NORMALIZED_VECTORS  (1ULL << 5)
#define MC2_FEAT_JEFFEREY_DIV        (1ULL << 7)
#define MC2_FEAT_PEARSON_COEFF       (1ULL << 9)
#define MC2_FEAT_INTERSECTION        (1ULL << 13)
#define MC2_FEAT_EMD                 (1ULL << 18)
#define MC2_FEAT_LENGTHD             (1ULL << 21)
#define MC2_FEAT_KULCZYNSKI2         (1ULL << 27)
#define MC2_FEAT_SIMRATIO            (1ULL << 28)
#define MC2_FEAT_JENSEN_SHANNON      (1ULL << 29)
/* src/predict/Predictor.h:23-24 */
#define MC2_PRED_FEAT_FAST (MC2_FEAT_EUCLIDEAN | MC2_FEAT_MANHATTAN | MC2_FEAT_INTERSECTION | MC2_FEAT_KULCZYNSKI2 | \
			    MC2_FEAT_SIMRATIO | MC2_FEAT_NORMALIZED_VECTORS | MC2_FEAT_PEARSON_COEFF | MC2_FEAT_EMD | MC2_FEAT_LENGTHD)
#define MC2_PRED_FEAT_DIV (MC2_FEAT_JEFFEREY_DIV | MC2_FEAT_JENSEN_SHANNON)

/* combo codes as stored in weights.txt: src/predict/Predictor.cpp:96-110 (enum class Combo, Feature.h:66-71) */
#define MC2_COMBO_XY   0
#define MC2_COMBO_XY2  1
#define MC2_COMBO_X2Y  2
#define MC2_COMBO_X2Y2 3

#define MC2_MAX_SINGLES 16
#define MC2_MAX_COMBOS 16
#define MC2_MAX_COMBO_IDX 4

/* A trained Feature<T> + GLM weight column, i.e. what Predictor::get_class() hands to Trainer
 * (src/predict/Predictor.h:57, src/cluster/Trainer.cpp:160-182) and what weights.txt stores. */
typedef struct {
	int32_t n_singles;                                   /* Feature::lookup.size() */
	uint64_t single_flag[MC2_MAX_SINGLES];               /* Feature::lookup, in add_feature order */
	double single_min[MC2_MAX_SINGLES];                  /* Feature::mins */
	double single_max[MC2_MAX_SINGLES];                  /* Feature::maxs */
	int32_t n_combos;                                    /* Feature::size() */
	int32_t combo_kind[MC2_MAX_COMBOS];                  /* MC2_COMBO_* */
	int32_t combo_nidx[MC2_MAX_COMBOS];
	int32_t combo_idx[MC2_MAX_COMBOS][MC2_MAX_COMBO_IDX];/* indices into singles, ascending flag bit */
	double weight[MC2_MAX_COMBOS + 1];                   /* GLM weights, [0] = intercept */
	double bias;                                         /* Predictor::set_bias (src/predict/Predictor.cpp:307-313) */
	int32_t regression;                                  /* 0: classifier (logistic + cutoff); 1: Predictor::p_predict clamp */
} mc2_model_desc;

typedef struct mc2_ctx mc2_ctx;     /* one GPU: device id, stream, scratch, pinned result slots */
typedef struct mc2_seqs mc2_seqs;   /* device-resident 2-bit packed sequences + segment lists */
typedef struct mc2_hset mc2_hset;   /* device-resident histogram matrix n x 4^k (elem_bytes wide) + side-band SoA */
typedef struct mc2_model mc2_model; /* device-side copy of a mc2_model_desc */

/* ---- context ---------------------------------------------------------------------------------- */
int mc2_abi_version(void);
const char *mc2_last_error(void);
int mc2_device_count(void);
int mc2_ctx_create(int device, mc2_ctx **out);
void mc2_ctx_destroy(mc2_ctx *ctx);
int mc2_ctx_sync(mc2_ctx *ctx);
int mc2_ctx_device(const mc2_ctx *ctx);
int mc2_ctx_sm_count(const mc2_ctx *ctx);
void *mc2_ctx_stream(mc2_ctx *ctx);                 /* the cudaStream_t every launch of this ctx goes to */
/* CUDA-event stopwatch on the ctx stream (bench.py times kernels with it, not wall clock) */
int mc2_timer_start(mc2_ctx *ctx);
int mc2_timer_stop(mc2_ctx *ctx, float *ms);
/* count of this library's kernel launches on this ctx since creation (bench.py's gpu_launches) */
uint64_t mc2_ctx_launch_count(const mc2_ctx *ctx);
/* Per-kernel device timing (CUDA events around each launch on the ctx stream), for bench.py's roofline object.
 * kinds: 0 pack, 1 k-mer count, 2 pair score (gather / one-vs-many), 3 sweep (query-vs-database), 4 argmax, 5 side-band,
 * 6 batched update / merge stage.
 * mc2_ctx_profile(ctx, 1) starts collecting (and clears the totals), (ctx, 0) stops;
 * mc2_ctx_kernel_time synchronises the stream and returns the summed milliseconds and launch count of one kind. */
#define MC2_KERNEL_KINDS 7
int mc2_ctx_profile(mc2_ctx *ctx, int enable);
int mc2_ctx_kernel_time(mc2_ctx *ctx, int kind, double *total_ms, uint64_t *launches);
/* write `bytes` of zeros to a scratch buffer (L2 flush between timed iterations) */
int mc2_ctx_flush_l2(mc2_ctx *ctx, size_t bytes);

/* ---- host-side input contract (no GPU involved) ------------------------------------------------ */
/* For callers that do not already hold a reference ChromosomeOneDigit: raw DNA text -> one-digit codes + inclusive
 * segments + effective size, exactly as Chromosome::help + ChromosomeOneDigit::encode produce them
 * (src/nonltr/Chromosome.cpp:130-154, 263-385; src/nonltr/ChromosomeOneDigit.cpp:79-133;
 * src/nonltr/ChromosomeOneDigitDna.cpp:48-68).  Stays on the host, as in the reference (SURVEY.md section 8 a1).
 * MC2_ERR_INPUT where the reference throws InvalidInputException. */
int mc2_encode_dna(const char *text, uint64_t len, char *codes_out, int32_t *segs_out, uint64_t max_segs,
		   uint64_t *n_segs, uint64_t *effective_size);
/* n sequences at text[off[i]..off[i+1]); codes_out has off[n]-off[0] bytes; segs_out 2*max_segs ints (sequence-relative);
 * seg_off_out n+1; effective_sizes n (may be NULL). OpenMP over sequences with `threads` threads. */
int mc2_encode_dna_batch(const char *text, const uint64_t *off, uint64_t n, char *codes_out, int32_t *segs_out,
			 uint64_t max_segs, uint64_t *seg_off_out, uint64_t *effective_sizes, int threads);

/* ---- K1: k-mer histograms ---------------------------------------------------------------------- */
/* Input contract = ChromosomeOneDigit after finalize() (src/nonltr/ChromosomeOneDigit.cpp:79-133):
 * codes[seq_off[i] .. seq_off[i+1]) is sequence i, one byte per base, values 0..3 inside segments
 * (anything outside); segs holds inclusive [start,end] pairs relative to the sequence start, sequence i
 * owning segs[2*seg_off[i] .. 2*seg_off[i+1]).  Replaces the std::string base + vector<vector<int>*>* segment
 * that Loader<T>::fill_table reads (src/clutil/Loader.cpp:42-49). Copies host->device and packs to 2 bits/base. */
int mc2_seqs_upload(mc2_ctx *ctx, const char *codes, const uint64_t *seq_off, uint64_t n, const int32_t *segs,
		    const uint64_t *seg_off, mc2_seqs **out);
/* Refill an existing set with another batch: device arrays are reused (grow-only), so a steady stream of batches of similar
 * size never calls cudaMalloc / cudaFree.  On error the set is left empty (still to be freed by the caller). */
int mc2_seqs_upload_into(mc2_ctx *ctx, mc2_seqs *dst, const char *codes, const uint64_t *seq_off, uint64_t n,
			 const int32_t *segs, const uint64_t *seg_off);
/* The input contract itself on the device (SURVEY 8f-3): raw nucleotide text of n sequences (concatenated, no headers, no
 * line breaks; seq_off[n+1] byte offsets) -> segments + 2-bit packed bases, following Chromosome::help
 * (src/nonltr/Chromosome.cpp:130-154: upper-case; removeAmbiguous :263-291; mergeSegments :298-353; makeSegmentList
 * :355-385) and ChromosomeOneDigit::encode with the DNA code map (src/nonltr/ChromosomeOneDigit.cpp:79-133,
 * src/nonltr/ChromosomeOneDigitDna.cpp:48-68).  Same result as mc2_encode_dna_batch + mc2_seqs_upload, without the host
 * pass.  MC2_ERR_INPUT for a byte that is not a nucleotide letter in a sequence that has at least one segment
 * (InvalidInputException, ChromosomeOneDigit.cpp:86-95). */
int mc2_seqs_from_text(mc2_ctx *ctx, const char *text, const uint64_t *seq_off, uint64_t n, mc2_seqs **out);
/* same, refilling an existing set (device arrays reused, as mc2_seqs_upload_into) */
int mc2_seqs_from_text_into(mc2_ctx *ctx, mc2_seqs *dst, const char *text, const uint64_t *seq_off, uint64_t n);
/* segments of a sequence set back on the host (inclusive, sequence-relative pairs; seg_off[n+1]; lengths[n] = bases per
 * sequence); any pointer may be NULL.  mc2_seqs_total_segments sizes segs_out. */
int mc2_seqs_download_segments(mc2_ctx *ctx, const mc2_seqs *s, int32_t *segs_out, uint64_t *seg_off_out,
			       uint64_t *lengths_out);
uint64_t mc2_seqs_total_segments(const mc2_seqs *s);
/* Page-lock / unlock a caller-owned host range (cudaHostRegister) so that uploads from it are asynchronous DMA copies.
 * Optional: every entry point also accepts pageable memory. */
int mc2_host_register(void *ptr, uint64_t bytes);
int mc2_host_unregister(void *ptr);
void mc2_seqs_free(mc2_seqs *s);
uint64_t mc2_seqs_count(const mc2_seqs *s);
uint64_t mc2_seqs_total_bases(const mc2_seqs *s);

/* Loader<T>::get_point for a whole batch (src/clutil/Loader.cpp:138-179): per sequence a 4^k histogram of
 * elem_bytes-wide counts initialised to 1 and saturating at max(T) (KmerHashTable::wholesaleIncrementNoOverflow,
 * src/nonltr/KmerHashTable.cpp:236-256), the k=1 table (u64, init 1), mag = sum of bins
 * (DivergencePoint ctor, src/clutil/DivergencePoint.cpp:99-110), length = sum of segment lengths
 * (Chromosome::getEffectiveSize), stddev (Loader.cpp:162-171) and the number of overflowing segments
 * (Loader.cpp:55-56).  elem_bytes in {1,2,4,8} = --datatype 8/16/32/64 (src/cluster/CRunner.cpp:278-291). */
int mc2_count_kmers(mc2_ctx *ctx, const mc2_seqs *seqs, int k, int elem_bytes, mc2_hset **out);

/* Histogram-width detection fused with counting (Runner::run, src/cluster/CRunner.cpp:57-127; the free fill_table<V>,
 * src/cluster/ClusterFactory.h:40-54).  The reference first counts every sequence into a u64 table just to find
 * "Largest count" = 1 + the largest k-mer multiplicity, picks the narrowest of 8/16/32/64 bits that holds it
 * (CRunner.cpp:108-126) and then counts everything again at that width.  K1 counts in 32-bit shared-memory bins
 * whatever the output width, so the multiplicities come for free: mc2_count_kmers_auto counts once at 8 bits, and only
 * when the largest count exceeds 255 counts again at the detected width.  *largest_count / *elem_bytes (may be NULL)
 * receive what the reference prints as "Largest count" and the chosen width in bytes.
 * MC2_ERR_INPUT if a segment is shorter than k: the reference's detection pass (unlike Loader::fill_table) has no length
 * guard and hashes k characters from the segment start, reading past it (quirk Q6) - there is no result to reproduce. */
int mc2_count_kmers_auto(mc2_ctx *ctx, const mc2_seqs *seqs, int k, uint64_t *largest_count, int *elem_bytes,
			 mc2_hset **out);
/* Multi-GPU exchange without staging copies (SURVEY.md section 8e: per-rank K1 shards all-gathered into the full set):
 * mc2_hset_alloc makes an n-row set with zeroed rows; mc2_count_kmers_into_rows runs K1 (Loader<T>::get_point,
 * src/clutil/Loader.cpp:138-179) for `seqs` straight into rows [first_row, first_row + n_seqs) of it; the caller then
 * lets the collective (e.g. an in-place NCCL all-gather) write the other ranks' bins / mag / len through the device
 * pointers (mc2_hset_device_bins, mc2_hset_device_sideband) and calls mc2_hset_refresh, which recomputes the true bin
 * sums (and the magnitudes when set_mag != 0) and drops every derived cache. */
int mc2_hset_alloc(mc2_ctx *ctx, uint64_t n, int k, int elem_bytes, mc2_hset **out);
int mc2_count_kmers_into_rows(mc2_ctx *ctx, const mc2_seqs *seqs, mc2_hset *dst, uint64_t first_row);
int mc2_hset_refresh(mc2_ctx *ctx, mc2_hset *h, int32_t set_mag);

/* "Largest count" of a set produced by mc2_count_kmers(_into/_auto); MC2_ERR_UNSUPPORTED for sets built from
 * histograms (their multiplicities before saturation are unknown). */
int mc2_hset_largest_count(const mc2_hset *h, uint64_t *largest_count);
/* CRunner.cpp:108-126: bytes per bin for a largest count: 1, 2, 4 or 8 */
int mc2_width_for_count(uint64_t largest_count);

/* Same, into an existing set of the same shape (n, k, elem_bytes): no allocation in steady state (repeated batches). */
int mc2_count_kmers_into(mc2_ctx *ctx, const mc2_seqs *seqs, mc2_hset *dst);

/* KmerHashTable<unsigned long,V>(k, init).wholesaleIncrementNoOverflow(codes, first, last) on ONE sequence
 * (src/nonltr/KmerHashTable.h:20-79): values_out receives the 4^k table; *ret = 0 or -1 (saturation).
 * MC2_ERR_INPUT where the reference throws InvalidInputException. */
int mc2_kmer_table_increment(mc2_ctx *ctx, const char *codes, int32_t first_kmer_start, int32_t last_kmer_start, int k,
			     int elem_bytes, uint64_t init_value, void *values_out, int32_t *ret);

/* ---- histogram sets ----------------------------------------------------------------------------- */
/* Build a set from host DivergencePoint<T> state: bins (n x 4^k, row-major), pseudo-magnitude and length per
 * point (src/clutil/DivergencePoint.h:80-88).  mag may be NULL (= sum of bins, as the ctor computes) or carry
 * the host object's possibly stale value (DivergencePoint::set does not refresh it, DivergencePoint.cpp:182-190). */
int mc2_hset_from_host(mc2_ctx *ctx, const void *bins, uint64_t n, int k, int elem_bytes, const uint64_t *mag,
		       const uint64_t *len, mc2_hset **out);
/* Same from DEVICE memory on ctx's GPU (e.g. a torch tensor that an NCCL all-gather of per-rank shards just filled):
 * bins n x 4^k row-major, d_len n u64, d_mag n u64 or NULL (= sum of bins). The data is copied; the caller keeps
 * ownership of its buffers. */
int mc2_hset_from_device(mc2_ctx *ctx, const void *d_bins, uint64_t n, int k, int elem_bytes, const uint64_t *d_mag,
			 const uint64_t *d_len, mc2_hset **out);
/* Refill an existing set of the same shape from device memory (no allocation). */
int mc2_hset_update_from_device(mc2_ctx *ctx, mc2_hset *h, const void *d_bins, const uint64_t *d_mag, const uint64_t *d_len);
/* device pointer of a side-band column: which = 0 mag, 1 len, 2 sum of bins, 3 sum of squared bins (n u64 each) */
void *mc2_hset_device_sideband(const mc2_hset *h, int which);
void mc2_hset_free(mc2_hset *h);
uint64_t mc2_hset_count(const mc2_hset *h);
int mc2_hset_k(const mc2_hset *h);
int mc2_hset_elem_bytes(const mc2_hset *h);
/* device pointers (for NCCL all-gather of shards through torch tensors; rows are contiguous, stride 4^k elements) */
void *mc2_hset_device_bins(const mc2_hset *h);
/* copy rows [first, first+count) back: any output pointer may be NULL. mers1: count x 4; n_overflow: count */
int mc2_hset_download(mc2_ctx *ctx, const mc2_hset *h, uint64_t first, uint64_t count, void *bins, uint64_t *mag,
		      uint64_t *len, uint64_t *mers1, double *stddev, int32_t *n_overflow, uint32_t *max_count);
/* same as mc2_hset_download but into DEVICE buffers on ctx's GPU (bins / mag / len; any may be NULL); the copy has
 * completed when the call returns, so another stream (e.g. NCCL's) may read the buffers */
int mc2_hset_copy_to_device(mc2_ctx *ctx, const mc2_hset *h, uint64_t first, uint64_t count, void *d_bins,
			    uint64_t *d_mag, uint64_t *d_len);
/* overwrite pseudo-magnitudes / lengths of selected rows (mirror of host objects mutated by set()/set_length()) */
int mc2_hset_set_sideband(mc2_ctx *ctx, mc2_hset *h, uint64_t count, const uint64_t *rows, const uint64_t *mag,
			  const uint64_t *len);
/* copy row `src_row` of `src` over row `dst_row` of `dst` the way DivergencePoint::set does: bins + length, NOT mag */
int mc2_hset_set_row(mc2_ctx *ctx, mc2_hset *dst, uint64_t dst_row, const mc2_hset *src, uint64_t src_row);

/* Batched form of the two calls above, one launch: dst row dst_rows[i] receives the bins (and true sums) of src row
 * src_rows[i]; its length becomes len[i] (NULL: the src row's length) and its pseudo-magnitude mag[i] (NULL: the dst row
 * keeps the magnitude it had, i.e. DivergencePoint::set semantics).  Used to assemble the (possibly stale-magnitude)
 * center rows that Trainer::filter / merge compare (src/cluster/ClusterFactory.cpp:288-335, 383-401). */
int mc2_hset_assign_rows(mc2_ctx *ctx, mc2_hset *dst, uint64_t n, const uint64_t *dst_rows, const mc2_hset *src,
			 const uint64_t *src_rows, const uint64_t *mag, const uint64_t *len);

/* The other strand: row i of *out is the histogram of the reverse complement of the sequence row i of src counted.  The
 * bin index is the big-endian base-4 k-mer (A=0, C=1, G=2, T=3), so out[i][rc(j)] = src[i][j] with
 * rc(j) = reverse_base4_digits(j) XOR (4^k - 1); this is exact, saturated bins included (rc is a bijection on k-mers, a bin
 * is min(max(T), 1 + count) whatever the order of the bases, and mirroring a segment maps its k-mers to their reverse
 * complements).  Every k (1..12) and width.  Side-band: mag (stale or not), len, the true sums, stddev and the per-row
 * largest count are copied; the k = 1 table swaps A<->T and C<->G; mc2_hset_largest_count answers as for src.  The
 * per-row count of overflowing segments depends on segment order, which reversal changes: *out reports 0, as a set made by
 * mc2_hset_from_host does.  Derived operands that depend on bin order are built for *out when first needed. */
int mc2_hset_reverse_complement(mc2_ctx *ctx, const mc2_hset *src, mc2_hset **out);

/* ---- model -------------------------------------------------------------------------------------- */
int mc2_model_create(mc2_ctx *ctx, const mc2_model_desc *desc, mc2_model **out);
void mc2_model_free(mc2_model *m);
/* Parse a weights file written by Predictor::save (src/predict/Predictor.cpp:28-44, 82-121) the way the file ctor
 * does (Predictor.cpp:47-79, 125-185). which = 0: classifier block, 1: regression block.
 * k/id/elem_bytes/mode outputs may be NULL. */
int mc2_model_desc_from_file(const char *path, int which, mc2_model_desc *desc, int *k, double *id, int *elem_bytes,
			     int *mode);

/* ---- K2: pair features + GLM -------------------------------------------------------------------- */
/* What to score.  first/second follow the reference's argument order of Feature::compute(first, second). */
typedef struct {
	const mc2_hset *set_a;     /* rows ia[] index into set_a */
	const mc2_hset *set_b;     /* rows ib[] index into set_b (may equal set_a) */
	uint64_t n_pairs;
	const uint64_t *ia;        /* host array, or NULL: ia[j] = a_begin + (a_broadcast ? 0 : j) */
	const uint64_t *ib;        /* host array, or NULL: ib[j] = b_begin + (b_broadcast ? 0 : j) */
	uint64_t a_begin, b_begin;
	int32_t a_broadcast, b_broadcast;
	/* length prefilter of Trainer::get_close/merge/filter (src/cluster/Trainer.cpp:39-48, 82-91, 126-130):
	 * when len_filter != 0 a pair is skipped (close=0, score=dist=NaN, skipped=1) unless the NON-anchor length lies in
	 * [(u64)(len_anchor*cutoff), (u64)(len_anchor/cutoff)]; anchor = side b if anchor_is_b else side a. */
	int32_t len_filter;
	int32_t anchor_is_b;
	double cutoff;
	/* optional (bc_override != 0): the broadcast row reports this pseudo-magnitude and length instead of its set's own.
	 * A cluster center carries the bins of the point it was last set() to but keeps its own magnitude (quirk Q4,
	 * ClusterFactory.cpp:328); this scores it straight from the point set without staging a copy of the row. */
	int32_t bc_override;
	int32_t reserved_;
	uint64_t bc_mag, bc_len;
} mc2_pairs;

/* Feature<T>::compute + operator() + Trainer<T>::classify / Predictor<T>::p_close / p_predict
 * (src/predict/Feature.h:197-239, src/cluster/Trainer.cpp:112-120, src/predict/Predictor.cpp:284-333).
 * Outputs (host, each may be NULL): score[n_pairs] = logistic(sum)+bias (or the clamped sum for a regression model),
 * dist[n_pairs] = first combo value, close[n_pairs] = round(score) > 0, cache[n_pairs x n_singles] = normalised singles,
 * raw[n_pairs x n_singles] = raw singles (what Feature::normalize / BestFirstSelector::calculate_table consume),
 * skipped[n_pairs] = 1 where the length prefilter dropped the pair. */
int mc2_score_pairs(mc2_ctx *ctx, const mc2_model *model, const mc2_pairs *pairs, double *score, double *dist,
		    uint8_t *close, double *cache, double *raw, uint8_t *skipped);

/* Trainer<T>::get_close (src/cluster/Trainer.cpp:23-71): query row `q` of set_q against candidate rows cand[0..n_cand)
 * of set_c (cand NULL = rows cand_begin .. cand_begin+n_cand).  Feature order compute(candidate, query).
 * *best = position in the candidate list of the max first-combo value over all in-window candidates (first such position on
 * ties, -1 if none in window), *best_dist its value (-1 if none), *is_min = no candidate classified close,
 * marks[n_cand] = 1 for candidates classified close (the reference sets (*i).second = true). */
int mc2_get_close(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q, const mc2_hset *set_c,
		  const uint64_t *cand, uint64_t cand_begin, uint64_t n_cand, double cutoff, int64_t *best,
		  double *best_dist, int32_t *is_min, uint8_t *marks);

/* Trainer<T>::filter (src/cluster/Trainer.cpp:123-141): keep[j] = 1 iff member j survives (in window and
 * round(classify(center, member)) != 0). Feature order compute(center, member). */
/* mc2_get_close / mc2_filter for a query (center) that is row `q` of set_q as far as bins and true sums go, but reports
 * q_mag / q_len as its pseudo-magnitude and length (mc2_pairs.bc_override): one call, no staging of the row. */
int mc2_get_close_as(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q, uint64_t q_mag, uint64_t q_len,
		     const mc2_hset *set_c, const uint64_t *cand, uint64_t cand_begin, uint64_t n_cand, double cutoff,
		     int64_t *best, double *best_dist, int32_t *is_min, uint8_t *marks);
int mc2_filter_as(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_c, uint64_t center, uint64_t c_mag, uint64_t c_len,
		  const mc2_hset *set_m, const uint64_t *members, uint64_t n_members, double id, uint8_t *keep);
int mc2_filter(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_c, uint64_t center, const mc2_hset *set_m,
	       const uint64_t *members, uint64_t n_members, double id, uint8_t *keep);

/* Trainer<T>::merge (src/cluster/Trainer.cpp:74-109): center row rows[cur] vs rows[begin..last] of `centers`;
 * *out = chosen index in [begin,last] or 0 when none is close. 
 * MC2_ERR_UNSUPPORTED for a regression model or a bias outside [-0.5, 0.5): the reference merges on round(score) == 1
 * (Trainer.cpp:100-103), the device flags round(score) > 0; callers then apply the rule to mc2_score_pairs outputs. */
int mc2_merge(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *centers, const uint64_t *rows, int64_t cur,
	      int64_t begin, int64_t last, double id, int64_t *out);

/* Batched update stage (SURVEY section 8e: "batching independent queries (update stage: all centers are independent)").
 * `centers` holds one staged row per center (mc2_hset_assign_rows: bins of the point whose id the center carries + the host
 * object's own pseudo-magnitude and length); the members of center c are rows members[member_off[c] .. member_off[c+1]) of
 * set_m.
 *
 * mc2_update_centers = mean_shift_update (src/cluster/ClusterFactory.cpp:288-335) for every center of one pass of the loops at
 * :639-642 / :650-653: Trainer::filter (src/cluster/Trainer.cpp:123-141: length window, then round(classify(center, member))
 * != 0), the per-bin mean of the survivors, Trainer::closest (:144-157: first minimum of distance_d).  next[c] = position
 * inside center c's member list of the chosen member, -1 when no member survives; n_good[c] = number of survivors (may be
 * NULL).  One pair-scoring launch + one launch of a CTA per center, whatever the number of centers.
 *
 * mc2_merge_centers = Trainer::merge (src/cluster/Trainer.cpp:74-109) for every center of one pass of merge()
 * (src/cluster/ClusterFactory.cpp:382-401): center c against centers c+1 .. min(n_centers-1, c+delta); out[c] = the chosen
 * center index, or 0 when none is close (the reference's return value; callers test `ret > c`).  trn.merge never looks at
 * the lazily removed flag, so the passes of one merge() call are independent of each other. */
int mc2_update_centers(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *centers, uint64_t n_centers, const mc2_hset *set_m,
		       const uint64_t *member_off, const uint64_t *members, double id, int64_t *next, uint64_t *n_good);
int mc2_merge_centers(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *centers, uint64_t n_centers, int64_t delta, double id,
		      int64_t *out);

/* All-pairs / query-vs-database sweep with the length prefilter, as fastcar's work() does
 * (src/fastcar/FC_Runner.cpp:427-470): for every query row r in [q_begin,q_end) of set_q and database row c in
 * [d_begin,d_end) of set_d with len_c in [(size_t)(len_r*cutoff), (size_t)(len_r/cutoff)] evaluate close(c, r);
 * upper_only != 0 restricts to c > r (set_q == set_d, unordered pairs).  Survivors (close pairs) are appended to
 * out_q/out_d/out_score (capacity max_out); *n_out returns the TOTAL number of survivors (may exceed max_out),
 * *n_scored the number of pairs that passed the prefilter and were scored. Order of survivors is unspecified. */
int mc2_all_pairs(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q_begin, uint64_t q_end,
		  const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end, int32_t upper_only, double cutoff,
		  uint64_t max_out, uint64_t *out_q, uint64_t *out_d, double *out_score, uint64_t *n_out,
		  uint64_t *n_scored);

/* Identity search: every (query, database) pair of the two row ranges inside the length window, as mc2_all_pairs
 * (FC_Runner.cpp:435-444; upper_only: c > r; feature order compute(database c, query r)), scored with a REGRESSION model
 * (Predictor<T>::similarity = p_predict, Predictor.cpp:284-300: identity = GLM sum clamped to [0, 1]).
 * Survivors are the pairs with identity >= min_identity (the >= of the reference's --id labels, FeatureSelector.cpp:27):
 * min_identity <= 0 keeps every in-window pair, a value above 1 keeps none, and fastcar's `sim > 0` is min_identity = the
 * smallest positive double (4.9406564584124654e-324).  out_identity[i] is the same bits as the score mc2_score_pairs gives
 * the pair (set_a = set_d row out_d[i], set_b = set_q row out_q[i]), and the decision is made on that value.
 * Ranges, capacity (*n_out is the total, which may exceed max_out), *n_scored (equal to mc2_all_pairs' for the same
 * ranges and cutoff) and the unspecified survivor order are those of mc2_all_pairs; every shape it serves is served.
 * MC2_ERR_ARG for a classifier model or a NaN min_identity, besides mc2_all_pairs' argument checks; MC2_ERR_FEATURE when
 * an in-window pair hits the reference's throw (length 0 with length_difference, NaN after normalising). */
int mc2_identity_pairs(mc2_ctx *ctx, const mc2_model *model, double min_identity, const mc2_hset *set_q, uint64_t q_begin,
		       uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end, int32_t upper_only, double cutoff,
		       uint64_t max_out, uint64_t *out_q, uint64_t *out_d, double *out_identity, uint64_t *n_out,
		       uint64_t *n_scored);

/* Both-strand identity search: mc2_identity_pairs over each in-window (query, database) pair on both strands of the query.
 * id+ = similarity(database d, query q) as mc2_identity_pairs scores it; id- = similarity(database d, reverse complement of q)
 * (mc2_hset_reverse_complement: only the query is flipped, the database stays forward).  A pair survives iff
 * max(id+, id-) >= min_identity; out_identity[i] is that max and out_strand[i] the strand it came from, 0 forward or 1
 * reverse, a tie (equal values) going to forward.  out_identity[i] is the same bits as the score mc2_score_pairs gives the pair
 * on the reported strand (set_a = set_d row out_d[i], set_b = set_q or its reverse-complement set, row out_q[i]).
 * The reverse complement has the query's length, so both strands have the same length window and *n_scored is the number
 * mc2_identity_pairs reports.  Ranges, window, upper_only (c > r on row indices, which the reverse-complement rows keep),
 * capacity (*n_out is the total, which may exceed max_out; out_strand may be NULL), the unspecified survivor order and the
 * error codes are those of mc2_identity_pairs.
 * How: the forward sweep gives A = {id+ >= t}, at most max_out of it kept; the reverse sweep over the reverse-complement
 * rows gives B = {id- >= t}, query-row block by block into a fixed scratch of max(d_end - d_begin, 2^20) pairs (a block
 * whose survivors overflow it is split and swept again); id+ is recomputed for B's pairs and those with id+ < t join A;
 * id- is scored for the returned members of A.  Extra device memory does not grow with the number of survivors.  For
 * min_identity <= 0 every in-window pair is in A and only the returned entries' id- is scored.  The reverse-complement set
 * of set_q is built on first use and kept with set_q until its bins, magnitudes or lengths change.
 * mc2_debug_last_sweep afterwards: n_exact summed over every sweep of both strands, coarse = 1 iff every sweep took the
 * coarse form. */
int mc2_identity_pairs_both_strands(mc2_ctx *ctx, const mc2_model *model, double min_identity, const mc2_hset *set_q,
				    uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end,
				    int32_t upper_only, double cutoff, uint64_t max_out, uint64_t *out_q, uint64_t *out_d,
				    double *out_identity, int8_t *out_strand, uint64_t *n_out, uint64_t *n_scored);

/* Top-K identity search: for each query row r in [q_begin, q_end), its k_best best database hits.
 * Hits: exactly the pairs (r, c) that mc2_identity_pairs keeps for the same arguments (same length window, upper_only rule
 * c > r, feature order compute(database c, query r), same decision on the same bits).  exclude_self != 0 also drops c == r
 * (an all-vs-all neighbour table without the self hit); it needs set_q == set_d.
 * Order: identity descending, then database row ascending; the comparison is numeric (-0.0 equals +0.0).  Row r - q_begin of
 * the output holds the first min(k_best, hits) entries of that order: out_d and out_identity are (q_end - q_begin) x k_best,
 * row-major; out_identity[i] is the same bits as the score mc2_score_pairs gives the pair (set_a = set_d row out_d[i],
 * set_b = set_q row r); unused slots hold d = UINT64_MAX and identity -1.0.  out_count[r - q_begin] = the filled slots,
 * out_n_hits[r - q_begin] (may be NULL) = the query's total hit count, which may exceed k_best.  The order is total, so the
 * result does not depend on survivor order, block sizes or how the query rows are split over calls or GPUs.
 * *n_scored (may be NULL) equals mc2_identity_pairs'.  min_identity <= 0: every in-window pair is a hit; min_identity > 1:
 * no query has one; empty ranges give zero counts.
 * MC2_ERR_ARG: a classifier model, a NaN min_identity, k_best == 0 or > 1024, a (q_end - q_begin) x k_best table whose
 * size in bytes overflows, a database range of 2^32 rows or more, exclude_self with two different sets, and every argument
 * check of mc2_identity_pairs.  MC2_ERR_FEATURE as mc2_identity_pairs returns it.
 * How: the unchanged identity sweep runs over blocks of query rows into a fixed scratch of max(d_end - d_begin, 2^22)
 * pairs, starting with the whole range; a block whose survivors overflow it is swept again in smaller blocks, and blocks
 * grow again while survivors stay sparse.  Each block's survivors are bucketed by query on the device and each bucket is
 * reduced to its top k_best there (topk.cu), straight into the output table; one copy to the host at the end.  Extra device
 * memory is the output table plus the fixed scratch: it does not grow with the number of hits.
 * mc2_debug_last_sweep afterwards: n_exact summed over every block sweep run, coarse = 1 iff every one took the coarse form.
 * One strand: mc2_identity_topk_both_strands ranks each pair's better strand. */
int mc2_identity_topk(mc2_ctx *ctx, const mc2_model *model, double min_identity, uint32_t k_best, const mc2_hset *set_q,
		      uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end, int32_t upper_only,
		      int32_t exclude_self, double cutoff, uint64_t *out_d, double *out_identity, uint32_t *out_count,
		      uint64_t *out_n_hits, uint64_t *n_scored);

/* Both-strand top-K identity search: for each query row r in [q_begin, q_end), its k_best best database hits over both
 * strands, with the strand of each.
 * Hits: exactly the pairs (r, c) that mc2_identity_pairs_both_strands returns for the same arguments (and a large enough
 * max_out): the identity is max(id+, id-), the same bits that call reports, and the strand is the one it reports (0 forward,
 * 1 reverse, equal identities forward).  exclude_self != 0 drops (r, r) on both strands; it needs set_q == set_d.
 * Order: that of mc2_identity_topk (identity descending, then database row ascending, -0.0 equal to +0.0).  A (r, c) pair
 * appears once after the strand merge, so the order stays total; the strand is payload and never takes part in it.  The
 * result therefore does not depend on survivor order, block sizes or how the query rows are split over calls or GPUs.
 * Outputs: out_d, out_identity and out_strand (may be NULL) are (q_end - q_begin) x k_best, row-major; row r - q_begin holds
 * the first min(k_best, hits) entries; unused slots hold d = UINT64_MAX, identity -1.0 and strand -1.  out_count and
 * out_n_hits (may be NULL; the hit count over both strands) as in mc2_identity_topk.  *n_scored (may be NULL) is the forward
 * in-window pair count, as mc2_identity_pairs_both_strands reports it.
 * MC2_ERR_ARG, MC2_ERR_FEATURE: as mc2_identity_topk.
 * How: one loop over blocks of query rows (the first block is the whole range) sweeps each block's rows forward and, for
 * min_identity > 0, on the reverse-complement set, each into its own scratch of max(d_end - d_begin, 2^22) pairs; a block
 * whose survivors overflow either scratch is swept again in smaller blocks.  The forward survivors keep max(id+, id-) with
 * its strand; the reverse survivors whose id+ fails the threshold (the forward sweep's own decision) join them on strand 1;
 * both lists are bucketed by query and each bucket is reduced to its top k_best on the device (topk.cu).  Extra device memory
 * is the output table plus scratches of fixed size: it does not grow with the number of hits.  The reverse-complement set
 * of set_q is built on first use and kept, as in mc2_identity_pairs_both_strands.
 * mc2_debug_last_sweep afterwards: n_exact summed over every sweep of both strands, coarse = 1 iff every one took the coarse
 * form. */
int mc2_identity_topk_both_strands(mc2_ctx *ctx, const mc2_model *model, double min_identity, uint32_t k_best,
				   const mc2_hset *set_q, uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin,
				   uint64_t d_end, int32_t upper_only, int32_t exclude_self, double cutoff, uint64_t *out_d,
				   double *out_identity, int8_t *out_strand, uint32_t *out_count, uint64_t *out_n_hits,
				   uint64_t *n_scored);

/* Identity clustering: single-linkage clusters (connected components) of the identity graph over rows [begin, end) of set.
 * Vertices: the rows [begin, end).  Edges: exactly the pairs (r, c), r < c, that mc2_identity_pairs(set, [q_begin, q_end), set,
 * [begin, end), upper_only = 1, cutoff) returns (same length window, feature order compute(database c, query r), same decision
 * on the same bits); with both_strands != 0 exactly those mc2_identity_pairs_both_strands returns (max(id+, id-) >= t).
 * begin <= q_begin <= q_end <= end: a query sub-range covers part of the triangle (q_begin == q_end: no edge).
 * out_label[i - begin] = the smallest row of row i's component, as an absolute row number (a row without an edge is its own
 * label); *n_components = the number of distinct labels.  The label is canonical: it does not depend on block sizes, on how
 * the query rows are split over calls (join the parts with mc2_components_merge) or GPUs.  *n_scored (may be NULL) is the
 * forward in-window pair count, equal to mc2_identity_pairs' for the same ranges.
 * MC2_ERR_ARG: a classifier model, a NaN min_identity, a NULL set / out_label / n_components, [q_begin, q_end) not inside
 * [begin, end), end > the set's rows, end - begin >= 2^32, and the (query row, 32-column block) and cutoff checks of
 * mc2_identity_pairs.  MC2_ERR_FEATURE as mc2_identity_pairs returns it.
 * How: the unchanged identity sweep runs over blocks of query rows (the first block is the whole range) into a scratch of
 * max(end - begin, 2^24) pairs per strand (with both_strands and min_identity > 0 the block's rows are swept again on the
 * reverse-complement set, built on first use and kept as in mc2_identity_pairs_both_strands); a block whose survivors
 * overflow it is swept again in smaller blocks.  Each block's survivors are joined on the device into a union-find over the
 * rows (components.cu) as soon as the block is swept, and dropped; one flatten and one copy to the host at the end.  Extra
 * device memory: 24 bytes per scratch pair per strand, plus 12 bytes per row; it does not grow with the number of edges.
 * min_identity <= 0 is served through the same sweeps (every in-window pair is an edge).
 * mc2_debug_last_sweep afterwards: n_exact summed over every sweep of both strands, coarse = 1 iff every one took the coarse
 * form (0 when there was no sweep). */
int mc2_identity_components(mc2_ctx *ctx, const mc2_model *model, double min_identity, int32_t both_strands, const mc2_hset *set,
			    uint64_t q_begin, uint64_t q_end, uint64_t begin, uint64_t end, double cutoff, uint64_t *out_label,
			    uint64_t *n_components, uint64_t *n_scored);

/* Identity clustering: greedy representative clusters of the identity graph over rows [begin, end) of set, as CD-HIT and
 * UCLUST build them (CD-HIT's -g 1, "most similar" assignment).  Single linkage (mc2_identity_components) chains; here no
 * member is further than min_identity from its representative.
 * Graph: the vertices are the rows [begin, end); the edges are exactly the pairs (r, c), r < c, that mc2_identity_pairs(set,
 * [begin, end), set, [begin, end), upper_only = 1, cutoff) returns (same length window, feature order compute(database c,
 * query r), so the earlier row is the query, same decision on the same bits), or with both_strands != 0 exactly those
 * mc2_identity_pairs_both_strands returns.  Edge weight w(r, c): the identity that call reports, bit for bit (on both strands
 * max(id+, id-), with the strand it reports).
 * Representatives: c = begin .. end - 1 is visited in ascending order, and row c is a representative iff no representative
 * r < c has an edge (r, c) (the lexicographically first maximal independent set in row order).  ROW ORDER IS THE VISITING
 * ORDER: for CD-HIT's longest-first order, build the set with its rows in that order.
 * Assignment: every other row c goes to the representative r < c with an edge (r, c) of the largest w; on a numeric tie
 * (-0.0 equals +0.0) the smallest r.  Only earlier representatives count, as in CD-HIT.
 * Outputs, indexed by i - begin: out_rep = the representative as an absolute row (a representative is its own);
 * out_identity (may be NULL) = w(rep, i), the same bits the flat call reports for that pair, -1.0 for a representative;
 * out_strand (may be NULL) = 0 or 1 (always 0 without both_strands), -1 for a representative.  *n_clusters = the number of
 * representatives; *n_scored (may be NULL) = the forward in-window pair count, equal to mc2_identity_pairs' for the same
 * ranges.  The result does not depend on block sizes.
 * MC2_ERR_ARG: a classifier model, a NaN min_identity, a NULL set / out_rep / n_clusters, begin > end or end > the set's
 * rows, end - begin >= 2^32, cutoff <= 0, more than 2^32 (query row, 32-column block) groups.  MC2_ERR_FEATURE as
 * mc2_identity_pairs returns it.  min_identity <= 0 is served through the same sweeps (every in-window pair is an edge).
 * How: the unchanged identity sweep runs over blocks of query rows in row order (the first block is the whole range) into
 * the scratch of mc2_identity_components, max(end - begin, 2^24) pairs per strand; with both_strands the block's pairs are
 * merged over the strands as in mc2_identity_topk_both_strands.  An edge arrives with the block of its smaller row, so when
 * a block arrives every earlier row is final.  Each block's edges are bucketed by their larger row; one cooperative launch
 * decides the block's rows in rounds, with no host round trip (greedy.cu), and one more brings every later row's best
 * in-edge from a representative up to date.  Extra device memory: 40 bytes per scratch pair on one strand (91 on both),
 * plus 50 bytes per row; it does not grow with the number of edges.
 * mc2_debug_last_sweep afterwards: as for mc2_identity_components. */
int mc2_identity_greedy_clusters(mc2_ctx *ctx, const mc2_model *model, double min_identity, int32_t both_strands,
				 const mc2_hset *set, uint64_t begin, uint64_t end, double cutoff, uint64_t *out_rep,
				 double *out_identity, int8_t *out_strand, uint64_t *n_clusters, uint64_t *n_scored);

/* Staged greedy clustering: mc2_identity_greedy_clusters split into stages that a caller can spread over calls and GPUs.
 * The result of mc2_greedy_end is bit for bit that of mc2_identity_greedy_clusters with the same model, min_identity,
 * both_strands, set, [begin, end) and cutoff (out_rep, out_identity, out_strand, *n_clusters; the n_scored of the sweeps of
 * the blocks added sum to its *n_scored), whatever the block tiling, the split of each block into parts, the order of the
 * sweeps and the calls made between stages: the result depends only on the edge set and the row order.
 * The object sweeps query-row blocks [qb, qe) in row order, starting at the next undecided row (begin at first):
 *   1. mc2_greedy_sweep_part(part p, [q_begin, q_end)) sweeps those query rows against the columns (r, end) into slot p: its
 *      records are exactly the edges (r, c), r in [q_begin, q_end), that mc2_identity_greedy_clusters takes, with the same
 *      identity bits and strand.  *n_edges = how many (may exceed the capacity; the slot's contents are then unspecified and
 *      the caller sweeps a smaller block), *n_scored = the forward in-window pair count.  Returns once the slot is written.
 *   2. The caller may copy slots between objects (one per GPU, each with n_parts = the number of GPUs): a slot is
 *      mc2_greedy_part_buffers' *capacity records of 16 bytes {uint32 r - begin, uint32 c - begin, float64 identity} at
 *      *d_records (device memory) and, with both_strands, *capacity strand bytes at *d_strand (NULL on one strand); only the
 *      first n_edges of each are read.
 *   3. mc2_greedy_add_block(qb, qe, part ranges, part edge counts) decides the rows of [qb, qe) from every slot's records.
 *      The part ranges tile [qb, qe) in part order (empty ranges allowed).  Every record is checked on the device first (r
 *      in its part's range, c in (r, end)); a bad one gives MC2_ERR_ARG and leaves the object unchanged.  Returns once the
 *      slots have been read.
 * mc2_greedy_end writes the outputs once every row up to end has been added.  The set (and its reverse complement) must not
 * change or be freed while the object lives; the object keeps its own copy of the model.  Calls on other objects and any
 * other call may run between stages on the same context.
 * part_capacity: records per slot; 0 = max(end - begin, ceil(2^24 / n_parts)).  One query row has at most end - begin - 1
 * edges, so a one-row block always fits.
 * Extra device memory of the object, n = end - begin, E = n_parts x part_capacity: 50 n + 32 E bytes on one strand, 50 n +
 * 34 E on both, plus 24 n_parts + 44.  A sweep uses the context's scratch: 24 part_capacity bytes on one strand, 56 on
 * both.  None of it grows with the number of edges.
 * MC2_ERR_ARG: the checks of mc2_identity_greedy_clusters (at begin); n_parts == 0; part_capacity below end - begin; a part
 * index >= n_parts; a sweep range outside [next undecided row, end); a block that does not start at the next undecided row
 * or ends past end; part ranges that do not tile the block; a count above part_capacity; a bad record; mc2_greedy_end before
 * every row was added; a NULL argument.
 * mc2_debug_last_sweep after mc2_greedy_sweep_part: as for the flat identity calls. */
typedef struct mc2_greedy mc2_greedy;
int mc2_greedy_begin(mc2_ctx *ctx, const mc2_model *model, double min_identity, int32_t both_strands, const mc2_hset *set,
		     uint64_t begin, uint64_t end, double cutoff, uint32_t n_parts, uint64_t part_capacity, mc2_greedy **out);
int mc2_greedy_sweep_part(mc2_ctx *ctx, mc2_greedy *g, uint32_t part, uint64_t q_begin, uint64_t q_end, uint64_t *n_edges,
			  uint64_t *n_scored);
int mc2_greedy_part_buffers(const mc2_greedy *g, uint32_t part, void **d_records, int8_t **d_strand, uint64_t *capacity);
int mc2_greedy_add_block(mc2_ctx *ctx, mc2_greedy *g, uint64_t qb, uint64_t qe, const uint64_t *part_q_begin,
			 const uint64_t *part_q_end, const uint64_t *part_edges);
int mc2_greedy_end(mc2_ctx *ctx, mc2_greedy *g, uint64_t *out_rep, double *out_identity, int8_t *out_strand,
		   uint64_t *n_clusters);
void mc2_greedy_free(mc2_greedy *g);

/* The union of n_parts partitions of the rows [begin, end): labels holds n_parts row-major arrays of end - begin labels in
 * [begin, end) each (for example mc2_identity_components over disjoint query sub-ranges, or from different GPUs).  Joining
 * the edges {i, labels_p[i]} of every part gives exactly the components of the union of the parts' edge sets; out_label and
 * *n_components as in mc2_identity_components (the smallest row of each component).  The labels are checked on the host
 * before the upload.  Extra device memory: 8 bytes per label plus 12 bytes per row.
 * MC2_ERR_ARG: n_parts == 0, a label outside [begin, end), end < begin, end - begin >= 2^32, a NULL pointer. */
int mc2_components_merge(mc2_ctx *ctx, uint64_t begin, uint64_t end, uint32_t n_parts, const uint64_t *labels,
			 uint64_t *out_label, uint64_t *n_components);

/* Measured issue rate (warp-instructions per second, whole GPU) of the tile sweep's inner instruction pair -- VIMNMX.U16x2 on
 * the ALU pipe feeding IDP.2A on the FMA pipe, register operands only, 32 resident warps per SM: the denominator of
 * bench.py's roofline for the CUDA-core EMD term (SURVEY.md section 8d: "achieved ... vs a measured ALU peak"). */
int mc2_bench_issue_rate(mc2_ctx *ctx, int iters, double *warp_instr_per_s);

/* Diagnostic (tests): the integer reductions of the tile sweep for every (query, database) pair of the two row ranges, as
 * dense row-major (q_end-q_begin) x (d_end-d_begin) uint32 matrices: need is a mask of 1 = sum|p-q| (Feature.cpp:858-871),
 * 2 = sum p*q (Feature.cpp:1112-1124, 1170-1184), 4 = sum|cumP-cumQ| (Feature.cpp:1504-1518).  Outputs not selected by
 * `need` may be NULL.  No length window, no model.  Sets of uint8 / uint16 rows of whole 1 KiB slabs (k >= 5, at most 4^8
 * bins) whose row sums fit 16 bits once the pseudo-count per bin is taken out; MC2_ERR_UNSUPPORTED when the rows do not
 * fit the tile form (a uint16 bin above 255, a bin below the pseudo-count in rows that need it taken out). */
int mc2_debug_tile_reductions(mc2_ctx *ctx, const mc2_hset *set_q, uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d,
			      uint64_t d_begin, uint64_t d_end, int32_t need, uint32_t *out_dot, uint32_t *out_emd, uint32_t *out_sad);

/* Diagnostic (tests, benchmarks): of the last mc2_all_pairs / mc2_identity_pairs call on this context (for
 * mc2_identity_pairs_both_strands, the top-K searches and mc2_identity_components see there), *n_exact = the pairs the tile sweep sent through the exact fp64 epilogue (those its fp32 screen could not reject; 0 for the row-streaming
 * kernels) and *coarse = 1 if it took the coarse form (the screen on 64 sampled cumulative bins), else 0.  *n_inline (may
 * be NULL) = how many of the n_exact pairs the coarse form refined inside the sweep because its candidate buffer (2^23
 * records) was full; the others were refined by the kernel that follows the sweep. */
int mc2_debug_last_sweep(mc2_ctx *ctx, uint64_t *n_exact, int32_t *coarse, uint64_t *n_inline);

/* DivergencePoint<T>::distance (src/clutil/DivergencePoint.cpp:70-82) for pairs of rows */
int mc2_distance(mc2_ctx *ctx, const mc2_pairs *pairs, uint64_t *out);

/* K3 — cluster mean + closest member: get_mean (src/cluster/ClusterFactory.cpp:338-380) and the mean of mean_shift_update
 * (:288-335) followed by Trainer<T>::closest (src/cluster/Trainer.cpp:144-157).  mean = per-bin average (double) of rows
 * members[0..n) of `set`; *best = position in members of the FIRST member minimising DivergencePoint<T>::distance_d to that
 * mean (src/clutil/DivergencePoint.cpp:55-66, with its per-bin u64 truncation), *best_dist its distance.
 * mean_out (4^k doubles) and dist_out (n doubles) may be NULL. */
int mc2_mean_closest(mc2_ctx *ctx, const mc2_hset *set, const uint64_t *members, uint64_t n, int64_t *best, double *best_dist,
		     double *mean_out, double *dist_out);

/* Trainer<T>::closest (src/cluster/Trainer.cpp:144-157) alone: the mean is supplied by the caller (the Point<double> that
 * mean_shift_update built on the host); returns the first member minimising distance_d to it. */
int mc2_closest(mc2_ctx *ctx, const mc2_hset *set, const uint64_t *members, uint64_t n, const double *mean, int64_t *best,
		double *best_dist, double *dist_out);

/* Device-timed variants used by bench.py: run the scoring kernel `iters` times on inputs already resident
 * (pair lists uploaded once), return the average milliseconds per launch measured with CUDA events on the ctx stream. */
int mc2_bench_score_pairs(mc2_ctx *ctx, const mc2_model *model, const mc2_pairs *pairs, int iters, int flush_l2,
			  float *avg_ms, uint64_t *n_close);
int mc2_bench_count_kmers(mc2_ctx *ctx, const mc2_seqs *seqs, int k, int elem_bytes, int iters, int flush_l2,
			  float *avg_ms);

#ifdef __cplusplus
}
#endif
#endif
