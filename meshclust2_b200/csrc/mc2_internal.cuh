// mc2_internal.cuh — shared device/host structures of libmeshclust2_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string>
#include "../../include/meshclust2_b200.h"

typedef unsigned long long u64;
typedef long long s64;
typedef unsigned int u32;

namespace mc2 {

void set_error(const std::string &msg);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define MC2_CUDA(expr)                                                         \
	do {                                                                   \
		cudaError_t _e = (expr);                                       \
		if (_e != cudaSuccess) {                                       \
			return mc2::cuda_fail(_e, #expr, __FILE__, __LINE__);  \
		}                                                              \
	} while (0)

#define MC2_REQUIRE(cond, msg)                         \
	do {                                           \
		if (!(cond)) {                         \
			mc2::set_error(msg);           \
			return MC2_ERR_ARG;            \
		}                                      \
	} while (0)

// internal single-feature codes (dense, so the kernel can switch on a small int)
enum SingleCode : int {
	SC_MANHATTAN = 0,
	SC_EUCLIDEAN,
	SC_NORMALIZED_VECTORS,
	SC_JEFFEREY,
	SC_PEARSON,
	SC_INTERSECTION,
	SC_EMD,
	SC_LENGTHD,
	SC_KULCZYNSKI2,
	SC_SIMRATIO,
	SC_JENSEN_SHANNON,
	SC_COUNT
};

// Slots of the tile sweep's screen scratch: the fast singles the kernel instantiation computes (those its reductions
// `need` give: 1 = sum|p-q|, 2 = sum p*q, 4 = sum|cumP-cumQ|; length_difference always), densely, then the constant 1.
__host__ __device__ constexpr bool scr_has(int need, int code)
{
	return (code == SC_MANHATTAN || code == SC_INTERSECTION || code == SC_KULCZYNSKI2) ? (need & 1) != 0 :
	       (code == SC_EUCLIDEAN || code == SC_NORMALIZED_VECTORS || code == SC_PEARSON || code == SC_SIMRATIO) ? (need & 2) != 0 :
	       code == SC_EMD ? (need & 4) != 0 : code == SC_LENGTHD;
}
__host__ __device__ constexpr int scr_slot(int need, int code)
{
	int n = 0;
	for (int c = 0; c < SC_COUNT; c++) {
		if (c == code) {
			return n; // meaningful only for singles the instantiation has
		}
		n += scr_has(need, c) ? 1 : 0;
	}
	return n; // code == SC_COUNT: the constant 1
}
__host__ __device__ constexpr int scr_slots(int need)
{
	return scr_slot(need, SC_COUNT) + 1;
}

#define MC2_SCR_MAX_COMBOS 8

// which reductions over the bins a model needs
enum NeedBits : int { NEED_MIN = 1, NEED_DOT = 2, NEED_EMD = 4, NEED_LOG = 8 };

struct DevModel {
	int n_singles;
	int code[MC2_MAX_SINGLES];
	int is_sim[MC2_MAX_SINGLES];
	double smin[MC2_MAX_SINGLES];
	double smax[MC2_MAX_SINGLES];
	int n_combos;
	int kind[MC2_MAX_COMBOS];
	int nidx[MC2_MAX_COMBOS];
	int idx[MC2_MAX_COMBOS][MC2_MAX_COMBO_IDX];
	double weight[MC2_MAX_COMBOS + 1];
	double bias;
	int regression;
	int need;
	// straight-line epilogue (eval_pair_fast): constants indexed by single CODE instead of by position, so the kernel
	// reads them at fixed constant-bank offsets.  slot = position of the code in the model's cache order, -1 = absent.
	int fast_epi;                 // 0: a single appears twice -> interpretive epilogue only
	int slot[SC_COUNT];
	int csim[SC_COUNT];
	int crcp_ok[SC_COUNT];        // crcp usable (finite, normal range): division by crange = two fused multiply-adds
	double cmin[SC_COUNT];
	double crange[SC_COUNT];      // max - min, the divisor of Feature::normalize_cache (Feature.cpp:136-154)
	double crcp[SC_COUNT];        // correctly rounded 1 / crange
	// fp32 screen of the tile sweep (tile_sweep.cu): normalised single = scr_a * raw + scr_b; combo c is
	// x[scr_ka[c]]^(1 + scr_pa2[c]) * x[scr_kb[c]]^(1 + scr_pb2[c]) with single CODES as indices (SC_COUNT = the constant 1);
	// |fp32 sum - exact sum| <= scr_k1 * (1 + max |x|)^4 + scr_k0 (derivation: build_screen in mc2_api.cu)
	int scr_ok;                   // 0: the model is outside what the screen covers -> every pair takes the exact path
	float scr_a[SC_COUNT], scr_b[SC_COUNT];
	float scr_w[MC2_SCR_MAX_COMBOS + 1];
	int scr_ka[MC2_SCR_MAX_COMBOS], scr_kb[MC2_SCR_MAX_COMBOS], scr_pa2[MC2_SCR_MAX_COMBOS], scr_pb2[MC2_SCR_MAX_COMBOS];
	float scr_k1, scr_k0;
	float scr_dx;                 // |fl(x) - x| <= scr_dx * (1 + max |x|) for every single x (the coarse form's sign test)
	// a pair whose fp32 sum + bound stays below this is not close: logit(0.5 - bias) - margin for a classifier; for a
	// regression model it is set per call on a copy (min_identity - margin, mc2_identity_pairs)
	float scr_thr;
};

// Mailbox of the resident scan server: the accumulate stage of the mean-shift driver issues one Trainer::get_close per
// query, each depending on the previous result (src/cluster/ClusterFactory.cpp:560-605), tens of candidates at a time, so
// the cost of a call is launch + copy latency.  The host writes a request into this mapped page-locked block and bumps
// `seq`; a resident CTA polls it, scores the candidates, reduces the arg-max and writes the answer back; the host polls
// `seq_done`.  No launch, no memcpy, no stream synchronisation per call.
#define MC2_SCAN_CAP 512        // longer candidate lists take the launch path
#define MC2_SCAN_INLINE 80      // candidates that travel inside the request header (32-bit row numbers, two per word)
// the header word that holds inline ids 2k and 2k + 1 (the words between the fixed fields and the sequence copies)
__host__ __device__ constexpr int scan_id_word(int k) { return k < 3 ? 20 + k : k < 10 ? 24 + (k - 3) : k < 25 ? 32 + (k - 10) : 48 + (k - 25); }
#define MC2_SCAN_MARKS_INLINE 192 // marks that travel inside the answer line (one bit each)
struct ScanMailbox {
	// Request header: 64 words = four 128-byte lines, fetched by the server with ONE coalesced read per poll (16 bytes per
	// lane).  The host writes word 0 (the sequence number) last and repeats it in words 15, 23, 31, 47 and 63, so a header
	// whose copies agree is complete even if the lines were fetched separately.
	//  [0] seq  [1] q_row  [2] q_mag  [3] q_len  [4] cand_begin  [5] cutoff (double bits)
	//  [6] n_cand | has_list << 32 | ovr << 33 | ids inline << 34   [7] quit
	//  [8] binsQ  [9] binsC  [10] magQ  [11] sumQ  [12] sumsqQ  [13] lenQ  [14] N  [15] seq
	//  [16] magC  [17] sumC  [18] sumsqC  [19] lenC  [20..22] ids 0-5  [23] seq  [24..30] ids 6-19  [31] seq
	//  [32..46] ids 20-49  [47] seq  [48..62] ids 50-79  [63] seq
	volatile unsigned long long w[64];
	unsigned long long cand[MC2_SCAN_CAP];      // the whole list when it is longer than MC2_SCAN_INLINE
	// answer (written by the device with one eight-lane store): one 64-byte line, the sequence number closing both halves
	//  [0] best  [1] best_dist (double bits)  [2] is_min | err << 32  [3] seq_done  [4..6] mark bits of the first 192 candidates
	//  [7] seq_done
	volatile unsigned long long r[8];
	volatile int running;
	int pad1[15];
	unsigned char marks[MC2_SCAN_CAP];          // all marks when there are more than MC2_SCAN_MARKS_INLINE candidates
};
static_assert(offsetof(ScanMailbox, cand) == 512, "the scan server reads the request header as 64 eight-byte words");

// side-band SoA of a histogram set (device pointers)
struct Sideband {
	const u64 *mag;   // pseudo-magnitude as the host object reports it (may be stale, quirk Q4)
	const u64 *sum;   // true sum of the bins
	const u64 *sumsq; // true sum of squared bins (exact for u8/u16; wraps like the reference's u64 for wider)
	const u64 *len;   // get_length()
};

} // namespace mc2

struct mc2_ctx {
	int device;
	int sm_count;
	cudaStream_t stream;
	cudaEvent_t ev0, ev1;
	u64 launches;
	// scratch
	void *flush_buf;
	size_t flush_bytes;
	int *d_err;       // device error word (sticky per call)
	int *h_err;       // pinned mirror
	void *h_slot;     // pinned result slot (4 KB)
	void *d_slot;     // device result slot (4 KB)
	void *extra;      // CtxExtra (growable scratch buffers), owned by mc2_api.cu
	int prof_on;      // per-kernel event timing enabled
	int err_dirty;    // the device error word may be non-zero (set by reset_err, cleared by a clean check_err)
	void *d_sched;    // tile schedule of the tile sweep (tile_sweep.cu), allocated on first use
	void *d_cand;     // the coarse tile sweep's candidate buffer (tile_sweep.cu), allocated on first use
	// resident scan server (pair_score.cu scan_server_kernel): mailbox in mapped page-locked memory, its own stream
	mc2::ScanMailbox *mb;
	cudaStream_t server_stream;
	u64 mb_seq;           // sequence number of the last request posted
	u64 server_model_uid; // model the running server was launched with
	int server_eb;
};

namespace mc2 {
// event-pair bracket around one kernel launch when profiling is on (no-ops otherwise)
void prof_begin(mc2_ctx *ctx, int kind);
void prof_end(mc2_ctx *ctx);
}

struct mc2_seqs {
	mc2_ctx *ctx;
	u64 n;
	u64 total_bases;
	u64 max_len;
	u32 *packed;      // 2-bit packed, big-endian within each 32-bit word; every sequence starts on a 16-byte boundary
	u64 *word_off;    // [n+1] word offset of each sequence
	u64 *len;         // [n] bases
	int *segs;        // [2*total_segs] inclusive, sequence-relative
	u64 *seg_off;     // [n+1]
	u64 total_segs;
	u64 total_words;
	u64 min_seg_len;  // shortest segment (bases); ~0 when there is none
	u64 cap_packed, cap_word_off, cap_len, cap_segs, cap_seg_off; // bytes allocated (grow-only, mc2_seqs_upload_into)
};

struct mc2_hset {
	mc2_ctx *ctx;
	u64 n;
	int k;
	u64 N;
	int eb;
	void *bins;       // n x N elements
	u64 *mag, *sum, *sumsq, *len;
	u64 *mers1;       // n x 4 (0 when built from host)
	double *stddev;   // n
	int *novf;        // n
	u32 *maxc;        // n : largest unsaturated count+1
	u64 max_sum;      // host-known upper bound of sum[] (selects fast paths)
	u64 max_count;    // host-known max of maxc[] (raw multiplicity; valid while `counted`)
	int counted;      // rows came from mc2_count_kmers(_into) with init 1 and were not overwritten since
	// 1 KiB uint8 rows only: exclusive prefix of the bin sums at the 32 lane boundaries (bins [32l, 32l+32) belong to lane
	// l), u16, n x 32.  Lets the EMD reduction start each lane's prefix chain without a per-pair warp scan.  Built lazily,
	// dropped whenever bins change.
	unsigned short *lane_off;
	int lane_off_valid;
	// Operands of the tile sweep (tile_sweep.cu; uint8 / uint16 rows of whole 1 KiB slabs): inclusive cumulative rows of
	// (bin - cum_base) as u16 (n x N), each row's sum of them (u32), and for uint16 bins the rows as bytes.  Built lazily,
	// dropped whenever bins change.  cum16_valid: 0 not built, 1 built, -1 the set cannot be served with cum_base.
	// Rows of one slab (N = 1024) also get cum16s: the cumulative values at bins 16 j + 15 (n x 64, u16), the operand of
	// the tile sweep's coarse form; same lifetime as cum16.
	unsigned short *cum16;
	unsigned short *cum16s;
	u32 *cumsum;
	unsigned char *plane8;
	int cum16_valid;
	int cum_base;
	// the reverse-complement set (strand.cu) that mc2_identity_pairs_both_strands sweeps for the other strand of these rows;
	// built lazily, freed whenever bins, magnitudes or lengths change.
	mc2_hset *rc;
};

struct mc2_model {
	mc2_ctx *ctx;
	mc2_model_desc desc;
	mc2::DevModel dm;
	u64 uid; // identifies the model a resident scan server was started with
};

namespace mc2 {

// launchers implemented in the .cu files
struct PairArgs {
	const void *binsA;
	const void *binsB;
	Sideband sbA, sbB;
	u64 N;
	int eb;
	u64 n_pairs;
	const u64 *ia; // device or NULL
	const u64 *ib;
	u64 a_begin, b_begin;
	int a_bc, b_bc;
	int len_filter, anchor_is_b;
	double cutoff;
	double *score;
	double *dist;
	uint8_t *close;
	double *cache;
	double *raw;
	uint8_t *skipped;
	u64 *n_close;  // optional device counter
	int *err;      // device error word
	u64 max_sum;   // bound on bin sums of both sets
	const unsigned short *loffA, *loffB; // lane-boundary prefix sums (see mc2_hset::lane_off) or NULL
	int group;     // pairs per warp group (1..32, power of two; 0 = 32): small batches of wide rows spread over more warps
};

int launch_pair_score(mc2_ctx *ctx, const DevModel &dm, const PairArgs &a);
// text_ingest.cu
int launch_segment(mc2_ctx *ctx, bool write, const char *d_text, const u64 *d_seq_off, u64 n, u32 *d_count, const u64 *d_seg_off,
		   int *d_segs, unsigned long long *d_min_seg);
int launch_seg_scan(mc2_ctx *ctx, const u32 *d_count, u64 n, u64 *d_seg_off);
int launch_pack_text(mc2_ctx *ctx, const char *d_text, const u64 *d_seq_off, mc2_seqs *s);
int launch_argmax(mc2_ctx *ctx, const double *dist, const uint8_t *skipped, const uint8_t *close, u64 n, int mode, void *d_out,
		  uint8_t *d_flags_out = nullptr);
int launch_count(mc2_ctx *ctx, const mc2_seqs *s, int k, int eb, mc2_hset *h, u64 init_value);
int launch_sideband(mc2_ctx *ctx, mc2_hset *h, bool set_mag);
int launch_pack(mc2_ctx *ctx, const char *d_codes, const u64 *d_seq_off, mc2_seqs *s);
// identity != 0 (mc2_identity_pairs, regression models): a pair survives on score >= min_identity instead of `close`
int launch_all_pairs(mc2_ctx *ctx, const DevModel &dm, const mc2_hset *q, u64 q0, u64 q1, const mc2_hset *d, u64 d0, u64 d1,
		     int upper_only, double cutoff, u64 max_out, u64 *d_out_q, u64 *d_out_d, double *d_out_score,
		     u64 *d_counters, int identity, double min_identity);
int launch_distance(mc2_ctx *ctx, const PairArgs &a, u64 *d_out);
int ensure_lane_off(mc2_ctx *ctx, const mc2_hset *h); // builds h->lane_off if the shape allows; no-op otherwise
// tile_sweep.cu: the all-pairs sweep over 1 KiB uint8 rows as 64 x 128 pair tiles (TMA ring, tcgen05 Gram term, u16 cumulative EMD)
int ensure_tile_operands(mc2_ctx *ctx, const mc2_hset *h, int base);
// identity: the model must be a regression model (identity search), else a classifier (mc2_all_pairs)
bool tile_sweep_supported(const DevModel &dm, const mc2_hset *q, const mc2_hset *d, int identity);
bool tile_sweep_shape_ok(const mc2_hset *q, const mc2_hset *d);
int launch_issue_probe(mc2_ctx *ctx, int iters, u32 *d_out, u64 *warp_instr);
// pair_score.cu: start the resident scan server for 1- or 2-byte bins on ctx->server_stream
int launch_scan_server(mc2_ctx *ctx, const DevModel &dm, int eb, u64 first_seq);
int launch_tile_sweep(mc2_ctx *ctx, const DevModel &dm, int need, const mc2_hset *q, u64 q0, u64 q1, const mc2_hset *d, u64 d0, u64 d1,
		      int upper_only, double cutoff, u64 max_out, u64 *d_out_q, u64 *d_out_d, double *d_out_score, u64 *d_counters,
		      u32 *raw_dot, u32 *raw_emd, u32 *raw_sad, int identity, double min_identity);
int launch_mean_closest(mc2_ctx *ctx, const mc2_hset *h, const u64 *d_members, u64 n, u64 *d_sums, double *d_mean, double *d_dist,
			void *d_out, bool have_mean);
int launch_update_batch(mc2_ctx *ctx, const mc2_hset *h, const u64 *d_member_off, const u64 *d_members, const uint8_t *d_close,
			const uint8_t *d_skipped, u64 c_begin, u64 count, double *d_mean, long long *d_next, u64 *d_n_good);
// strand.cu: dst (same shape as src) receives the reverse-complement bins and the swapped k = 1 table of every row
int launch_revcomp(mc2_ctx *ctx, const mc2_hset *src, mc2_hset *dst);
int launch_strand_pick(mc2_ctx *ctx, double *score, const double *rev, int8_t *strand, u64 n);
int launch_strand_append(mc2_ctx *ctx, const u64 *bq, const u64 *bd, const double *bs, const double *fwd, u64 n, double t,
			 u64 *counter, u64 max_out, u64 *oq, u64 *od, double *os, int8_t *ostr);
// topk.cu: survivors (sq, sd, ss)[0..n) of query rows [qb, ...) -> per-query counts, buckets at the counts' exclusive scan
// off, and each query's first k_best (1..1024) entries by (identity desc, d asc) into its output row.  by_d: the count and
// scatter bucket by database row d - qb instead, and the bucket holds (identity, q); no self pair is dropped.
int launch_topk_count(mc2_ctx *ctx, const u64 *sq, const u64 *sd, u64 n, u64 qb, int exclude_self, bool by_d, u32 *cnt);
int launch_topk_scatter(mc2_ctx *ctx, const u64 *sq, const u64 *sd, const double *ss, u64 n, u64 qb, int exclude_self, bool by_d,
			const u64 *off, u32 *cur, double *bid, u64 *bd);
int launch_topk_select(mc2_ctx *ctx, const u64 *off, const double *bid, const u64 *bd, u64 rows, u32 k_best, u64 d_begin,
		       u64 *out_d, double *out_id, u32 *out_cnt, u64 *out_hits);
// the same with a strand per entry: a list with fwd != NULL keeps only its entries with !(fwd[i] >= t); sstr NULL = strand 1
int launch_topk_count_strand(mc2_ctx *ctx, const u64 *sq, const u64 *sd, const double *fwd, double t, u64 n, u64 qb,
			     int exclude_self, bool by_d, u32 *cnt);
int launch_topk_scatter_strand(mc2_ctx *ctx, const u64 *sq, const u64 *sd, const double *ss, const int8_t *sstr,
			       const double *fwd, double t, u64 n, u64 qb, int exclude_self, bool by_d, const u64 *off, u32 *cur,
			       double *bid, u64 *bd, int8_t *bstr);
int launch_topk_select_strand(mc2_ctx *ctx, const u64 *off, const double *bid, const u64 *bd, const int8_t *bstr, u64 rows,
			      u32 k_best, u64 d_begin, u64 *out_d, double *out_id, int8_t *out_str, u32 *out_cnt,
			      u64 *out_hits);
// components.cu: union-find over rows [begin, begin + n) in a uint32 parent array relative to begin; init sets parent[i] = i,
// the hooks join the edges {q[i], d[i]} (absolute rows) or {i mod n, labels[i]} of n_parts stacked label arrays, flatten
// writes out[i] = begin + the smallest row of i's component and *n_roots = the number of components
int launch_cc_init(mc2_ctx *ctx, u32 *parent, u64 n);
int launch_cc_hook_pairs(mc2_ctx *ctx, const u64 *q, const u64 *d, u64 n, u64 begin, u32 *parent);
int launch_cc_hook_labels(mc2_ctx *ctx, const u64 *labels, u64 n_parts, u64 n, u64 begin, u32 *parent);
int launch_cc_flatten(mc2_ctx *ctx, u32 *parent, u64 n, u64 begin, u64 *out, u64 *n_roots);
// greedy.cu: greedy representative clustering over rows [begin, begin + n), state relative to begin.  Per row: status
// (undecided 0, representative 1, member 2), the bucket cursor of the resolve rounds, and the best in-edge from a
// representative so far (rep relative to begin, 0xffffffff none; its identity and strand).  A block of query rows [qb, qb +
// rows) is resolved from the buckets of its edges keyed by database row - qb (off, br: query rows); assign merges each
// bucket of (qb, qb + rows) (here rows = end - qb) into the best in-edges; finish writes out_rep (absolute), out_id
// (-1.0 for a representative), out_str (-1) and *n_reps.
struct GreedyRows {
	u32 *status, *cursor, *rep;
	double *id;
	int8_t *str;
};
int launch_greedy_init(mc2_ctx *ctx, const GreedyRows &g, u64 n);
int launch_greedy_resolve(mc2_ctx *ctx, const u64 *off, const u64 *br, u64 qb, u64 rows, u64 begin, const GreedyRows &g,
			  u32 *remain);
int launch_greedy_assign(mc2_ctx *ctx, const u64 *off, const double *bid, const u64 *br, const int8_t *bstr, u64 qb, u64 rows,
			 u64 begin, const GreedyRows &g);
int launch_greedy_finish(mc2_ctx *ctx, const GreedyRows &g, u64 n, u64 begin, u64 *out_rep, double *out_id, int8_t *out_str,
			 u64 *n_reps);
// the part slots of a staged greedy clustering (mc2_greedy_*): slot p holds records rec[p * cap + j], j < its count, of edges
// (begin + r, begin + c) with their identity, and with both strands a strand byte str[p * cap + j] (str NULL: one strand).
// part[3 p .. 3 p + 2] = (query range begin, end, count) of part p; stride = the largest count.  bad (the count pass; NULL
// in the scatter) is raised by a record with r outside its part's range or c outside (r, end).
struct GreedyEdge {
	u32 r, c;
	double id;
};
struct GreedyParts {
	const GreedyEdge *rec;
	const int8_t *str;
	const u64 *part;
	u64 n_parts, stride, cap, begin, end;
	u32 *bad;
};
int launch_greedy_parts_count(mc2_ctx *ctx, const GreedyParts &parts, u64 qb, u32 *cnt);
int launch_greedy_parts_scatter(mc2_ctx *ctx, const GreedyParts &parts, u64 qb, const u64 *off, u32 *cur, double *bid, u64 *bd,
				int8_t *bstr);
// the first n survivors (sq, sd, ss) as records relative to begin
int launch_greedy_pack(mc2_ctx *ctx, const u64 *sq, const u64 *sd, const double *ss, u64 n, u64 begin, GreedyEdge *out);
int launch_merge_batch(mc2_ctx *ctx, const double *d_dist, const uint8_t *d_skipped, const uint8_t *d_close, const u64 *d_off,
		       u64 n_centers, long long *d_out);

} // namespace mc2
