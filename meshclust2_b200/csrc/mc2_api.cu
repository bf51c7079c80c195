// mc2_api.cu — the C ABI declared in include/meshclust2_b200.h: contexts, device-resident objects, host glue.
// No compute happens on the host here; every entry point launches the sm_100a kernels in kmer_count.cu /
// pair_score.cu / pair_tile.cu or fails loudly.
#include "mc2_internal.cuh"
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <new>
#include <string>
#include <vector>

namespace mc2 {

static thread_local std::string g_err;

void set_error(const std::string &msg)
{
	g_err = msg;
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
	char buf[512];
	snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d in %s", (int)e, cudaGetErrorString(e), file, line, what);
	g_err = buf;
	return MC2_ERR_CUDA;
}

// growable device / pinned scratch
struct Buf {
	void *p = nullptr;
	size_t cap = 0;
	bool pinned = false;
};

static int ensure(Buf &b, size_t bytes, bool pinned)
{
	if (bytes <= b.cap) {
		return MC2_OK;
	}
	if (b.p) {
		if (b.pinned) {
			cudaFreeHost(b.p);
		} else {
			cudaFree(b.p);
		}
		b.p = nullptr;
		b.cap = 0;
	}
	size_t want = bytes + bytes / 4 + 256;
	if (pinned) {
		MC2_CUDA(cudaMallocHost(&b.p, want));
	} else {
		MC2_CUDA(cudaMalloc(&b.p, want));
	}
	b.cap = want;
	b.pinned = pinned;
	return MC2_OK;
}

static void release(Buf &b)
{
	if (b.p) {
		if (b.pinned) {
			cudaFreeHost(b.p);
		} else {
			cudaFree(b.p);
		}
	}
	b.p = nullptr;
	b.cap = 0;
}

enum { B_IA = 0, B_IB, B_SCORE, B_DIST, B_CLOSE, B_SKIP, B_CACHE, B_RAW, B_MISC, B_OUTQ, B_OUTD, B_OUTS, B_STAGE_CODES, B_STAGE_BOFF, B_ROWMAX, B_ROWMAX_H, B_SEGCOUNT, B_OVERRIDE,
       B_STR_Q, B_STR_D, B_STR_S, B_STR_F, B_STR_OQ, B_STR_OD, B_STR_OS, B_STR_OSTR, B_STR_CNT,
       B_TOPK_Q, B_TOPK_D, B_TOPK_S, B_TOPK_BID, B_TOPK_BD, B_TOPK_CNT, B_TOPK_OFF, B_TOPK_OD, B_TOPK_OID, B_TOPK_OCNT, B_TOPK_OHITS,
       B_TK2_RQ, B_TK2_RD, B_TK2_RS, B_TK2_X, B_TK2_SSTR, B_TK2_BSTR, B_TK2_OSTR,
       B_CC_PARENT, B_CC_LABEL, B_GR_ROWS, B_GR_OUT,
       B_COUNT };

struct ProfRec {
	int kind;
	cudaEvent_t e0, e1;
};

struct Deferred {
	void *dst;
	const void *src;
	size_t bytes;
};

struct CtxExtra {
	Buf d[B_COUNT];
	// page-locked staging for the small copies of the one-query entry points (index lists in, flags / results out): a
	// copy from or to pageable memory costs ~10 us of driver staging each, the same copy through pinned memory ~2 us.
	// Bump-allocated; reset at the synchronisation that ends the call.
	char *stage = nullptr;
	size_t stage_cap = 0, stage_used = 0;
	std::vector<Deferred> deferred; // device -> pinned copies in flight, to be handed to the caller after the sync
	std::vector<ProfRec> pending;
	std::vector<cudaEvent_t> pool;
	double prof_ms[MC2_KERNEL_KINDS] = {0};
	u64 prof_n[MC2_KERNEL_KINDS] = {0};
	// the last all-pairs / identity sweep: pairs the tile sweep sent through the exact epilogue, 1 if it took the coarse form
	u64 last_exact = 0;
	int last_coarse = 0;
	u64 last_inline = 0; // of those, the pairs the coarse sweep refined inline because its candidate buffer was full
	u64 sum_inline = 0;  // last_inline summed over the sweeps of the current call
};

static cudaEvent_t prof_event(CtxExtra *x)
{
	cudaEvent_t e;
	if (!x->pool.empty()) {
		e = x->pool.back();
		x->pool.pop_back();
		return e;
	}
	cudaEventCreate(&e);
	return e;
}

void prof_begin(mc2_ctx *ctx, int kind)
{
	if (!ctx->prof_on) {
		return;
	}
	CtxExtra *x = reinterpret_cast<CtxExtra *>(ctx->extra);
	ProfRec r;
	r.kind = kind;
	r.e0 = prof_event(x);
	r.e1 = prof_event(x);
	cudaEventRecord(r.e0, ctx->stream);
	x->pending.push_back(r);
}

void prof_end(mc2_ctx *ctx)
{
	if (!ctx->prof_on) {
		return;
	}
	CtxExtra *x = reinterpret_cast<CtxExtra *>(ctx->extra);
	cudaEventRecord(x->pending.back().e1, ctx->stream);
}

static void prof_drain(mc2_ctx *ctx)
{
	CtxExtra *x = reinterpret_cast<CtxExtra *>(ctx->extra);
	for (ProfRec &r : x->pending) {
		float ms = 0;
		if (cudaEventSynchronize(r.e1) == cudaSuccess && cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) {
			x->prof_ms[r.kind] += ms;
			x->prof_n[r.kind]++;
		}
		x->pool.push_back(r.e0);
		x->pool.push_back(r.e1);
	}
	x->pending.clear();
}

static CtxExtra *extra_of(mc2_ctx *ctx)
{
	return reinterpret_cast<CtxExtra *>(ctx->extra);
}

// end-of-call synchronisation: waits for the stream, delivers the staged device->host results, recycles the staging area
static int sync_stage(mc2_ctx *ctx)
{
	CtxExtra *x = extra_of(ctx);
	cudaError_t e = cudaStreamSynchronize(ctx->stream);
	if (e == cudaSuccess) {
		for (const Deferred &c : x->deferred) {
			memcpy(c.dst, c.src, c.bytes);
		}
	}
	x->deferred.clear();
	x->stage_used = 0;
	MC2_CUDA(e);
	return MC2_OK;
}

// Entry points that stage copies end with sync_stage(); an early error return between a d2h() and that sync leaves entries
// behind whose destination may be gone by the next call.  Every public entry point that stages starts by dropping them.
static void drop_stale_stage(mc2_ctx *ctx)
{
	CtxExtra *x = extra_of(ctx);
	if (!x->deferred.empty() || x->stage_used) {
		cudaStreamSynchronize(ctx->stream);
		cudaGetLastError();
		x->deferred.clear();
		x->stage_used = 0;
	}
}

static const size_t kStageBytes = 4u << 20, kStageMaxCopy = 1u << 20;

static char *stage_take(mc2_ctx *ctx, size_t bytes)
{
	CtxExtra *x = extra_of(ctx);
	if (bytes > kStageMaxCopy) {
		return nullptr;
	}
	if (!x->stage) {
		if (cudaHostAlloc((void **)&x->stage, kStageBytes, cudaHostAllocDefault) != cudaSuccess) {
			cudaGetLastError();
			x->stage = nullptr;
			return nullptr;
		}
		x->stage_cap = kStageBytes;
	}
	const size_t need = (bytes + 63) & ~(size_t)63;
	if (x->stage_used + need > x->stage_cap) {
		if (sync_stage(ctx) != MC2_OK) { // everything staged so far has been consumed once the stream is idle
			return nullptr;
		}
	}
	char *p = x->stage + x->stage_used;
	x->stage_used += need;
	return p;
}

// host -> device on the context's stream; src may be released as soon as this returns when the copy was staged, so callers
// that pass temporaries must still synchronise if it reports "not staged"
static int h2d(mc2_ctx *ctx, void *dst, const void *src, size_t bytes, bool *staged = nullptr)
{
	char *p = stage_take(ctx, bytes);
	if (staged) *staged = p != nullptr;
	if (p) {
		memcpy(p, src, bytes);
		src = p;
	}
	MC2_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
	return MC2_OK;
}

// device -> host, delivered by the next sync_stage()
static int d2h(mc2_ctx *ctx, void *dst, const void *src, size_t bytes)
{
	char *p = stage_take(ctx, bytes);
	if (p) {
		MC2_CUDA(cudaMemcpyAsync(p, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
		extra_of(ctx)->deferred.push_back(Deferred{dst, p, bytes});
		return MC2_OK;
	}
	MC2_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
	return MC2_OK;
}

// Constants of the tile sweep's fp32 screen (tile_sweep.cu, screen_pairs).  Per single k present in the model the
// normalised value of Feature::normalize_cache (Feature.cpp:136-154) is x = a*raw + b with a = +-1/range, b folded from
// min, range and the 1 - v of distance-like singles.  Error model, eps = 2^-23 (twice the unit round-off):
//   raw is a cancellation-free fp32 expression of exact integers, relative error <= 16 eps;
//   |fl(x) - x| <= eps * 18 * (|x| + 2|b|) <= eps * gamma * u,  gamma = 18 * max(1, 2 max|b|),  u = 1 + max_k |x_k|;
//   a combo of total degree P <= 4 in factors bounded by u with that error: |delta| <= u^4 * eps * (1.01 P gamma + P);
//   weights in fp32 and the fused accumulation add eps * (2 + n_combos + 1) per term.
// Hence |fp32 sum - exact sum| <= eps * (K1 * u^4 + K0); both constants are doubled before rounding to float.
// The coarse form of the sweep knows the EMD only as an interval [e1, e2] of exact integers and bounds the sum from
// above: each combo with the EMD factor takes the larger of its values at x(e1), x(e2) (and 0 for a squared factor whose
// interval spans 0).  Both ends are the same cancellation-free expressions as the exact EMD's, so the per-term bound holds
// at each end with u = 1 + max |x| over both; the max of two fused sums fma(w, f_i, s) is the rounding of
// max(w f_i) + s (rounding is monotone), so the accumulation's term is unchanged; the ends' fp32 values are each within
// eps * gamma * u of the exact ones, so the spans-0 test on the interval widened by scr_dx * u = eps * gamma * u never
// misses a sign change.  The bound, hence K1 and K0, is the same: |fp32 sum - exact upper bound| <= eps * (K1 u^4 + K0).
// The threshold on the sum, rounded down past that margin: a pair whose fp32 sum + bound stays below it has exact sum < t.
static float screen_threshold(double t)
{
	return nextafterf((float)(t - 1e-6 - fabs(t) * 1e-6), -INFINITY);
}

// The constants depend on the model alone.  A classifier's threshold is fixed by its bias; a regression model's is the
// identity a search asks for, set per call (mc2_identity_pairs).
static void build_screen(DevModel &dm)
{
	dm.scr_ok = 0;
	dm.scr_k1 = dm.scr_k0 = dm.scr_dx = 0;
	dm.scr_thr = 0;
	memset(dm.scr_a, 0, sizeof dm.scr_a);
	memset(dm.scr_b, 0, sizeof dm.scr_b);
	memset(dm.scr_w, 0, sizeof dm.scr_w);
	if (!dm.fast_epi || dm.n_combos > MC2_SCR_MAX_COMBOS || (dm.need & NEED_LOG)) {
		return;
	}
	if (!dm.regression) {
		// close <=> round(logistic(sum) + bias) > 0 <=> logistic(sum) >= 0.5 - bias (Predictor.cpp:323-333): a threshold on
		// the sum while 0.5 - bias lies strictly inside (0, 1); outside it every pair (or none) is close and nothing can be
		// screened
		if (!(dm.bias > -0.499999 && dm.bias < 0.499999)) {
			return;
		}
		const double pth = 0.5 - dm.bias, t = log(pth / (1.0 - pth));
		dm.scr_thr = screen_threshold(t);
	}
	const double eps = 1.1920928955078125e-07;
	double beta = 0;
	for (int k = 0; k < SC_COUNT; k++) {
		if (dm.slot[k] < 0) {
			continue;
		}
		if (!dm.crcp_ok[k] || !std::isfinite(dm.cmin[k])) {
			return;
		}
		const double rcp = dm.crcp[k];
		const double a = dm.csim[k] ? rcp : -rcp;
		const double b = dm.csim[k] ? -dm.cmin[k] * rcp : 1.0 + dm.cmin[k] * rcp;
		if (!(fabs(a) < 1e30 && fabs(b) < 1e6)) {
			return;
		}
		dm.scr_a[k] = (float)a;
		dm.scr_b[k] = (float)b;
		beta = std::max(beta, fabs(b));
	}
	const double gamma = 18.0 * std::max(1.0, 2.0 * beta);
	if (!(eps * gamma * 4 < 0.01)) {
		return;
	}
	double K1 = 0;
	for (int c = 0; c < MC2_SCR_MAX_COMBOS; c++) {
		dm.scr_ka[c] = dm.scr_kb[c] = scr_slot(dm.need & 7, SC_COUNT); // the constant 1
		dm.scr_pa2[c] = dm.scr_pb2[c] = 0;
	}
	for (int c = 0; c < dm.n_combos; c++) {
		int pw[SC_COUNT] = {0};
		int P = 0;
		for (int t = 0; t < dm.nidx[c]; t++) {
			const int code = dm.code[dm.idx[c][t]];
			const int kind = dm.kind[c];
			const int add = (kind == MC2_COMBO_X2Y2 || (kind == MC2_COMBO_XY2 && t == 1) || (kind == MC2_COMBO_X2Y && t == 0)) ? 2 : 1;
			pw[code] += add;
			P += add;
		}
		int nk = 0;
		for (int k = 0; k < SC_COUNT; k++) {
			if (pw[k] == 0) {
				continue;
			}
			if (pw[k] > 2 || nk == 2) {
				return; // more than two distinct singles, or one of them beyond its square: outside the screen's form
			}
			(nk == 0 ? dm.scr_ka[c] : dm.scr_kb[c]) = scr_slot(dm.need & 7, k);
			(nk == 0 ? dm.scr_pa2[c] : dm.scr_pb2[c]) = pw[k] == 2;
			nk++;
		}
		const double w = dm.weight[c + 1];
		if (!(fabs(w) < 1e6)) {
			return;
		}
		dm.scr_w[c + 1] = (float)w;
		K1 += fabs(w) * (1.01 * P * gamma + P + 2 + dm.n_combos + 1);
	}
	if (!(fabs(dm.weight[0]) < 1e6)) {
		return;
	}
	dm.scr_w[0] = (float)dm.weight[0];
	const double K0 = (dm.n_combos + 2) * fabs(dm.weight[0]);
	dm.scr_k1 = nextafterf((float)(2 * eps * K1), INFINITY);
	dm.scr_k0 = nextafterf((float)(2 * eps * K0), INFINITY);
	dm.scr_dx = nextafterf((float)(2 * eps * gamma), INFINITY);
	dm.scr_ok = 1;
}

static int model_need(const mc2_model_desc &d, DevModel &dm)
{
	memset(&dm, 0, sizeof dm);
	if (d.n_singles < 1 || d.n_singles > MC2_MAX_SINGLES || d.n_combos < 1 || d.n_combos > MC2_MAX_COMBOS) {
		set_error("model: n_singles / n_combos out of range");
		return MC2_ERR_ARG;
	}
	dm.n_singles = d.n_singles;
	dm.n_combos = d.n_combos;
	int need = 0;
	for (int i = 0; i < d.n_singles; i++) {
		int code, sim;
		switch (d.single_flag[i]) {
		case MC2_FEAT_MANHATTAN: code = SC_MANHATTAN; sim = 0; need |= NEED_MIN; break;
		case MC2_FEAT_EUCLIDEAN: code = SC_EUCLIDEAN; sim = 0; need |= NEED_DOT; break;
		case MC2_FEAT_NORMALIZED_VECTORS: code = SC_NORMALIZED_VECTORS; sim = 1; need |= NEED_DOT; break;
		case MC2_FEAT_JEFFEREY_DIV: code = SC_JEFFEREY; sim = 0; need |= NEED_LOG; break;
		case MC2_FEAT_PEARSON_COEFF: code = SC_PEARSON; sim = 1; need |= NEED_DOT; break;
		case MC2_FEAT_INTERSECTION: code = SC_INTERSECTION; sim = 1; need |= NEED_MIN; break;
		case MC2_FEAT_EMD: code = SC_EMD; sim = 0; need |= NEED_EMD; break;
		case MC2_FEAT_LENGTHD: code = SC_LENGTHD; sim = 0; break;
		case MC2_FEAT_KULCZYNSKI2: code = SC_KULCZYNSKI2; sim = 1; need |= NEED_MIN; break;
		case MC2_FEAT_SIMRATIO: code = SC_SIMRATIO; sim = 1; need |= NEED_DOT; break;
		case MC2_FEAT_JENSEN_SHANNON: code = SC_JENSEN_SHANNON; sim = 0; need |= NEED_LOG; break;
		default: {
			char buf[160];
			snprintf(buf, sizeof buf,
				 "model: single feature flag %llu is outside the hot-path scope (fast + slow sets only)",
				 (unsigned long long)d.single_flag[i]);
			set_error(buf);
			return MC2_ERR_UNSUPPORTED;
		}
		}
		dm.code[i] = code;
		dm.is_sim[i] = sim; // Feature::feat_is_sim, src/predict/Feature.cpp:549-663
		dm.smin[i] = d.single_min[i];
		dm.smax[i] = d.single_max[i];
	}
	for (int c = 0; c < d.n_combos; c++) {
		int kind = d.combo_kind[c], n = d.combo_nidx[c];
		if (kind < 0 || kind > 3 || n < 1 || n > MC2_MAX_COMBO_IDX) {
			set_error("model: bad combo kind / index count");
			return MC2_ERR_ARG;
		}
		if ((kind == MC2_COMBO_XY2 || kind == MC2_COMBO_X2Y) && n != 2) {
			// Feature::operator() throws "invalid" (Feature.h:221-235)
			set_error("model: xy2 / x2y combos need exactly two singles");
			return MC2_ERR_ARG;
		}
		dm.kind[c] = kind;
		dm.nidx[c] = n;
		for (int t = 0; t < n; t++) {
			int ix = d.combo_idx[c][t];
			if (ix < 0 || ix >= d.n_singles) {
				set_error("model: combo index out of range");
				return MC2_ERR_ARG;
			}
			dm.idx[c][t] = ix;
		}
	}
	for (int c = 0; c <= d.n_combos; c++) {
		dm.weight[c] = d.weight[c];
	}
	dm.bias = d.bias;
	dm.regression = d.regression;
	dm.need = need;
	dm.fast_epi = 1;
	for (int c = 0; c < SC_COUNT; c++) {
		dm.slot[c] = -1;
	}
	for (int i = 0; i < d.n_singles; i++) {
		const int c = dm.code[i];
		if (dm.slot[c] >= 0) {
			dm.fast_epi = 0; // the same single twice (never produced by the reference's selector)
			continue;
		}
		dm.slot[c] = i;
		dm.csim[c] = dm.is_sim[i];
		dm.cmin[c] = dm.smin[i];
		dm.crange[c] = dm.smax[i] - dm.smin[i];
		dm.crcp[c] = 1.0 / dm.crange[c];
		const double ar = fabs(dm.crange[c]);
		dm.crcp_ok[c] = std::isfinite(dm.crcp[c]) && ar > 1e-100 && ar < 1e100;
	}
	build_screen(dm);
	return MC2_OK;
}

static CtxExtra *extra(mc2_ctx *ctx)
{
	return reinterpret_cast<CtxExtra *>(ctx->extra);
}

static int check_err(mc2_ctx *ctx)
{
	int e = *ctx->h_err;
	if (e == 0) {
		ctx->err_dirty = 0; // the device word is known to be zero: the next call need not clear it
		return MC2_OK;
	}
	if (e & 16) {
		set_error("tile sweep: a pipeline barrier timed out (internal error)");
		return MC2_ERR_CUDA;
	}
	if (e & 4) {
		set_error("invalid nucleotide code inside a segment (reference: InvalidInputException, KmerHashTable.cpp:138-149)");
		return MC2_ERR_INPUT;
	}
	if (e & 1) {
		set_error("a single feature failed the way the reference throws (zero length in length_difference or NaN after normalisation)");
		return MC2_ERR_FEATURE;
	}
	set_error("internal: unknown single-feature code on device");
	return MC2_ERR_FEATURE;
}

static int reset_err(mc2_ctx *ctx)
{
	if (ctx->err_dirty) {
		MC2_CUDA(cudaMemsetAsync(ctx->d_err, 0, sizeof(int), ctx->stream));
	}
	ctx->err_dirty = 1; // until a check_err() has seen it clean
	return MC2_OK;
}

static int fetch_err(mc2_ctx *ctx)
{
	MC2_CUDA(cudaMemcpyAsync(ctx->h_err, ctx->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
	return MC2_OK;
}

static int alloc_hset(mc2_ctx *ctx, u64 n, int k, int eb, mc2_hset **out)
{
	mc2_hset *h = new (std::nothrow) mc2_hset();
	if (!h) {
		set_error("out of host memory");
		return MC2_ERR_ARG;
	}
	memset(h, 0, sizeof *h);
	h->ctx = ctx;
	h->n = n;
	h->k = k;
	h->N = 1ULL << (2 * k);
	h->eb = eb;
	u64 nn = n ? n : 1;
	cudaError_t e;
#define A(ptr, bytes)                                                \
	e = cudaMalloc((void **)&(ptr), (bytes));                    \
	if (e != cudaSuccess) {                                      \
		mc2_hset_free(h);                                    \
		return cuda_fail(e, "cudaMalloc", __FILE__, __LINE__); \
	}
	A(h->bins, nn * h->N * (u64)eb);
	A(h->mag, nn * 8);
	A(h->sum, nn * 8);
	A(h->sumsq, nn * 8);
	A(h->len, nn * 8);
	A(h->mers1, nn * 32);
	A(h->stddev, nn * 8);
	A(h->novf, nn * 4);
	A(h->maxc, nn * 4);
#undef A
	*out = h;
	return MC2_OK;
}

// the derived reverse-complement set carries bins, magnitudes and lengths: every write to one of them drops it
static void drop_rc(mc2_hset *h)
{
	if (h->rc) {
		mc2_hset_free(h->rc);
		h->rc = nullptr;
	}
}

// max over rows of the bin sums and of the raw k-mer multiplicities: out[0], out[1] (zeroed by the caller)
__global__ void __launch_bounds__(256) row_max_kernel(const u64 *sum, const u32 *maxc, u64 n, unsigned long long *out)
{
	u64 ms = 0;
	u32 mc = 0;
	for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
		ms = sum[i] > ms ? sum[i] : ms;
		mc = maxc[i] > mc ? maxc[i] : mc;
	}
	for (int o = 16; o; o >>= 1) {
		u64 t = __shfl_xor_sync(0xffffffffu, ms, o);
		ms = t > ms ? t : ms;
	}
	mc = __reduce_max_sync(0xffffffffu, mc);
	if ((threadIdx.x & 31) == 0) {
		atomicMax(out, (unsigned long long)ms);
		atomicMax(out + 1, (unsigned long long)mc);
	}
}

static int refresh_max_sum(mc2_ctx *ctx, mc2_hset *h)
{
	// host-side bounds used to pick the 32-bit fast paths and the histogram width: one 16-byte D2H per set (re)fill
	h->max_sum = 0;
	h->max_count = 0;
	if (h->n == 0) {
		return MC2_OK;
	}
	CtxExtra *x = reinterpret_cast<CtxExtra *>(ctx->extra);
	int rc = ensure(x->d[B_ROWMAX], 16, false);
	if (rc != MC2_OK) return rc;
	rc = ensure(x->d[B_ROWMAX_H], 16, true);
	if (rc != MC2_OK) return rc;
	unsigned long long *dv = (unsigned long long *)x->d[B_ROWMAX].p, *hv = (unsigned long long *)x->d[B_ROWMAX_H].p;
	MC2_CUDA(cudaMemsetAsync(dv, 0, 16, ctx->stream));
	u64 want = (h->n + 255) / 256, cap = (u64)ctx->sm_count * 4;
	row_max_kernel<<<(int)(want < cap ? want : cap), 256, 0, ctx->stream>>>(h->sum, h->maxc, h->n, dv);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	MC2_CUDA(cudaMemcpyAsync(hv, dv, 16, cudaMemcpyDeviceToHost, ctx->stream));
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	h->max_sum = hv[0];
	h->max_count = hv[1];
	return MC2_OK;
}

// one warp per row: copy bins + true sums; length / magnitude from the optional override arrays
__global__ void __launch_bounds__(256) assign_rows_kernel(char *dbins, u64 *dmag, u64 *dsum, u64 *dsumsq, u64 *dlen, const char *sbins,
							   const u64 *ssum, const u64 *ssumsq, const u64 *slen, u64 row_bytes, u64 n,
							   const u64 *idx /* [dst | src | mag? | len?] x n */, int has_mag, int has_len,
							   unsigned short *dloff, const unsigned short *sloff)
{
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	for (u64 i = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps_total) {
		const u64 d = idx[i], s = idx[n + i];
		const uint32_t *src = reinterpret_cast<const uint32_t *>(sbins + s * row_bytes);
		uint32_t *dst = reinterpret_cast<uint32_t *>(dbins + d * row_bytes);
		for (u64 w = lane; w < row_bytes / 4; w += 32) {
			dst[w] = src[w];
		}
		if (dloff) { // lane offsets depend on the bins only: they travel with the row
			dloff[d * 32 + lane] = sloff[s * 32 + lane];
		}
		if (lane == 0) {
			dsum[d] = ssum[s];
			dsumsq[d] = ssumsq[s];
			dlen[d] = has_len ? idx[(2 + has_mag) * n + i] : slen[s];
			if (has_mag) {
				dmag[d] = idx[2 * n + i];
			}
		}
	}
}

} // namespace mc2

using namespace mc2;

extern "C" {

int mc2_abi_version(void)
{
	return MC2_ABI_VERSION;
}

const char *mc2_last_error(void)
{
	return g_err.c_str();
}

int mc2_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	return n;
}

int mc2_ctx_create(int device, mc2_ctx **out)
{
	MC2_REQUIRE(out != nullptr, "mc2_ctx_create: out is NULL");
	*out = nullptr;
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess || n == 0) {
		cudaGetLastError();
		set_error("no CUDA device available: libmeshclust2_b200 has no CPU fallback");
		return MC2_ERR_CUDA;
	}
	MC2_REQUIRE(device >= 0 && device < n, "mc2_ctx_create: device index out of range");
	cudaDeviceProp prop;
	MC2_CUDA(cudaGetDeviceProperties(&prop, device));
	if (prop.major != 10) {
		char buf[200];
		snprintf(buf, sizeof buf, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major,
			 prop.minor);
		set_error(buf);
		return MC2_ERR_CUDA;
	}
	MC2_CUDA(cudaSetDevice(device));
	mc2_ctx *c = new (std::nothrow) mc2_ctx();
	MC2_REQUIRE(c != nullptr, "out of host memory");
	memset(c, 0, sizeof *c);
	c->device = device;
	c->sm_count = prop.multiProcessorCount;
	MC2_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	MC2_CUDA(cudaEventCreate(&c->ev0));
	MC2_CUDA(cudaEventCreate(&c->ev1));
	// result slot: [0,64) reduction result, [64,128) the sticky error word, [128,4096) close flags of small batches, so that
	// one device->host copy ends a one-query call
	MC2_CUDA(cudaMallocHost(&c->h_slot, 4096));
	MC2_CUDA(cudaMalloc(&c->d_slot, 4096));
	MC2_CUDA(cudaMemset(c->d_slot, 0, 4096));
	memset(c->h_slot, 0, 4096);
	c->d_err = reinterpret_cast<int *>(reinterpret_cast<char *>(c->d_slot) + 64);
	c->h_err = reinterpret_cast<int *>(reinterpret_cast<char *>(c->h_slot) + 64);
	c->err_dirty = 1;
	CtxExtra *x = new (std::nothrow) CtxExtra();
	c->extra = x;
	*out = c;
	return MC2_OK;
}

void mc2_ctx_destroy(mc2_ctx *ctx)
{
	if (!ctx) {
		return;
	}
	cudaSetDevice(ctx->device);
	if (ctx->mb) {
		ctx->mb->w[7] = 1;
		cudaStreamSynchronize(ctx->server_stream);
		cudaStreamDestroy(ctx->server_stream);
		cudaFreeHost(ctx->mb);
		ctx->mb = nullptr;
	}
	cudaStreamSynchronize(ctx->stream);
	CtxExtra *x = extra(ctx);
	if (x) {
		prof_drain(ctx);
		for (auto e : x->pool) {
			cudaEventDestroy(e);
		}
		for (auto &b : x->d) {
			release(b);
		}
		if (x->stage) {
			cudaFreeHost(x->stage);
		}
		delete x;
	}
	if (ctx->flush_buf) {
		cudaFree(ctx->flush_buf);
	}
	cudaFreeHost(ctx->h_slot);
	cudaFree(ctx->d_slot);
	cudaFree(ctx->d_sched);
	cudaFree(ctx->d_cand);
	cudaEventDestroy(ctx->ev0);
	cudaEventDestroy(ctx->ev1);
	cudaStreamDestroy(ctx->stream);
	delete ctx;
}

int mc2_ctx_sync(mc2_ctx *ctx)
{
	MC2_REQUIRE(ctx != nullptr, "ctx is NULL");
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC2_OK;
}

int mc2_ctx_device(const mc2_ctx *ctx)
{
	return ctx ? ctx->device : -1;
}

int mc2_ctx_sm_count(const mc2_ctx *ctx)
{
	return ctx ? ctx->sm_count : 0;
}

void *mc2_ctx_stream(mc2_ctx *ctx)
{
	return ctx ? (void *)ctx->stream : nullptr;
}

int mc2_timer_start(mc2_ctx *ctx)
{
	MC2_REQUIRE(ctx != nullptr, "ctx is NULL");
	MC2_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
	return MC2_OK;
}

int mc2_timer_stop(mc2_ctx *ctx, float *ms)
{
	MC2_REQUIRE(ctx != nullptr && ms != nullptr, "ctx / ms is NULL");
	MC2_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
	MC2_CUDA(cudaEventSynchronize(ctx->ev1));
	MC2_CUDA(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
	return MC2_OK;
}

uint64_t mc2_ctx_launch_count(const mc2_ctx *ctx)
{
	return ctx ? ctx->launches : 0;
}

int mc2_ctx_profile(mc2_ctx *ctx, int enable)
{
	MC2_REQUIRE(ctx != nullptr, "ctx is NULL");
	CtxExtra *x = extra(ctx);
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	prof_drain(ctx);
	if (enable) {
		for (int i = 0; i < MC2_KERNEL_KINDS; i++) {
			x->prof_ms[i] = 0;
			x->prof_n[i] = 0;
		}
	}
	ctx->prof_on = enable ? 1 : 0;
	return MC2_OK;
}

int mc2_ctx_kernel_time(mc2_ctx *ctx, int kind, double *total_ms, uint64_t *launches)
{
	MC2_REQUIRE(ctx && total_ms && launches, "mc2_ctx_kernel_time: NULL argument");
	MC2_REQUIRE(kind >= 0 && kind < MC2_KERNEL_KINDS, "mc2_ctx_kernel_time: kind out of range");
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	prof_drain(ctx);
	CtxExtra *x = extra(ctx);
	*total_ms = x->prof_ms[kind];
	*launches = x->prof_n[kind];
	return MC2_OK;
}

int mc2_ctx_flush_l2(mc2_ctx *ctx, size_t bytes)
{
	MC2_REQUIRE(ctx != nullptr, "ctx is NULL");
	if (bytes > ctx->flush_bytes) {
		if (ctx->flush_buf) {
			cudaFree(ctx->flush_buf);
			ctx->flush_buf = nullptr;
			ctx->flush_bytes = 0;
		}
		MC2_CUDA(cudaMalloc(&ctx->flush_buf, bytes));
		ctx->flush_bytes = bytes;
	}
	MC2_CUDA(cudaMemsetAsync(ctx->flush_buf, 0, bytes, ctx->stream));
	return MC2_OK;
}

/* ---- sequences -------------------------------------------------------------------------------- */
// grow-only device array of a sequence set: reallocates only when the capacity is too small, so a set that is refilled
// with batches of similar size (mc2_seqs_upload_into) never touches cudaMalloc / cudaFree (both stall the device)
extern "C++" {
template <typename P>
static int seq_reserve(P *&p, u64 &cap_bytes, u64 bytes)
{
	if (p != nullptr && cap_bytes >= bytes) {
		return MC2_OK;
	}
	if (p) {
		cudaFree(p);
		p = nullptr;
		cap_bytes = 0;
	}
	u64 want = bytes + bytes / 8 + 256;
	MC2_CUDA(cudaMalloc((void **)&p, want));
	cap_bytes = want;
	return MC2_OK;
}
} // extern "C++"

static int seqs_fill(mc2_ctx *ctx, mc2_seqs *s, const char *codes, const uint64_t *seq_off, uint64_t n, const int32_t *segs,
		     const uint64_t *seg_off)
{
	const u64 total_bases = seq_off[n] - seq_off[0];
	const u64 total_segs = seg_off[n] - seg_off[0];
	MC2_REQUIRE(total_segs == 0 || segs != nullptr, "mc2_seqs_upload: segs is NULL");
	// host-side shape checks only (no per-base work on the host)
	std::vector<u64> word_off(n + 1), len(n), soff(n + 1), boff(n + 1);
	u64 w = 0, max_len = 0, min_seg = ~0ULL;
	for (u64 i = 0; i < n; i++) {
		MC2_REQUIRE(seq_off[i + 1] >= seq_off[i] && seg_off[i + 1] >= seg_off[i], "mc2_seqs_upload: offsets must be non-decreasing");
		u64 L = seq_off[i + 1] - seq_off[i];
		MC2_REQUIRE(L < (1ULL << 31), "mc2_seqs_upload: a sequence is longer than 2^31-1 bases (reference positions are int)");
		len[i] = L;
		max_len = L > max_len ? L : max_len;
		word_off[i] = w;
		boff[i] = seq_off[i] - seq_off[0];
		soff[i] = seg_off[i] - seg_off[0];
		u64 nw = (L + 15) / 16 + 1; // one spare word so the k-mer window may read past the end
		w += (nw + 3) & ~3ULL;
		for (u64 sg = seg_off[i]; sg < seg_off[i + 1]; sg++) {
			long long s0 = segs[2 * sg], e0 = segs[2 * sg + 1];
			MC2_REQUIRE(s0 >= 0 && e0 >= s0 && (u64)e0 < L, "mc2_seqs_upload: segment outside its sequence");
			MC2_REQUIRE(sg == seg_off[i] || s0 > segs[2 * sg - 1], "mc2_seqs_upload: segments must be sorted and disjoint");
			min_seg = (u64)(e0 - s0 + 1) < min_seg ? (u64)(e0 - s0 + 1) : min_seg;
		}
	}
	word_off[n] = w;
	boff[n] = total_bases;
	soff[n] = total_segs;
	s->n = n;
	s->total_bases = total_bases;
	s->max_len = max_len;
	s->total_segs = total_segs;
	s->total_words = w;
	s->min_seg_len = min_seg;
	CtxExtra *x = reinterpret_cast<CtxExtra *>(ctx->extra);
	int rc;
	if ((rc = seq_reserve(s->packed, s->cap_packed, (w ? w : 1) * 4)) != MC2_OK) return rc;
	if ((rc = seq_reserve(s->word_off, s->cap_word_off, (n + 1) * 8)) != MC2_OK) return rc;
	if ((rc = seq_reserve(s->len, s->cap_len, (n ? n : 1) * 8)) != MC2_OK) return rc;
	if ((rc = seq_reserve(s->segs, s->cap_segs, (total_segs ? total_segs : 1) * 8)) != MC2_OK) return rc;
	if ((rc = seq_reserve(s->seg_off, s->cap_seg_off, (n + 1) * 8)) != MC2_OK) return rc;
	// staging for the byte-per-base codes: owned by the context, reused by every upload
	if ((rc = ensure(x->d[B_STAGE_CODES], total_bases ? total_bases : 1, false)) != MC2_OK) return rc;
	if ((rc = ensure(x->d[B_STAGE_BOFF], (n + 1) * 8, false)) != MC2_OK) return rc;
	char *d_codes = (char *)x->d[B_STAGE_CODES].p;
	u64 *d_boff = (u64 *)x->d[B_STAGE_BOFF].p;
	cudaStream_t st = ctx->stream;
	MC2_CUDA(cudaMemcpyAsync(s->word_off, word_off.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
	if (n) MC2_CUDA(cudaMemcpyAsync(s->len, len.data(), n * 8, cudaMemcpyHostToDevice, st));
	if (total_segs) MC2_CUDA(cudaMemcpyAsync(s->segs, segs + 2 * seg_off[0], total_segs * 8, cudaMemcpyHostToDevice, st));
	MC2_CUDA(cudaMemcpyAsync(s->seg_off, soff.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
	if (total_bases) MC2_CUDA(cudaMemcpyAsync(d_codes, codes + seq_off[0], total_bases, cudaMemcpyHostToDevice, st));
	MC2_CUDA(cudaMemcpyAsync(d_boff, boff.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
	rc = reset_err(ctx);
	if (rc == MC2_OK) rc = launch_pack(ctx, d_codes, d_boff, s);
	if (rc == MC2_OK) rc = fetch_err(ctx);
	cudaError_t e = cudaStreamSynchronize(st); // the host vectors above go out of scope; the error word is read below
	if (rc == MC2_OK && e != cudaSuccess) rc = cuda_fail(e, "pack", __FILE__, __LINE__);
	if (rc == MC2_OK) rc = check_err(ctx);
	return rc;
}

int mc2_seqs_upload(mc2_ctx *ctx, const char *codes, const uint64_t *seq_off, uint64_t n, const int32_t *segs,
		    const uint64_t *seg_off, mc2_seqs **out)
{
	MC2_REQUIRE(ctx && seq_off && seg_off && out, "mc2_seqs_upload: NULL argument");
	MC2_REQUIRE(n == 0 || codes != nullptr, "mc2_seqs_upload: codes is NULL");
	*out = nullptr;
	MC2_CUDA(cudaSetDevice(ctx->device));
	mc2_seqs *s = new (std::nothrow) mc2_seqs();
	MC2_REQUIRE(s != nullptr, "out of host memory");
	memset(s, 0, sizeof *s);
	s->ctx = ctx;
	int rc = seqs_fill(ctx, s, codes, seq_off, n, segs, seg_off);
	if (rc != MC2_OK) {
		mc2_seqs_free(s);
		return rc;
	}
	*out = s;
	return MC2_OK;
}

int mc2_seqs_upload_into(mc2_ctx *ctx, mc2_seqs *dst, const char *codes, const uint64_t *seq_off, uint64_t n,
			 const int32_t *segs, const uint64_t *seg_off)
{
	MC2_REQUIRE(ctx && dst && seq_off && seg_off, "mc2_seqs_upload_into: NULL argument");
	MC2_REQUIRE(n == 0 || codes != nullptr, "mc2_seqs_upload_into: codes is NULL");
	MC2_REQUIRE(dst->ctx == ctx, "mc2_seqs_upload_into: the set belongs to another context");
	MC2_CUDA(cudaSetDevice(ctx->device));
	int rc = seqs_fill(ctx, dst, codes, seq_off, n, segs, seg_off);
	if (rc != MC2_OK) {
		dst->n = 0; // contents undefined after a failed refill: leave an empty, still freeable set
		dst->total_bases = dst->total_segs = dst->total_words = dst->max_len = 0;
	}
	return rc;
}

static int text_fill(mc2_ctx *ctx, mc2_seqs *s, const char *text, const uint64_t *seq_off, uint64_t n)
{
	const u64 total_bases = seq_off[n] - seq_off[0];
	std::vector<u64> word_off(n + 1), len(n), boff(n + 1);
	u64 w = 0, max_len = 0;
	for (u64 i = 0; i < n; i++) {
		MC2_REQUIRE(seq_off[i + 1] >= seq_off[i], "mc2_seqs_from_text: offsets must be non-decreasing");
		const u64 L = seq_off[i + 1] - seq_off[i];
		MC2_REQUIRE(L < (1ULL << 31), "mc2_seqs_from_text: a sequence is longer than 2^31-1 bases (reference positions are int)");
		len[i] = L;
		max_len = L > max_len ? L : max_len;
		word_off[i] = w;
		boff[i] = seq_off[i] - seq_off[0];
		const u64 nw = (L + 15) / 16 + 1;
		w += (nw + 3) & ~3ULL;
	}
	word_off[n] = w;
	boff[n] = total_bases;
	s->n = n;
	s->total_bases = total_bases;
	s->max_len = max_len;
	s->total_words = w;
	s->min_seg_len = ~0ULL;
	CtxExtra *x = extra(ctx);
	cudaStream_t st = ctx->stream;
	int rc = MC2_OK;
	auto fail = [&](int code) { // contents undefined after a failed fill: leave an empty, still freeable set
		s->n = 0;
		s->total_bases = s->total_segs = s->total_words = s->max_len = 0;
		return code;
	};
	if ((rc = seq_reserve(s->packed, s->cap_packed, (w ? w : 1) * 4)) != MC2_OK) return fail(rc);
	if ((rc = seq_reserve(s->word_off, s->cap_word_off, (n + 1) * 8)) != MC2_OK) return fail(rc);
	if ((rc = seq_reserve(s->len, s->cap_len, (n ? n : 1) * 8)) != MC2_OK) return fail(rc);
	if ((rc = seq_reserve(s->seg_off, s->cap_seg_off, (n + 1) * 8)) != MC2_OK) return fail(rc);
	if ((rc = ensure(x->d[B_STAGE_CODES], total_bases ? total_bases : 1, false)) != MC2_OK) return fail(rc);
	if ((rc = ensure(x->d[B_STAGE_BOFF], (n + 1) * 8, false)) != MC2_OK) return fail(rc);
	if ((rc = ensure(x->d[B_SEGCOUNT], (n ? n : 1) * 4, false)) != MC2_OK) return fail(rc);
	if ((rc = ensure(x->d[B_ROWMAX], 16, false)) != MC2_OK) return fail(rc);
	if ((rc = ensure(x->d[B_ROWMAX_H], 16, true)) != MC2_OK) return fail(rc);
	char *d_text = (char *)x->d[B_STAGE_CODES].p;
	u64 *d_boff = (u64 *)x->d[B_STAGE_BOFF].p;
	u32 *d_count = (u32 *)x->d[B_SEGCOUNT].p;
	unsigned long long *d_word = (unsigned long long *)x->d[B_ROWMAX].p, *h_word = (unsigned long long *)x->d[B_ROWMAX_H].p;
	cudaError_t e = cudaSuccess;
#define MC2_TRY(call)                                                  \
	if ((e = (call)) != cudaSuccess) {                             \
		return fail(cuda_fail(e, #call, __FILE__, __LINE__)); \
	}
	MC2_TRY(cudaMemcpyAsync(s->word_off, word_off.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
	if (n) MC2_TRY(cudaMemcpyAsync(s->len, len.data(), n * 8, cudaMemcpyHostToDevice, st));
	if (total_bases) MC2_TRY(cudaMemcpyAsync(d_text, text + seq_off[0], total_bases, cudaMemcpyHostToDevice, st));
	MC2_TRY(cudaMemcpyAsync(d_boff, boff.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st));
	// pass 1: segments per sequence -> exclusive scan -> total
	if ((rc = launch_segment(ctx, false, d_text, d_boff, n, d_count, nullptr, nullptr, nullptr)) != MC2_OK) return fail(rc);
	if ((rc = launch_seg_scan(ctx, d_count, n, s->seg_off)) != MC2_OK) return fail(rc);
	MC2_TRY(cudaMemcpyAsync(h_word, s->seg_off + n, 8, cudaMemcpyDeviceToHost, st));
	MC2_TRY(cudaStreamSynchronize(st));
	s->total_segs = h_word[0];
	if ((rc = seq_reserve(s->segs, s->cap_segs, (s->total_segs ? s->total_segs : 1) * 8)) != MC2_OK) return fail(rc);
	// pass 2: write the segments, then letters -> 2-bit words
	MC2_TRY(cudaMemsetAsync(d_word, 0xff, 8, st));
	if ((rc = launch_segment(ctx, true, d_text, d_boff, n, d_count, s->seg_off, s->segs, d_word)) != MC2_OK) return fail(rc);
	if ((rc = reset_err(ctx)) != MC2_OK) return fail(rc);
	if ((rc = launch_pack_text(ctx, d_text, d_boff, s)) != MC2_OK) return fail(rc);
	if ((rc = fetch_err(ctx)) != MC2_OK) return fail(rc);
	MC2_TRY(cudaMemcpyAsync(h_word, d_word, 8, cudaMemcpyDeviceToHost, st));
	MC2_TRY(cudaStreamSynchronize(st));
#undef MC2_TRY
	s->min_seg_len = h_word[0];
	if ((rc = check_err(ctx)) != MC2_OK) return fail(rc);
	return MC2_OK;
}

int mc2_seqs_from_text(mc2_ctx *ctx, const char *text, const uint64_t *seq_off, uint64_t n, mc2_seqs **out)
{
	MC2_REQUIRE(ctx && seq_off && out, "mc2_seqs_from_text: NULL argument");
	MC2_REQUIRE(n == 0 || text != nullptr, "mc2_seqs_from_text: text is NULL");
	*out = nullptr;
	MC2_CUDA(cudaSetDevice(ctx->device));
	mc2_seqs *s = new (std::nothrow) mc2_seqs();
	MC2_REQUIRE(s != nullptr, "out of host memory");
	memset(s, 0, sizeof *s);
	s->ctx = ctx;
	int rc = text_fill(ctx, s, text, seq_off, n);
	if (rc != MC2_OK) {
		mc2_seqs_free(s);
		return rc;
	}
	*out = s;
	return MC2_OK;
}

int mc2_seqs_from_text_into(mc2_ctx *ctx, mc2_seqs *dst, const char *text, const uint64_t *seq_off, uint64_t n)
{
	MC2_REQUIRE(ctx && dst && seq_off, "mc2_seqs_from_text_into: NULL argument");
	MC2_REQUIRE(n == 0 || text != nullptr, "mc2_seqs_from_text_into: text is NULL");
	MC2_REQUIRE(dst->ctx == ctx, "mc2_seqs_from_text_into: the set belongs to another context");
	MC2_CUDA(cudaSetDevice(ctx->device));
	return text_fill(ctx, dst, text, seq_off, n);
}

int mc2_seqs_download_segments(mc2_ctx *ctx, const mc2_seqs *s, int32_t *segs_out, uint64_t *seg_off_out, uint64_t *lengths_out)
{
	MC2_REQUIRE(ctx && s, "mc2_seqs_download_segments: NULL argument");
	MC2_CUDA(cudaSetDevice(ctx->device));
	cudaStream_t st = ctx->stream;
	if (segs_out && s->total_segs) MC2_CUDA(cudaMemcpyAsync(segs_out, s->segs, s->total_segs * 8, cudaMemcpyDeviceToHost, st));
	if (seg_off_out) MC2_CUDA(cudaMemcpyAsync(seg_off_out, s->seg_off, (s->n + 1) * 8, cudaMemcpyDeviceToHost, st));
	if (lengths_out && s->n) MC2_CUDA(cudaMemcpyAsync(lengths_out, s->len, s->n * 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	return MC2_OK;
}

uint64_t mc2_seqs_total_segments(const mc2_seqs *s)
{
	return s ? s->total_segs : 0;
}

int mc2_host_register(void *ptr, uint64_t bytes)
{
	MC2_REQUIRE(ptr != nullptr && bytes > 0, "mc2_host_register: NULL or empty range");
	MC2_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
	return MC2_OK;
}

int mc2_host_unregister(void *ptr)
{
	MC2_REQUIRE(ptr != nullptr, "mc2_host_unregister: NULL");
	MC2_CUDA(cudaHostUnregister(ptr));
	return MC2_OK;
}

void mc2_seqs_free(mc2_seqs *s)
{
	if (!s) {
		return;
	}
	cudaFree(s->packed);
	cudaFree(s->word_off);
	cudaFree(s->len);
	cudaFree(s->segs);
	cudaFree(s->seg_off);
	delete s;
}

uint64_t mc2_seqs_count(const mc2_seqs *s)
{
	return s ? s->n : 0;
}

uint64_t mc2_seqs_total_bases(const mc2_seqs *s)
{
	return s ? s->total_bases : 0;
}

static int check_k_eb(int k, int eb)
{
	MC2_REQUIRE(k >= 1 && k <= 12, "k must be in 1..12");
	MC2_REQUIRE(eb == 1 || eb == 2 || eb == 4 || eb == 8, "elem_bytes must be 1, 2, 4 or 8 (--datatype 8/16/32/64)");
	return MC2_OK;
}

static int count_into(mc2_ctx *ctx, const mc2_seqs *seqs, int k, int eb, u64 init, mc2_hset *h)
{
	int rc = reset_err(ctx);
	if (rc == MC2_OK) rc = launch_count(ctx, seqs, k, eb, h, init);
	if (rc == MC2_OK) rc = fetch_err(ctx);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	return check_err(ctx);
}

int mc2_count_kmers(mc2_ctx *ctx, const mc2_seqs *seqs, int k, int elem_bytes, mc2_hset **out)
{
	MC2_REQUIRE(ctx && seqs && out, "mc2_count_kmers: NULL argument");
	*out = nullptr;
	int rc = check_k_eb(k, elem_bytes);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaSetDevice(ctx->device));
	mc2_hset *h = nullptr;
	rc = alloc_hset(ctx, seqs->n, k, elem_bytes, &h);
	if (rc != MC2_OK) return rc;
	rc = count_into(ctx, seqs, k, elem_bytes, 1, h);
	if (rc == MC2_OK) rc = refresh_max_sum(ctx, h);
	if (rc != MC2_OK) {
		mc2_hset_free(h);
		return rc;
	}
	h->counted = 1;
	*out = h;
	return MC2_OK;
}

int mc2_hset_alloc(mc2_ctx *ctx, uint64_t n, int k, int elem_bytes, mc2_hset **out)
{
	MC2_REQUIRE(ctx && out, "mc2_hset_alloc: NULL argument");
	*out = nullptr;
	int rc = check_k_eb(k, elem_bytes);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaSetDevice(ctx->device));
	mc2_hset *h = nullptr;
	rc = alloc_hset(ctx, n, k, elem_bytes, &h);
	if (rc != MC2_OK) return rc;
	const u64 nn = n ? n : 1;
	cudaStream_t st = ctx->stream;
	cudaError_t e = cudaMemsetAsync(h->bins, 0, nn * h->N * (u64)elem_bytes, st);
	if (e == cudaSuccess) e = cudaMemsetAsync(h->mag, 0, nn * 8, st);
	if (e == cudaSuccess) e = cudaMemsetAsync(h->sum, 0, nn * 8, st);
	if (e == cudaSuccess) e = cudaMemsetAsync(h->sumsq, 0, nn * 8, st);
	if (e == cudaSuccess) e = cudaMemsetAsync(h->len, 0, nn * 8, st);
	if (e == cudaSuccess) e = cudaMemsetAsync(h->mers1, 0, nn * 32, st);
	if (e == cudaSuccess) e = cudaMemsetAsync(h->stddev, 0, nn * 8, st);
	if (e == cudaSuccess) e = cudaMemsetAsync(h->novf, 0, nn * 4, st);
	if (e == cudaSuccess) e = cudaMemsetAsync(h->maxc, 0, nn * 4, st);
	if (e == cudaSuccess) e = cudaStreamSynchronize(st);
	if (e != cudaSuccess) {
		mc2_hset_free(h);
		return cuda_fail(e, "mc2_hset_alloc", __FILE__, __LINE__);
	}
	*out = h;
	return MC2_OK;
}

int mc2_count_kmers_into_rows(mc2_ctx *ctx, const mc2_seqs *seqs, mc2_hset *dst, uint64_t first_row)
{
	MC2_REQUIRE(ctx && seqs && dst, "mc2_count_kmers_into_rows: NULL argument");
	MC2_REQUIRE(first_row <= dst->n && seqs->n <= dst->n - first_row, "mc2_count_kmers_into_rows: rows out of range");
	MC2_CUDA(cudaSetDevice(ctx->device));
	dst->lane_off_valid = 0;
	dst->cum16_valid = 0;
	dst->counted = 0;
	drop_rc(dst);
	if (seqs->n == 0) {
		return MC2_OK;
	}
	// a window of the destination set: the same arrays, offset by first_row
	mc2_hset view = *dst;
	view.n = seqs->n;
	view.bins = (char *)dst->bins + first_row * dst->N * (u64)dst->eb;
	view.mag = dst->mag + first_row;
	view.sum = dst->sum + first_row;
	view.sumsq = dst->sumsq + first_row;
	view.len = dst->len + first_row;
	view.mers1 = dst->mers1 + first_row * 4;
	view.stddev = dst->stddev + first_row;
	view.novf = dst->novf + first_row;
	view.maxc = dst->maxc + first_row;
	view.lane_off = nullptr;
	view.cum16 = nullptr;
	view.cum16s = nullptr;
	view.plane8 = nullptr;
	view.cumsum = nullptr;
	return count_into(ctx, seqs, dst->k, dst->eb, 1, &view);
}

int mc2_hset_refresh(mc2_ctx *ctx, mc2_hset *h, int32_t set_mag)
{
	MC2_REQUIRE(ctx && h, "mc2_hset_refresh: NULL argument");
	MC2_CUDA(cudaSetDevice(ctx->device));
	h->lane_off_valid = 0;
	h->cum16_valid = 0;
	h->counted = 0;
	drop_rc(h);
	if (h->n == 0) {
		return MC2_OK;
	}
	int rc = launch_sideband(ctx, h, set_mag != 0);
	if (rc == MC2_OK) rc = refresh_max_sum(ctx, h);
	return rc;
}

int mc2_hset_largest_count(const mc2_hset *h, uint64_t *largest_count)
{
	MC2_REQUIRE(h && largest_count, "mc2_hset_largest_count: NULL argument");
	if (!h->counted) {
		set_error("mc2_hset_largest_count: the set was not produced by mc2_count_kmers (or its rows were overwritten)");
		return MC2_ERR_UNSUPPORTED;
	}
	// u64 table initialised to 1 plus the multiplicity (CRunner.cpp:69-74); an empty input leaves largest_count at 0 (:57)
	*largest_count = h->n ? 1 + h->max_count : 0;
	return MC2_OK;
}

int mc2_width_for_count(uint64_t largest_count)
{
	// CRunner.cpp:108-126
	if (largest_count <= 0xFFull) return 1;
	if (largest_count <= 0xFFFFull) return 2;
	if (largest_count <= 0xFFFFFFFFull) return 4;
	return 8;
}

int mc2_count_kmers_auto(mc2_ctx *ctx, const mc2_seqs *seqs, int k, uint64_t *largest_count, int *elem_bytes, mc2_hset **out)
{
	MC2_REQUIRE(ctx && seqs && out, "mc2_count_kmers_auto: NULL argument");
	*out = nullptr;
	if (seqs->total_segs && seqs->min_seg_len < (u64)k) {
		// quirk Q6: the reference's detection pass has no `length >= k` guard and hashes k characters from the start of
		// a shorter segment, reading past it (it throws or reads foreign memory); there is no result to reproduce
		set_error("mc2_count_kmers_auto: a segment is shorter than k (the reference's width detection reads past it)");
		return MC2_ERR_INPUT;
	}
	mc2_hset *h = nullptr;
	int rc = mc2_count_kmers(ctx, seqs, k, 1, &h); // multiplicities are exact at any width; 8-bit output is the cheapest
	if (rc != MC2_OK) return rc;
	uint64_t largest = 0;
	mc2_hset_largest_count(h, &largest);
	const int eb = mc2_width_for_count(largest);
	if (eb != 1) {
		mc2_hset_free(h);
		h = nullptr;
		rc = mc2_count_kmers(ctx, seqs, k, eb, &h);
		if (rc != MC2_OK) return rc;
	}
	if (largest_count) *largest_count = largest;
	if (elem_bytes) *elem_bytes = eb;
	*out = h;
	return MC2_OK;
}

int mc2_count_kmers_into(mc2_ctx *ctx, const mc2_seqs *seqs, mc2_hset *dst)
{
	MC2_REQUIRE(ctx && seqs && dst, "mc2_count_kmers_into: NULL argument");
	MC2_REQUIRE(dst->n == seqs->n, "mc2_count_kmers_into: the set holds a different number of rows");
	MC2_CUDA(cudaSetDevice(ctx->device));
	dst->lane_off_valid = 0;
	dst->cum16_valid = 0;
	drop_rc(dst);
	int rc = count_into(ctx, seqs, dst->k, dst->eb, 1, dst);
	if (rc == MC2_OK) rc = refresh_max_sum(ctx, dst);
	dst->counted = rc == MC2_OK;
	return rc;
}

int mc2_kmer_table_increment(mc2_ctx *ctx, const char *codes, int32_t first, int32_t last, int k, int elem_bytes,
			     uint64_t init_value, void *values_out, int32_t *ret)
{
	MC2_REQUIRE(ctx && codes && values_out && ret, "mc2_kmer_table_increment: NULL argument");
	int rc = check_k_eb(k, elem_bytes);
	if (rc != MC2_OK) return rc;
	MC2_REQUIRE(first >= 0 && last >= first, "mc2_kmer_table_increment: need 0 <= first <= last");
	// the k-mers with starts first..last span codes[first .. last+k-1]: one sequence, one segment
	uint64_t seq_off[2] = {0, (uint64_t)last + (uint64_t)k};
	int32_t seg[2] = {first, last + k - 1};
	uint64_t seg_off[2] = {0, 1};
	mc2_seqs *s = nullptr;
	rc = mc2_seqs_upload(ctx, codes, seq_off, 1, seg, seg_off, &s);
	if (rc != MC2_OK) return rc;
	mc2_hset *h = nullptr;
	rc = alloc_hset(ctx, 1, k, elem_bytes, &h);
	if (rc == MC2_OK) rc = count_into(ctx, s, k, elem_bytes, init_value, h);
	int32_t novf = 0;
	if (rc == MC2_OK) rc = mc2_hset_download(ctx, h, 0, 1, values_out, nullptr, nullptr, nullptr, nullptr, &novf, nullptr);
	*ret = novf ? -1 : 0;
	mc2_hset_free(h);
	mc2_seqs_free(s);
	return rc;
}

/* ---- histogram sets --------------------------------------------------------------------------- */
int mc2_hset_from_host(mc2_ctx *ctx, const void *bins, uint64_t n, int k, int elem_bytes, const uint64_t *mag,
		       const uint64_t *len, mc2_hset **out)
{
	MC2_REQUIRE(ctx && out && (n == 0 || (bins && len)), "mc2_hset_from_host: NULL argument");
	*out = nullptr;
	int rc = check_k_eb(k, elem_bytes);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaSetDevice(ctx->device));
	mc2_hset *h = nullptr;
	rc = alloc_hset(ctx, n, k, elem_bytes, &h);
	if (rc != MC2_OK) return rc;
	cudaError_t e = cudaSuccess;
	if (n) {
		e = cudaMemcpyAsync(h->bins, bins, n * h->N * (u64)elem_bytes, cudaMemcpyHostToDevice, ctx->stream);
		if (e == cudaSuccess) e = cudaMemcpyAsync(h->len, len, n * 8, cudaMemcpyHostToDevice, ctx->stream);
		if (e == cudaSuccess && mag) e = cudaMemcpyAsync(h->mag, mag, n * 8, cudaMemcpyHostToDevice, ctx->stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(h->mers1, 0, n * 32, ctx->stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(h->stddev, 0, n * 8, ctx->stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(h->novf, 0, n * 4, ctx->stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(h->maxc, 0, n * 4, ctx->stream);
	}
	if (e != cudaSuccess) {
		mc2_hset_free(h);
		return cuda_fail(e, "mc2_hset_from_host copies", __FILE__, __LINE__);
	}
	rc = launch_sideband(ctx, h, mag == nullptr);
	if (rc == MC2_OK) rc = refresh_max_sum(ctx, h);
	if (rc != MC2_OK) {
		mc2_hset_free(h);
		return rc;
	}
	*out = h;
	return MC2_OK;
}

int mc2_hset_from_device(mc2_ctx *ctx, const void *d_bins, uint64_t n, int k, int elem_bytes, const uint64_t *d_mag,
			 const uint64_t *d_len, mc2_hset **out)
{
	MC2_REQUIRE(ctx && out && (n == 0 || (d_bins && d_len)), "mc2_hset_from_device: NULL argument");
	*out = nullptr;
	int rc = check_k_eb(k, elem_bytes);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaSetDevice(ctx->device));
	mc2_hset *h = nullptr;
	rc = alloc_hset(ctx, n, k, elem_bytes, &h);
	if (rc != MC2_OK) return rc;
	cudaError_t e = cudaSuccess;
	if (n) {
		e = cudaMemcpyAsync(h->bins, d_bins, n * h->N * (u64)elem_bytes, cudaMemcpyDeviceToDevice, ctx->stream);
		if (e == cudaSuccess) e = cudaMemcpyAsync(h->len, d_len, n * 8, cudaMemcpyDeviceToDevice, ctx->stream);
		if (e == cudaSuccess && d_mag) e = cudaMemcpyAsync(h->mag, d_mag, n * 8, cudaMemcpyDeviceToDevice, ctx->stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(h->mers1, 0, n * 32, ctx->stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(h->stddev, 0, n * 8, ctx->stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(h->novf, 0, n * 4, ctx->stream);
		if (e == cudaSuccess) e = cudaMemsetAsync(h->maxc, 0, n * 4, ctx->stream);
	}
	if (e != cudaSuccess) {
		mc2_hset_free(h);
		return cuda_fail(e, "mc2_hset_from_device copies", __FILE__, __LINE__);
	}
	rc = launch_sideband(ctx, h, d_mag == nullptr);
	if (rc == MC2_OK) rc = refresh_max_sum(ctx, h);
	if (rc != MC2_OK) {
		mc2_hset_free(h);
		return rc;
	}
	*out = h;
	return MC2_OK;
}

int mc2_hset_update_from_device(mc2_ctx *ctx, mc2_hset *h, const void *d_bins, const uint64_t *d_mag, const uint64_t *d_len)
{
	MC2_REQUIRE(ctx && h && d_bins && d_len, "mc2_hset_update_from_device: NULL argument");
	MC2_CUDA(cudaSetDevice(ctx->device));
	const u64 n = h->n;
	if (n == 0) {
		return MC2_OK;
	}
	h->lane_off_valid = 0;
	h->cum16_valid = 0;
	h->counted = 0;
	drop_rc(h);
	MC2_CUDA(cudaMemcpyAsync(h->bins, d_bins, n * h->N * (u64)h->eb, cudaMemcpyDeviceToDevice, ctx->stream));
	MC2_CUDA(cudaMemcpyAsync(h->len, d_len, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
	if (d_mag) MC2_CUDA(cudaMemcpyAsync(h->mag, d_mag, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
	int rc = launch_sideband(ctx, h, d_mag == nullptr);
	if (rc == MC2_OK) rc = refresh_max_sum(ctx, h);
	return rc;
}

void *mc2_hset_device_sideband(const mc2_hset *h, int which)
{
	if (!h) {
		return nullptr;
	}
	switch (which) {
	case 0: return h->mag;
	case 1: return h->len;
	case 2: return h->sum;
	case 3: return h->sumsq;
	}
	return nullptr;
}

void mc2_hset_free(mc2_hset *h)
{
	if (!h) {
		return;
	}
	cudaFree(h->bins);
	cudaFree(h->mag);
	cudaFree(h->sum);
	cudaFree(h->sumsq);
	cudaFree(h->len);
	cudaFree(h->mers1);
	cudaFree(h->stddev);
	cudaFree(h->novf);
	cudaFree(h->maxc);
	cudaFree(h->lane_off);
	cudaFree(h->cum16);
	cudaFree(h->cum16s);
	cudaFree(h->plane8);
	cudaFree(h->cumsum);
	mc2_hset_free(h->rc);
	delete h;
}

uint64_t mc2_hset_count(const mc2_hset *h)
{
	return h ? h->n : 0;
}

int mc2_hset_k(const mc2_hset *h)
{
	return h ? h->k : 0;
}

int mc2_hset_elem_bytes(const mc2_hset *h)
{
	return h ? h->eb : 0;
}

void *mc2_hset_device_bins(const mc2_hset *h)
{
	return h ? h->bins : nullptr;
}

int mc2_hset_download(mc2_ctx *ctx, const mc2_hset *h, uint64_t first, uint64_t count, void *bins, uint64_t *mag,
		      uint64_t *len, uint64_t *mers1, double *stddev, int32_t *n_overflow, uint32_t *max_count)
{
	MC2_REQUIRE(ctx && h, "mc2_hset_download: NULL argument");
	MC2_REQUIRE(first <= h->n && count <= h->n - first, "mc2_hset_download: row range out of bounds");
	if (count == 0) {
		return MC2_OK;
	}
	cudaStream_t st = ctx->stream;
	const u64 rb = h->N * (u64)h->eb;
	if (bins) MC2_CUDA(cudaMemcpyAsync(bins, (const char *)h->bins + first * rb, count * rb, cudaMemcpyDeviceToHost, st));
	if (mag) MC2_CUDA(cudaMemcpyAsync(mag, h->mag + first, count * 8, cudaMemcpyDeviceToHost, st));
	if (len) MC2_CUDA(cudaMemcpyAsync(len, h->len + first, count * 8, cudaMemcpyDeviceToHost, st));
	if (mers1) MC2_CUDA(cudaMemcpyAsync(mers1, h->mers1 + 4 * first, count * 32, cudaMemcpyDeviceToHost, st));
	if (stddev) MC2_CUDA(cudaMemcpyAsync(stddev, h->stddev + first, count * 8, cudaMemcpyDeviceToHost, st));
	if (n_overflow) MC2_CUDA(cudaMemcpyAsync(n_overflow, h->novf + first, count * 4, cudaMemcpyDeviceToHost, st));
	if (max_count) MC2_CUDA(cudaMemcpyAsync(max_count, h->maxc + first, count * 4, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	return MC2_OK;
}

int mc2_hset_copy_to_device(mc2_ctx *ctx, const mc2_hset *h, uint64_t first, uint64_t count, void *d_bins,
			    uint64_t *d_mag, uint64_t *d_len)
{
	MC2_REQUIRE(ctx && h, "mc2_hset_copy_to_device: NULL argument");
	MC2_REQUIRE(first <= h->n && count <= h->n - first, "mc2_hset_copy_to_device: row range out of bounds");
	if (count == 0) {
		return MC2_OK;
	}
	cudaStream_t st = ctx->stream;
	const u64 rb = h->N * (u64)h->eb;
	if (d_bins) MC2_CUDA(cudaMemcpyAsync(d_bins, (const char *)h->bins + first * rb, count * rb, cudaMemcpyDeviceToDevice, st));
	if (d_mag) MC2_CUDA(cudaMemcpyAsync(d_mag, h->mag + first, count * 8, cudaMemcpyDeviceToDevice, st));
	if (d_len) MC2_CUDA(cudaMemcpyAsync(d_len, h->len + first, count * 8, cudaMemcpyDeviceToDevice, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	return MC2_OK;
}

int mc2_hset_set_sideband(mc2_ctx *ctx, mc2_hset *h, uint64_t count, const uint64_t *rows, const uint64_t *mag,
			  const uint64_t *len)
{
	MC2_REQUIRE(ctx && h && (count == 0 || rows), "mc2_hset_set_sideband: NULL argument");
	drop_rc(h);
	for (u64 i = 0; i < count; i++) {
		MC2_REQUIRE(rows[i] < h->n, "mc2_hset_set_sideband: row out of range");
		if (mag) MC2_CUDA(cudaMemcpyAsync(h->mag + rows[i], mag + i, 8, cudaMemcpyHostToDevice, ctx->stream));
		if (len) MC2_CUDA(cudaMemcpyAsync(h->len + rows[i], len + i, 8, cudaMemcpyHostToDevice, ctx->stream));
	}
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC2_OK;
}

int mc2_hset_set_row(mc2_ctx *ctx, mc2_hset *dst, uint64_t dst_row, const mc2_hset *src, uint64_t src_row)
{
	MC2_REQUIRE(ctx && dst && src, "mc2_hset_set_row: NULL argument");
	MC2_REQUIRE(dst->k == src->k && dst->eb == src->eb, "mc2_hset_set_row: sets differ in k or width");
	MC2_REQUIRE(dst_row < dst->n && src_row < src->n, "mc2_hset_set_row: row out of range");
	dst->lane_off_valid = 0;
	dst->cum16_valid = 0;
	dst->counted = 0;
	drop_rc(dst);
	cudaStream_t st = ctx->stream;
	const u64 rb = dst->N * (u64)dst->eb;
	// DivergencePoint::set (src/clutil/DivergencePoint.cpp:182-190): points + length (+header/id), NOT mag
	MC2_CUDA(cudaMemcpyAsync((char *)dst->bins + dst_row * rb, (const char *)src->bins + src_row * rb, rb, cudaMemcpyDeviceToDevice, st));
	MC2_CUDA(cudaMemcpyAsync(dst->len + dst_row, src->len + src_row, 8, cudaMemcpyDeviceToDevice, st));
	MC2_CUDA(cudaMemcpyAsync(dst->sum + dst_row, src->sum + src_row, 8, cudaMemcpyDeviceToDevice, st));
	MC2_CUDA(cudaMemcpyAsync(dst->sumsq + dst_row, src->sumsq + src_row, 8, cudaMemcpyDeviceToDevice, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	if (src->max_sum > dst->max_sum) {
		dst->max_sum = src->max_sum;
	}
	return MC2_OK;
}

int mc2_hset_assign_rows(mc2_ctx *ctx, mc2_hset *dst, uint64_t n, const uint64_t *dst_rows, const mc2_hset *src,
			 const uint64_t *src_rows, const uint64_t *mag, const uint64_t *len)
{
	MC2_REQUIRE(ctx && dst && src && (n == 0 || (dst_rows && src_rows)), "mc2_hset_assign_rows: NULL argument");
	MC2_REQUIRE(dst->k == src->k && dst->eb == src->eb, "mc2_hset_assign_rows: sets differ in k or width");
	if (n == 0) {
		return MC2_OK;
	}
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	// the destination's lane offsets stay valid when both sides have them (they are copied with the rows)
	const bool keep_loff = dst->lane_off_valid && src->lane_off_valid && dst->lane_off && src->lane_off;
	dst->lane_off_valid = keep_loff ? 1 : 0;
	dst->cum16_valid = 0;
	dst->counted = 0;
	drop_rc(dst);
	const int parts = 2 + (mag ? 1 : 0) + (len ? 1 : 0);
	std::vector<u64> idx((size_t)parts * n);
	for (u64 i = 0; i < n; i++) {
		MC2_REQUIRE(dst_rows[i] < dst->n && src_rows[i] < src->n, "mc2_hset_assign_rows: row out of range");
		idx[i] = dst_rows[i];
		idx[n + i] = src_rows[i];
		if (mag) idx[2 * n + i] = mag[i];
		if (len) idx[(size_t)(2 + (mag ? 1 : 0)) * n + i] = len[i];
	}
	CtxExtra *x = extra(ctx);
	int rc = ensure(x->d[B_IA], idx.size() * 8, false);
	if (rc != MC2_OK) return rc;
	bool staged = false;
	rc = h2d(ctx, x->d[B_IA].p, idx.data(), idx.size() * 8, &staged);
	if (rc != MC2_OK) return rc;
	u64 want = (n + 7) / 8, cap = (u64)ctx->sm_count * 8;
	int grid = (int)(want < cap ? want : cap);
	assign_rows_kernel<<<grid, 256, 0, ctx->stream>>>((char *)dst->bins, dst->mag, dst->sum, dst->sumsq, dst->len,
							   (const char *)src->bins, src->sum, src->sumsq, src->len, dst->N * (u64)dst->eb, n,
							   (const u64 *)x->d[B_IA].p, mag ? 1 : 0, len ? 1 : 0,
							   keep_loff ? dst->lane_off : nullptr, keep_loff ? src->lane_off : nullptr);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	if (!staged) {
		MC2_CUDA(cudaStreamSynchronize(ctx->stream)); // idx is a host temporary; a staged copy is stream-ordered instead
	}
	if (src->max_sum > dst->max_sum) {
		dst->max_sum = src->max_sum;
	}
	return MC2_OK;
}

/* ---- model ------------------------------------------------------------------------------------ */
int mc2_model_create(mc2_ctx *ctx, const mc2_model_desc *desc, mc2_model **out)
{
	MC2_REQUIRE(ctx && desc && out, "mc2_model_create: NULL argument");
	*out = nullptr;
	DevModel dm;
	int rc = model_need(*desc, dm);
	if (rc != MC2_OK) return rc;
	mc2_model *m = new (std::nothrow) mc2_model();
	MC2_REQUIRE(m != nullptr, "out of host memory");
	m->ctx = ctx;
	m->desc = *desc;
	m->dm = dm;
	static std::atomic<unsigned long long> next_uid{1};
	m->uid = next_uid++;
	*out = m;
	return MC2_OK;
}

void mc2_model_free(mc2_model *m)
{
	delete m;
}

int mc2_model_desc_from_file(const char *path, int which, mc2_model_desc *desc, int *k_out, double *id_out,
			     int *elem_bytes_out, int *mode_out)
{
	MC2_REQUIRE(path && desc, "mc2_model_desc_from_file: NULL argument");
	MC2_REQUIRE(which == 0 || which == 1, "mc2_model_desc_from_file: which must be 0 (classifier) or 1 (regression)");
	std::ifstream in(path);
	if (!in) {
		set_error(std::string("cannot open weights file ") + path);
		return MC2_ERR_IO;
	}
	// header, Predictor.cpp:47-66
	std::string buf, datatype;
	int k = 0, max_feat = 0;
	unsigned mode = 0;
	double id = 0;
	uint64_t feats64 = 0;
	in >> buf >> k;
	in >> buf >> mode;
	in >> buf >> max_feat;
	in >> buf >> id;
	in >> buf >> datatype;
	in >> buf >> feats64;
	if (!in) {
		set_error("weights file: malformed header");
		return MC2_ERR_IO;
	}
	const bool has_c = mode & 1, has_r = mode & 2;
	if ((which == 0 && !has_c) || (which == 1 && !has_r)) {
		set_error("weights file does not contain the requested model block");
		return MC2_ERR_IO;
	}
	int blocks_to_skip = (which == 1 && has_c) ? 1 : 0;
	for (int blk = 0; blk <= blocks_to_skip; blk++) {
		// read_from, Predictor.cpp:125-185
		mc2_model_desc d;
		memset(&d, 0, sizeof d);
		int nc = 0;
		in >> buf >> nc;
		if (!in || nc < 1 || nc > MC2_MAX_COMBOS) {
			set_error("weights file: bad n_combos");
			return MC2_ERR_IO;
		}
		d.n_combos = nc;
		in >> d.weight[0];
		uint64_t have = 0;
		for (int c = 0; c < nc; c++) {
			int cmb;
			uint64_t flags;
			double wv;
			in >> cmb >> flags >> wv;
			if (!in || cmb < 0 || cmb > 3) {
				set_error("weights file: bad combo line");
				return MC2_ERR_IO;
			}
			d.weight[c + 1] = wv;
			d.combo_kind[c] = cmb;
			// Feature::add_feature, Feature.cpp:102-127: new singles appended in ascending flag-bit order
			int ni = 0;
			for (int b = 0; b < 64; b++) {
				uint64_t f = 1ULL << b;
				if (!(flags & f)) {
					continue;
				}
				if (!(have & f)) {
					if (d.n_singles >= MC2_MAX_SINGLES) {
						set_error("weights file: too many singles");
						return MC2_ERR_IO;
					}
					d.single_flag[d.n_singles++] = f;
					have |= f;
				}
				int ix = -1;
				for (int s = 0; s < d.n_singles; s++) {
					if (d.single_flag[s] == f) {
						ix = s;
					}
				}
				if (ni >= MC2_MAX_COMBO_IDX) {
					set_error("weights file: combo with too many singles");
					return MC2_ERR_IO;
				}
				d.combo_idx[c][ni++] = ix;
			}
			d.combo_nidx[c] = ni;
		}
		int ns = 0;
		in >> buf >> ns;
		if (!in || ns < 0 || ns > MC2_MAX_SINGLES) {
			set_error("weights file: bad n_singles");
			return MC2_ERR_IO;
		}
		for (int s = 0; s < ns; s++) {
			uint64_t f;
			double lo, hi;
			in >> f >> lo >> hi;
			if (!in) {
				set_error("weights file: bad single line");
				return MC2_ERR_IO;
			}
			for (int t = 0; t < d.n_singles; t++) { // Feature::set_normal, Feature.cpp:173-180
				if (d.single_flag[t] == f) {
					d.single_min[t] = lo;
					d.single_max[t] = hi;
				}
			}
		}
		d.bias = 0;
		d.regression = (blk == 1 || (which == 1 && !has_c)) ? 1 : 0;
		if (blk == blocks_to_skip) {
			*desc = d;
		}
	}
	if (k_out) *k_out = k;
	if (id_out) *id_out = id;
	if (mode_out) *mode_out = (int)mode;
	if (elem_bytes_out) {
		*elem_bytes_out = datatype == "uint8_t" ? 1 : datatype == "uint16_t" ? 2 : datatype == "uint32_t" ? 4 : datatype == "uint64_t" ? 8 : 0;
	}
	return MC2_OK;
}

/* ---- scoring ----------------------------------------------------------------------------------- */
static int fill_pair_args(mc2_ctx *ctx, const mc2_pairs *p, PairArgs &a, CtxExtra *x)
{
	MC2_REQUIRE(p->set_a && p->set_b, "pairs: set_a / set_b is NULL");
	const mc2_hset *A = p->set_a, *B = p->set_b;
	MC2_REQUIRE(A->k == B->k && A->eb == B->eb, "pairs: the two sets differ in k or histogram width");
	memset(&a, 0, sizeof a);
	a.binsA = A->bins;
	a.binsB = B->bins;
	a.sbA = Sideband{A->mag, A->sum, A->sumsq, A->len};
	a.sbB = Sideband{B->mag, B->sum, B->sumsq, B->len};
	a.N = A->N;
	a.eb = A->eb;
	a.n_pairs = p->n_pairs;
	a.a_begin = p->a_begin;
	a.b_begin = p->b_begin;
	a.a_bc = p->a_broadcast;
	a.b_bc = p->b_broadcast;
	a.len_filter = p->len_filter;
	a.anchor_is_b = p->anchor_is_b;
	a.cutoff = p->cutoff;
	a.err = ctx->d_err;
	a.max_sum = A->max_sum > B->max_sum ? A->max_sum : B->max_sum;
	a.loffA = a.loffB = nullptr;
	if (ensure_lane_off(ctx, A) == MC2_OK && ensure_lane_off(ctx, B) == MC2_OK && A->lane_off_valid && B->lane_off_valid) {
		a.loffA = A->lane_off;
		a.loffB = B->lane_off;
	}
	const u64 m = p->n_pairs;
	if (p->ia) {
		for (u64 j = 0; j < m; j++) {
			MC2_REQUIRE(p->ia[j] < A->n, "pairs: ia index out of range");
		}
		int rc = ensure(x->d[B_IA], m * 8, false);
		if (rc != MC2_OK) return rc;
		rc = h2d(ctx, x->d[B_IA].p, p->ia, m * 8);
		if (rc != MC2_OK) return rc;
		a.ia = (const u64 *)x->d[B_IA].p;
	} else {
		MC2_REQUIRE(m == 0 || (p->a_broadcast ? p->a_begin < A->n : (p->a_begin <= A->n && m <= A->n - p->a_begin)), "pairs: a range out of bounds");
	}
	if (p->ib) {
		for (u64 j = 0; j < m; j++) {
			MC2_REQUIRE(p->ib[j] < B->n, "pairs: ib index out of range");
		}
		int rc = ensure(x->d[B_IB], m * 8, false);
		if (rc != MC2_OK) return rc;
		rc = h2d(ctx, x->d[B_IB].p, p->ib, m * 8);
		if (rc != MC2_OK) return rc;
		a.ib = (const u64 *)x->d[B_IB].p;
	} else {
		MC2_REQUIRE(m == 0 || (p->b_broadcast ? p->b_begin < B->n : (p->b_begin <= B->n && m <= B->n - p->b_begin)), "pairs: b range out of bounds");
	}
	if (p->len_filter) {
		MC2_REQUIRE(p->cutoff > 0, "pairs: cutoff must be > 0 when len_filter is set");
	}
	if (p->bc_override) {
		// the broadcast row's mag / len come from the caller: a two-word device array addressed so that index `row` hits it
		const bool on_a = p->a_broadcast && !p->ia, on_b = p->b_broadcast && !p->ib;
		MC2_REQUIRE(on_a != on_b, "pairs: bc_override needs exactly one broadcast side without an index list");
		int rc = ensure(x->d[B_OVERRIDE], 16, false);
		if (rc != MC2_OK) return rc;
		const u64 two[2] = {p->bc_mag, p->bc_len};
		rc = h2d(ctx, x->d[B_OVERRIDE].p, two, 16);
		if (rc != MC2_OK) return rc;
		const u64 *dv = (const u64 *)x->d[B_OVERRIDE].p;
		if (on_a) {
			a.sbA.mag = dv - p->a_begin;
			a.sbA.len = dv + 1 - p->a_begin;
		} else {
			a.sbB.mag = dv - p->b_begin;
			a.sbB.len = dv + 1 - p->b_begin;
		}
	}
	return MC2_OK;
}

int mc2_score_pairs(mc2_ctx *ctx, const mc2_model *model, const mc2_pairs *pairs, double *score, double *dist,
		    uint8_t *close, double *cache, double *raw, uint8_t *skipped)
{
	MC2_REQUIRE(ctx && model && pairs, "mc2_score_pairs: NULL argument");
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	CtxExtra *x = extra(ctx);
	PairArgs a;
	int rc = fill_pair_args(ctx, pairs, a, x);
	if (rc != MC2_OK) return rc;
	const u64 m = pairs->n_pairs;
	if (m == 0) return MC2_OK;
	const u64 S = (u64)model->dm.n_singles;
	if (score) { rc = ensure(x->d[B_SCORE], m * 8, false); if (rc) return rc; a.score = (double *)x->d[B_SCORE].p; }
	if (dist) { rc = ensure(x->d[B_DIST], m * 8, false); if (rc) return rc; a.dist = (double *)x->d[B_DIST].p; }
	if (close) { rc = ensure(x->d[B_CLOSE], m, false); if (rc) return rc; a.close = (uint8_t *)x->d[B_CLOSE].p; }
	if (skipped) { rc = ensure(x->d[B_SKIP], m, false); if (rc) return rc; a.skipped = (uint8_t *)x->d[B_SKIP].p; }
	if (cache) { rc = ensure(x->d[B_CACHE], m * S * 8, false); if (rc) return rc; a.cache = (double *)x->d[B_CACHE].p; MC2_CUDA(cudaMemsetAsync(a.cache, 0, m * S * 8, ctx->stream)); }
	if (raw) { rc = ensure(x->d[B_RAW], m * S * 8, false); if (rc) return rc; a.raw = (double *)x->d[B_RAW].p; MC2_CUDA(cudaMemsetAsync(a.raw, 0, m * S * 8, ctx->stream)); }
	rc = reset_err(ctx);
	if (rc == MC2_OK) rc = launch_pair_score(ctx, model->dm, a);
	if (rc == MC2_OK) rc = fetch_err(ctx);
	if (rc != MC2_OK) return rc;
	if (score && (rc = d2h(ctx, score, a.score, m * 8)) != MC2_OK) return rc;
	if (dist && (rc = d2h(ctx, dist, a.dist, m * 8)) != MC2_OK) return rc;
	if (close && (rc = d2h(ctx, close, a.close, m)) != MC2_OK) return rc;
	if (skipped && (rc = d2h(ctx, skipped, a.skipped, m)) != MC2_OK) return rc;
	if (cache && (rc = d2h(ctx, cache, a.cache, m * S * 8)) != MC2_OK) return rc;
	if (raw && (rc = d2h(ctx, raw, a.raw, m * S * 8)) != MC2_OK) return rc;
	if ((rc = sync_stage(ctx)) != MC2_OK) return rc;
	return check_err(ctx);
}

struct ArgOutHost {
	long long best;
	double best_dist;
	int is_min;
	int has;
};

// shared by get_close / merge / filter: score on device, reduce on device, copy back only what the caller reads
static int score_and_reduce(mc2_ctx *ctx, const mc2_model *model, const mc2_pairs *pairs, int reduce_mode, ArgOutHost *red,
			    uint8_t *close_out, uint8_t *skipped_out)
{
	CtxExtra *x = extra(ctx);
	PairArgs a;
	int rc = fill_pair_args(ctx, pairs, a, x);
	if (rc != MC2_OK) return rc;
	const u64 m = pairs->n_pairs;
	rc = ensure(x->d[B_DIST], m * 8, false); if (rc) return rc;
	rc = ensure(x->d[B_CLOSE], m, false); if (rc) return rc;
	rc = ensure(x->d[B_SKIP], m, false); if (rc) return rc;
	a.dist = (double *)x->d[B_DIST].p;
	a.close = (uint8_t *)x->d[B_CLOSE].p;
	a.skipped = (uint8_t *)x->d[B_SKIP].p;
	// small batches with a reduction: the arg-max kernel also drops the close flags into the result slot, and ONE copy of
	// [result | error word | flags] ends the call
	const bool flags_in_slot = reduce_mode >= 0 && close_out && m <= 4096 - 128;
	uint8_t *d_flags = flags_in_slot ? reinterpret_cast<uint8_t *>(ctx->d_slot) + 128 : nullptr;
	rc = reset_err(ctx);
	if (rc == MC2_OK) rc = launch_pair_score(ctx, model->dm, a);
	if (rc == MC2_OK && reduce_mode >= 0) rc = launch_argmax(ctx, a.dist, a.skipped, a.close, m, reduce_mode, ctx->d_slot, d_flags);
	if (rc != MC2_OK) return rc;
	cudaStream_t st = ctx->stream;
	if (reduce_mode >= 0) {
		const size_t bytes = flags_in_slot ? 128 + (size_t)m : 128;
		MC2_CUDA(cudaMemcpyAsync(ctx->h_slot, ctx->d_slot, bytes, cudaMemcpyDeviceToHost, st)); // covers the error word
	} else {
		rc = fetch_err(ctx);
		if (rc != MC2_OK) return rc;
	}
	if (close_out && !flags_in_slot && (rc = d2h(ctx, close_out, a.close, m)) != MC2_OK) return rc;
	if (skipped_out && (rc = d2h(ctx, skipped_out, a.skipped, m)) != MC2_OK) return rc;
	rc = sync_stage(ctx);
	if (rc != MC2_OK) return rc;
	if (flags_in_slot) memcpy(close_out, reinterpret_cast<const char *>(ctx->h_slot) + 128, m);
	if (reduce_mode >= 0) *red = *reinterpret_cast<ArgOutHost *>(ctx->h_slot);
	return check_err(ctx);
}

static int get_close_impl(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q, int ovr, uint64_t q_mag,
			  uint64_t q_len, const mc2_hset *set_c, const uint64_t *cand, uint64_t cand_begin, uint64_t n_cand,
			  double cutoff, int64_t *best, double *best_dist, int32_t *is_min, uint8_t *marks);

int mc2_get_close(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q, const mc2_hset *set_c,
		  const uint64_t *cand, uint64_t cand_begin, uint64_t n_cand, double cutoff, int64_t *best,
		  double *best_dist, int32_t *is_min, uint8_t *marks)
{
	return get_close_impl(ctx, model, set_q, q, 0, 0, 0, set_c, cand, cand_begin, n_cand, cutoff, best, best_dist, is_min, marks);
}

int mc2_get_close_as(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q, uint64_t q_mag, uint64_t q_len,
		     const mc2_hset *set_c, const uint64_t *cand, uint64_t cand_begin, uint64_t n_cand, double cutoff,
		     int64_t *best, double *best_dist, int32_t *is_min, uint8_t *marks)
{
	return get_close_impl(ctx, model, set_q, q, 1, q_mag, q_len, set_c, cand, cand_begin, n_cand, cutoff, best, best_dist, is_min,
			      marks);
}

// ---- resident scan server (ScanMailbox, pair_score.cu scan_server_kernel) ----------------------------------------
// Small candidate lists over 1- or 2-byte histograms with a model the straight-line epilogue covers; everything else takes
// the launch path.  MC2_NO_SCAN_SERVER=1 (read per call, so tests can compare both paths in one process) turns it off.
static bool scan_server_eligible(const mc2_model *model, const mc2_hset *set_q, const mc2_hset *set_c, uint64_t n_cand)
{
	// measured from C++ (tools/call_latency.cpp): 9.3 us at <= 16 candidates, 11 us at 64, 17 us at 192; the launch path
	// costs 32 us whatever the count
	if (n_cand > 192 || getenv("MC2_NO_SCAN_SERVER")) {
		return false;
	}
	const DevModel &dm = model->dm;
	const u64 row_bytes = set_q->N * (u64)set_q->eb;
	const u64 ms = set_q->max_sum > set_c->max_sum ? set_q->max_sum : set_c->max_sum;
	return set_q->eb == set_c->eb && set_q->k == set_c->k && set_q->eb <= 2 && row_bytes % 1024 == 0 && dm.fast_epi && !dm.regression &&
	       !(dm.need & NEED_LOG) && ms < (1ULL << 26);
}

static int scan_server_start(mc2_ctx *ctx, const mc2_model *model, int eb, u64 first_seq)
{
	ctx->mb->w[7] = 0;
	ctx->mb->running = 1;
	std::atomic_thread_fence(std::memory_order_seq_cst);
	ctx->server_model_uid = model->uid;
	ctx->server_eb = eb;
	return launch_scan_server(ctx, model->dm, eb, first_seq);
}

static int scan_server_call(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q, int ovr, uint64_t q_mag,
			    uint64_t q_len, const mc2_hset *set_c, const uint64_t *cand, uint64_t cand_begin, uint64_t n_cand,
			    double cutoff, int64_t *best, double *best_dist, int32_t *is_min, uint8_t *marks)
{
	if (cand) {
		for (u64 j = 0; j < n_cand; j++) {
			MC2_REQUIRE(cand[j] < set_c->n, "mc2_get_close: candidate row out of range");
		}
	} else {
		MC2_REQUIRE(cand_begin <= set_c->n && n_cand <= set_c->n - cand_begin, "mc2_get_close: candidate range out of bounds");
	}
	if (!ctx->mb) {
		void *p = nullptr;
		if (cudaHostAlloc(&p, sizeof(ScanMailbox), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
			cudaGetLastError();
			return MC2_ERR_UNSUPPORTED; // no mapped memory: the launch path serves the call
		}
		memset(p, 0, sizeof(ScanMailbox));
		ctx->mb = reinterpret_cast<ScanMailbox *>(p);
		if (cudaStreamCreateWithFlags(&ctx->server_stream, cudaStreamNonBlocking) != cudaSuccess) {
			cudaGetLastError();
			cudaFreeHost(p);
			ctx->mb = nullptr;
			return MC2_ERR_UNSUPPORTED;
		}
		ctx->mb_seq = 0;
	}
	ScanMailbox *mb = ctx->mb;
	// rows written by work still queued on the context's stream must be complete before the server reads them
	if (cudaStreamQuery(ctx->stream) != cudaSuccess) {
		cudaGetLastError();
		MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	}
	// a server started with another model or element width leaves first
	if (mb->running && (ctx->server_model_uid != model->uid || ctx->server_eb != set_q->eb)) {
		mb->w[7] = 1;
		MC2_CUDA(cudaStreamSynchronize(ctx->server_stream));
	}
	const u64 seq = ++ctx->mb_seq;
	union { double d; unsigned long long u; } cu;
	cu.d = cutoff;
	volatile unsigned long long *w = mb->w;
	w[1] = q; w[2] = q_mag; w[3] = q_len; w[4] = cand_begin; w[5] = cu.u;
	// up to MC2_SCAN_INLINE ids of 32 bits ride in the header itself: one read of host memory fewer for the server
	bool ids_inline = cand != nullptr && n_cand <= MC2_SCAN_INLINE && set_c->n <= (1ull << 32);
	w[6] = (unsigned long long)(unsigned)n_cand | ((unsigned long long)(cand != nullptr) << 32) | ((unsigned long long)(ovr != 0) << 33) |
	       ((unsigned long long)ids_inline << 34);
	w[8] = (unsigned long long)set_q->bins; w[9] = (unsigned long long)set_c->bins;
	w[10] = (unsigned long long)set_q->mag; w[11] = (unsigned long long)set_q->sum;
	w[12] = (unsigned long long)set_q->sumsq; w[13] = (unsigned long long)set_q->len; w[14] = set_q->N;
	w[16] = (unsigned long long)set_c->mag; w[17] = (unsigned long long)set_c->sum;
	w[18] = (unsigned long long)set_c->sumsq; w[19] = (unsigned long long)set_c->len;
	if (cand) {
		if (ids_inline) {
			for (u64 j = 0; j < n_cand; j += 2) {
				const unsigned long long lo = cand[j], hi = j + 1 < n_cand ? cand[j + 1] : 0;
				w[scan_id_word((int)(j >> 1))] = lo | (hi << 32);
			}
		} else {
			memcpy(mb->cand, cand, n_cand * 8);
		}
	}
	std::atomic_thread_fence(std::memory_order_seq_cst);
	w[15] = seq; w[23] = seq; w[31] = seq; w[47] = seq; w[63] = seq;
	std::atomic_thread_fence(std::memory_order_seq_cst);
	w[0] = seq;
	std::atomic_thread_fence(std::memory_order_seq_cst);
	if (!mb->running) {
		int rc = scan_server_start(ctx, model, set_q->eb, seq);
		if (rc != MC2_OK) return rc;
	}
	const auto t0 = std::chrono::steady_clock::now();
	unsigned spins = 0;
	while (mb->r[7] != seq || mb->r[3] != seq) {
		if (!mb->running) {
			// the server left (idle) at the moment the request was posted: start it again for this request
			std::atomic_thread_fence(std::memory_order_seq_cst);
			if (mb->r[7] == seq && mb->r[3] == seq) break;
			MC2_CUDA(cudaStreamSynchronize(ctx->server_stream));
			int rc = scan_server_start(ctx, model, set_q->eb, seq);
			if (rc != MC2_OK) return rc;
		}
		if ((++spins & 0xFFF) == 0) {
			if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 5.0) {
				mb->w[7] = 1;
				cudaError_t e = cudaStreamSynchronize(ctx->server_stream);
				if (e != cudaSuccess) return cuda_fail(e, "scan server", __FILE__, __LINE__);
				set_error("mc2_get_close: the scan server did not answer");
				return MC2_ERR_CUDA;
			}
		}
#if defined(__x86_64__)
		__builtin_ia32_pause();
#endif
	}
	std::atomic_thread_fence(std::memory_order_seq_cst);
	union { double d; unsigned long long u; } bdv;
	bdv.u = mb->r[1];
	*best = (long long)mb->r[0];
	*best_dist = bdv.d;
	*is_min = (int)(mb->r[2] & 0xFFFFFFFFull);
	if (marks) {
		if (n_cand <= MC2_SCAN_MARKS_INLINE) {
			const unsigned long long m3[3] = {mb->r[4], mb->r[5], mb->r[6]};
			for (u64 j = 0; j < n_cand; j++) {
				marks[j] = (uint8_t)((m3[j >> 6] >> (j & 63)) & 1);
			}
		} else {
			memcpy(marks, mb->marks, n_cand);
		}
	}
	const int e = (int)(mb->r[2] >> 32);
	if (e & 1) {
		set_error("a feature threw in the reference (zero length in length_difference, or NaN after normalisation: Feature.cpp:136-154, 873-887)");
		return MC2_ERR_FEATURE;
	}
	if (e) {
		set_error("internal error in the scan server");
		return MC2_ERR_CUDA;
	}
	return MC2_OK;
}

static int get_close_impl(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q, int ovr, uint64_t q_mag,
			  uint64_t q_len, const mc2_hset *set_c, const uint64_t *cand, uint64_t cand_begin, uint64_t n_cand,
			  double cutoff, int64_t *best, double *best_dist, int32_t *is_min, uint8_t *marks)
{
	MC2_REQUIRE(ctx && model && set_q && set_c && best && best_dist && is_min, "mc2_get_close: NULL argument");
	MC2_REQUIRE(q < set_q->n, "mc2_get_close: query row out of range");
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	*best = -1;
	*best_dist = -1;
	*is_min = 1;
	if (n_cand == 0) return MC2_OK;
	if (scan_server_eligible(model, set_q, set_c, n_cand)) {
		const int rc = scan_server_call(ctx, model, set_q, q, ovr, q_mag, q_len, set_c, cand, cand_begin, n_cand, cutoff, best,
						best_dist, is_min, marks);
		if (rc != MC2_ERR_UNSUPPORTED) {
			return rc;
		}
	}
	mc2_pairs p;
	memset(&p, 0, sizeof p);
	p.set_a = set_c; // compute(candidate, query): candidate is the first argument (Trainer.cpp:49)
	p.set_b = set_q;
	p.n_pairs = n_cand;
	p.ia = cand;
	p.a_begin = cand_begin;
	p.b_begin = q;
	p.b_broadcast = 1;
	p.len_filter = 1;
	p.anchor_is_b = 1;
	p.cutoff = cutoff;
	p.bc_override = ovr;
	p.bc_mag = q_mag;
	p.bc_len = q_len;
	ArgOutHost r;
	int rc = score_and_reduce(ctx, model, &p, 0, &r, marks, nullptr);
	if (rc != MC2_OK) return rc;
	*best = r.best;
	*best_dist = r.best_dist;
	*is_min = r.is_min;
	return MC2_OK;
}

static int filter_impl(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_c, uint64_t center, int ovr, uint64_t c_mag,
		       uint64_t c_len, const mc2_hset *set_m, const uint64_t *members, uint64_t n_members, double id, uint8_t *keep);

int mc2_filter(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_c, uint64_t center, const mc2_hset *set_m,
	       const uint64_t *members, uint64_t n_members, double id, uint8_t *keep)
{
	return filter_impl(ctx, model, set_c, center, 0, 0, 0, set_m, members, n_members, id, keep);
}

int mc2_filter_as(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_c, uint64_t center, uint64_t c_mag, uint64_t c_len,
		  const mc2_hset *set_m, const uint64_t *members, uint64_t n_members, double id, uint8_t *keep)
{
	return filter_impl(ctx, model, set_c, center, 1, c_mag, c_len, set_m, members, n_members, id, keep);
}

static int filter_impl(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_c, uint64_t center, int ovr, uint64_t c_mag,
		       uint64_t c_len, const mc2_hset *set_m, const uint64_t *members, uint64_t n_members, double id, uint8_t *keep)
{
	MC2_REQUIRE(ctx && model && set_c && set_m && (n_members == 0 || (members && keep)), "mc2_filter: NULL argument");
	MC2_REQUIRE(center < set_c->n, "mc2_filter: center row out of range");
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	if (n_members == 0) return MC2_OK;
	mc2_pairs p;
	memset(&p, 0, sizeof p);
	p.set_a = set_c; // classify(center, member), Trainer.cpp:133
	p.set_b = set_m;
	p.n_pairs = n_members;
	p.a_begin = center;
	p.a_broadcast = 1;
	p.ib = members;
	p.len_filter = 1;
	p.anchor_is_b = 0;
	p.cutoff = id;
	p.bc_override = ovr;
	p.bc_mag = c_mag;
	p.bc_len = c_len;
	// keep <=> in window and round(score) != 0 ; the kernel's close flag is round(score) > 0 and score >= 0 always
	// holds for logistic(sum)+bias with bias >= -0.5; for generality fetch the scores when bias is negative.
	if (model->dm.bias < 0) {
		std::vector<double> sc(n_members);
		std::vector<uint8_t> sk(n_members);
		int rc = mc2_score_pairs(ctx, model, &p, sc.data(), nullptr, nullptr, nullptr, nullptr, sk.data());
		if (rc != MC2_OK) return rc;
		for (u64 j = 0; j < n_members; j++) {
			keep[j] = !sk[j] && std::round(sc[j]) != 0;
		}
		return MC2_OK;
	}
	return score_and_reduce(ctx, model, &p, -1, nullptr, keep, nullptr);
}

int mc2_merge(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *centers, const uint64_t *rows, int64_t cur,
	      int64_t begin, int64_t last, double id, int64_t *out)
{
	MC2_REQUIRE(ctx && model && centers && rows && out, "mc2_merge: NULL argument");
	MC2_REQUIRE(cur >= 0 && begin >= 0, "mc2_merge: negative index");
	// Trainer<T>::merge merges on round(classify_sum(sum)) == 1 (src/cluster/Trainer.cpp:100-103); the kernels flag
	// round(score) > 0, which is the same set only while logistic + bias stays below 1.5 and above -0.5
	if (model->dm.regression || model->dm.bias >= 0.5 || model->dm.bias < -0.5) {
		set_error("mc2_merge: needs a classifier with -0.5 <= bias < 0.5");
		return MC2_ERR_UNSUPPORTED;
	}
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	*out = 0;
	if (last < begin) return MC2_OK;
	mc2_pairs p;
	memset(&p, 0, sizeof p);
	p.set_a = centers; // compute(*cen, *p): the other center first (Trainer.cpp:93)
	p.set_b = centers;
	p.n_pairs = (u64)(last - begin + 1);
	p.ia = rows + begin;
	p.b_begin = rows[cur];
	p.b_broadcast = 1;
	p.len_filter = 1;
	p.anchor_is_b = 1;
	p.cutoff = id;
	MC2_REQUIRE(rows[cur] < centers->n, "mc2_merge: current center row out of range");
	ArgOutHost r;
	int rc = score_and_reduce(ctx, model, &p, 1, &r, nullptr, nullptr);
	if (rc != MC2_OK) return rc;
	// mode 1 returns the position inside [begin,last] of the winner; has == 0 when no candidate is close
	*out = r.has ? begin + r.best : 0;
	return MC2_OK;
}

// the model of an identity search for min_identity: clamp(sum, 0, 1) >= t <=> sum >= t for 0 < t <= 1 (and t > 1 keeps
// nothing, which the same threshold also rejects): the screen's threshold on the sum is t itself.  t <= 0 keeps every
// in-window pair: nothing to screen.
static DevModel identity_model(const mc2_model *model, double min_identity)
{
	DevModel dm = model->dm;
	if (min_identity > 0) {
		dm.scr_thr = screen_threshold(min_identity);
	} else {
		dm.scr_ok = 0;
	}
	return dm;
}

// One launch of the all-pairs sweep into device buffers of capacity max_out (arguments checked by the caller): *total = all
// survivors (may exceed max_out), the sweep's diagnostics in last_exact / last_coarse / last_inline.  The device error word is fetched
// into ctx->h_err, not checked.
static int run_sweep(mc2_ctx *ctx, const DevModel &dm, int identity, double min_identity, const mc2_hset *set_q, u64 q_begin,
		     u64 q_end, const mc2_hset *set_d, u64 d_begin, u64 d_end, int32_t upper_only, double cutoff, u64 max_out,
		     u64 *d_out_q, u64 *d_out_d, double *d_out_score, u64 *total, uint64_t *n_scored)
{
	CtxExtra *x = extra(ctx);
	int rc = ensure(x->d[B_MISC], 64, false);
	if (rc) return rc;
	u64 *d_counters = (u64 *)x->d[B_MISC].p;
	MC2_CUDA(cudaMemsetAsync(d_counters, 0, 64, ctx->stream));
	rc = reset_err(ctx);
	if (rc == MC2_OK)
		rc = launch_all_pairs(ctx, dm, set_q, q_begin, q_end, set_d, d_begin, d_end, upper_only, cutoff, max_out, d_out_q, d_out_d,
				      d_out_score, d_counters, identity, min_identity);
	if (rc == MC2_OK) rc = fetch_err(ctx);
	if (rc != MC2_OK) return rc;
	cudaStream_t st = ctx->stream;
	MC2_CUDA(cudaMemcpyAsync(ctx->h_slot, d_counters, 40, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	*total = ((u64 *)ctx->h_slot)[0];
	if (n_scored) *n_scored = ((u64 *)ctx->h_slot)[1];
	x->last_exact = ((u64 *)ctx->h_slot)[2];
	x->last_coarse = ((u64 *)ctx->h_slot)[3] != 0;
	x->last_inline = ((u64 *)ctx->h_slot)[4];
	x->sum_inline += x->last_inline;
	return MC2_OK;
}

// the sweep behind mc2_all_pairs and mc2_identity_pairs (`who` names the entry point in error messages); identity != 0:
// survivors are the pairs whose regression score is >= min_identity, dm carries the screen threshold of that search
static int sweep_pairs(const char *who, mc2_ctx *ctx, const DevModel &dm, int identity, double min_identity, const mc2_hset *set_q,
		       uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end, int32_t upper_only,
		       double cutoff, uint64_t max_out, uint64_t *out_q, uint64_t *out_d, double *out_score, uint64_t *n_out,
		       uint64_t *n_scored)
{
	const std::string w(who);
	MC2_REQUIRE(q_begin <= q_end && q_end <= set_q->n && d_begin <= d_end && d_end <= set_d->n, w + ": row range out of bounds");
	MC2_REQUIRE(set_q->k == set_d->k && set_q->eb == set_d->eb, w + ": the two sets differ in k or histogram width");
	MC2_REQUIRE(cutoff > 0, w + ": cutoff must be > 0");
	MC2_REQUIRE((q_end - q_begin) * ((d_end - d_begin + 31) / 32) < (1ULL << 32),
		    w + ": more than 2^32 (query row, 32-column block) groups in one call; split the query range");
	MC2_REQUIRE((dm.regression != 0) == (identity != 0), w + (identity ? ": needs a regression model" : ": needs a classifier model"));
	MC2_CUDA(cudaSetDevice(ctx->device));
	*n_out = 0;
	if (n_scored) *n_scored = 0;
	CtxExtra *x = extra(ctx);
	x->last_exact = 0;
	x->last_coarse = 0;
	x->last_inline = x->sum_inline = 0;
	if (q_begin == q_end || d_begin == d_end) return MC2_OK;
	int rc;
	u64 cap = max_out ? max_out : 1;
	rc = ensure(x->d[B_OUTQ], cap * 8, false); if (rc) return rc;
	rc = ensure(x->d[B_OUTD], cap * 8, false); if (rc) return rc;
	rc = ensure(x->d[B_OUTS], cap * 8, false); if (rc) return rc;
	u64 total = 0;
	rc = run_sweep(ctx, dm, identity, min_identity, set_q, q_begin, q_end, set_d, d_begin, d_end, upper_only, cutoff, max_out,
		       (u64 *)x->d[B_OUTQ].p, (u64 *)x->d[B_OUTD].p, (double *)x->d[B_OUTS].p, &total, n_scored);
	if (rc != MC2_OK) return rc;
	cudaStream_t st = ctx->stream;
	*n_out = total;
	u64 got = total < max_out ? total : max_out;
	if (got) {
		if (out_q) MC2_CUDA(cudaMemcpyAsync(out_q, x->d[B_OUTQ].p, got * 8, cudaMemcpyDeviceToHost, st));
		if (out_d) MC2_CUDA(cudaMemcpyAsync(out_d, x->d[B_OUTD].p, got * 8, cudaMemcpyDeviceToHost, st));
		if (out_score) MC2_CUDA(cudaMemcpyAsync(out_score, x->d[B_OUTS].p, got * 8, cudaMemcpyDeviceToHost, st));
		MC2_CUDA(cudaStreamSynchronize(st));
	}
	return check_err(ctx);
}

int mc2_all_pairs(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *set_q, uint64_t q_begin, uint64_t q_end,
		  const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end, int32_t upper_only, double cutoff,
		  uint64_t max_out, uint64_t *out_q, uint64_t *out_d, double *out_score, uint64_t *n_out,
		  uint64_t *n_scored)
{
	MC2_REQUIRE(ctx && model && set_q && set_d && n_out, "mc2_all_pairs: NULL argument");
	return sweep_pairs("mc2_all_pairs", ctx, model->dm, 0, 0.0, set_q, q_begin, q_end, set_d, d_begin, d_end, upper_only, cutoff,
			   max_out, out_q, out_d, out_score, n_out, n_scored);
}

int mc2_identity_pairs(mc2_ctx *ctx, const mc2_model *model, double min_identity, const mc2_hset *set_q, uint64_t q_begin,
		       uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end, int32_t upper_only, double cutoff,
		       uint64_t max_out, uint64_t *out_q, uint64_t *out_d, double *out_identity, uint64_t *n_out, uint64_t *n_scored)
{
	MC2_REQUIRE(ctx && model && set_q && set_d && n_out, "mc2_identity_pairs: NULL argument");
	MC2_REQUIRE(!std::isnan(min_identity), "mc2_identity_pairs: min_identity is NaN");
	const DevModel dm = identity_model(model, min_identity);
	return sweep_pairs("mc2_identity_pairs", ctx, dm, 1, min_identity, set_q, q_begin, q_end, set_d, d_begin, d_end, upper_only,
			   cutoff, max_out, out_q, out_d, out_identity, n_out, n_scored);
}

/* ---- the other strand ------------------------------------------------------------------------- */
static int reverse_complement_set(mc2_ctx *ctx, const mc2_hset *src, mc2_hset **out)
{
	mc2_hset *h = nullptr;
	int rc = alloc_hset(ctx, src->n, src->k, src->eb, &h);
	if (rc != MC2_OK) return rc;
	const u64 n = src->n;
	cudaStream_t st = ctx->stream;
	cudaError_t e = cudaSuccess;
	if (n) {
		// everything but the bins and the k = 1 table depends on the multiset of counts only, which the permutation keeps
		e = cudaMemcpyAsync(h->mag, src->mag, n * 8, cudaMemcpyDeviceToDevice, st);
		if (e == cudaSuccess) e = cudaMemcpyAsync(h->len, src->len, n * 8, cudaMemcpyDeviceToDevice, st);
		if (e == cudaSuccess) e = cudaMemcpyAsync(h->sum, src->sum, n * 8, cudaMemcpyDeviceToDevice, st);
		if (e == cudaSuccess) e = cudaMemcpyAsync(h->sumsq, src->sumsq, n * 8, cudaMemcpyDeviceToDevice, st);
		if (e == cudaSuccess) e = cudaMemcpyAsync(h->stddev, src->stddev, n * 8, cudaMemcpyDeviceToDevice, st);
		if (e == cudaSuccess) e = cudaMemcpyAsync(h->maxc, src->maxc, n * 4, cudaMemcpyDeviceToDevice, st);
		// the overflowing-segment count depends on the order of the segments: reported as for a set built from histograms
		if (e == cudaSuccess) e = cudaMemsetAsync(h->novf, 0, n * 4, st);
	}
	if (e != cudaSuccess) {
		mc2_hset_free(h);
		return cuda_fail(e, "reverse complement side-band copies", __FILE__, __LINE__);
	}
	rc = launch_revcomp(ctx, src, h);
	if (rc == MC2_OK) {
		e = cudaStreamSynchronize(st);
		if (e != cudaSuccess) rc = cuda_fail(e, "reverse complement", __FILE__, __LINE__);
	}
	if (rc != MC2_OK) {
		mc2_hset_free(h);
		return rc;
	}
	h->max_sum = src->max_sum;
	h->max_count = src->max_count;
	h->counted = src->counted;
	*out = h;
	return MC2_OK;
}

int mc2_hset_reverse_complement(mc2_ctx *ctx, const mc2_hset *src, mc2_hset **out)
{
	MC2_REQUIRE(ctx && src && out, "mc2_hset_reverse_complement: NULL argument");
	*out = nullptr;
	MC2_CUDA(cudaSetDevice(ctx->device));
	return reverse_complement_set(ctx, src, out);
}

// pair-scoring launch over device-resident index lists (set_a row ia[j], set_b row ib[j]), scores into d_score: the launch and
// arguments mc2_score_pairs uses for host lists, so the scores are the same bits
static int score_device_lists(mc2_ctx *ctx, const DevModel &dm, const mc2_hset *A, const mc2_hset *B, const u64 *d_ia,
			      const u64 *d_ib, u64 n, double *d_score)
{
	PairArgs a;
	memset(&a, 0, sizeof a);
	a.binsA = A->bins;
	a.binsB = B->bins;
	a.sbA = Sideband{A->mag, A->sum, A->sumsq, A->len};
	a.sbB = Sideband{B->mag, B->sum, B->sumsq, B->len};
	a.N = A->N;
	a.eb = A->eb;
	a.n_pairs = n;
	a.ia = d_ia;
	a.ib = d_ib;
	a.err = ctx->d_err;
	a.max_sum = A->max_sum > B->max_sum ? A->max_sum : B->max_sum;
	if (ensure_lane_off(ctx, A) == MC2_OK && ensure_lane_off(ctx, B) == MC2_OK && A->lane_off_valid && B->lane_off_valid) {
		a.loffA = A->lane_off;
		a.loffB = B->lane_off;
	}
	a.score = d_score;
	return launch_pair_score(ctx, dm, a);
}

// Sweeps query rows [q_begin, q_end) block by block into a scratch of `scratch` pairs (sq, sd, ss), starting with blocks of
// `rows` rows.  With a second query set set_q2 (may be NULL; same row count as set_q), each block's rows of set_q2 are swept
// too, into a second scratch (sq2, sd2, ss2) of the same size.  A block whose survivors overflow either scratch is swept
// again in smaller blocks (one row always fits: scratch >= d_end - d_begin); blocks double while both sweeps' survivors fill
// less than a quarter of it.  on_block(qb, qe, nb, nb2) runs, in row order, for each block [qb, qe) whose nb (set_q) and nb2
// (set_q2; 0 without it) survivors all sit in the scratches: every row lies in exactly one such block.  *exact and *coarse
// gather the diagnostics of every sweep run (sum, and); *n_scored (may be NULL) sums set_q's in-window pairs of the blocks
// handed to on_block.
extern "C++" { // a template: C++ linkage inside this file's extern "C" region
template <typename F>
static int sweep_row_blocks(mc2_ctx *ctx, const DevModel &dm, double t, const mc2_hset *set_q, const mc2_hset *set_q2, u64 q_begin,
			    u64 q_end, const mc2_hset *set_d, u64 d_begin, u64 d_end, int32_t upper_only, double cutoff, u64 scratch,
			    u64 rows, u64 *sq, u64 *sd, double *ss, u64 *sq2, u64 *sd2, double *ss2, u64 *exact, int *coarse,
			    uint64_t *n_scored, F &&on_block)
{
	CtxExtra *x = extra(ctx);
	const u64 all_rows = q_end - q_begin;
	u64 qb = q_begin;
	while (qb < q_end) {
		const u64 qe = qb + std::min<u64>(rows, q_end - qb);
		u64 nb = 0, nb2 = 0;
		uint64_t ns = 0;
		int rc = run_sweep(ctx, dm, 1, t, set_q, qb, qe, set_d, d_begin, d_end, upper_only, cutoff, scratch, sq, sd, ss, &nb,
				   n_scored ? &ns : nullptr);
		if (rc == MC2_OK) rc = check_err(ctx);
		if (rc != MC2_OK) return rc;
		*exact += x->last_exact;
		*coarse &= x->last_coarse;
		if (set_q2 && nb <= scratch) { // the second sweep only when the first one's block stands
			rc = run_sweep(ctx, dm, 1, t, set_q2, qb, qe, set_d, d_begin, d_end, upper_only, cutoff, scratch, sq2, sd2, ss2,
				       &nb2, nullptr);
			if (rc == MC2_OK) rc = check_err(ctx);
			if (rc != MC2_OK) return rc;
			*exact += x->last_exact;
			*coarse &= x->last_coarse;
		}
		const u64 most = std::max<u64>(nb, nb2);
		if (most > scratch) { // more than a scratch holds: sweep a smaller block again
			const u64 span = qe - qb;
			rows = std::max<u64>(1, std::min<u64>(span / 2, (u64)((double)span * (double)(scratch / 2) / (double)most)));
			continue;
		}
		if (n_scored) *n_scored += ns;
		if ((rc = on_block(qb, qe, nb, nb2)) != MC2_OK) return rc;
		qb = qe;
		if (most < scratch / 4) {
			rows = std::min<u64>(rows * 2, all_rows);
		}
	}
	return MC2_OK;
}
}

// survivors of one reverse-strand block that the scratch holds; a query row has at most d_end - d_begin of them
static const u64 kStrandScratch = 1ull << 20;

// The device stages of mc2_identity_pairs_both_strands: its first max_out pairs (q, d, identity, strand) into (oq, od, os,
// ostr), *total = all of them; the query set's reverse complement is made and kept when missing.  The reverse strand is
// swept in blocks whose survivors fit `scratch` pairs (>= d_end - d_begin).  Sets the sweep diagnostics.
static int sweep_both_strands(mc2_ctx *ctx, const DevModel &dm, double t, const mc2_hset *set_q, u64 q_begin, u64 q_end,
			      const mc2_hset *set_d, u64 d_begin, u64 d_end, int32_t upper_only, double cutoff, u64 max_out, u64 *oq,
			      u64 *od, double *os, int8_t *ostr, u64 scratch, u64 *total, uint64_t *n_scored)
{
	CtxExtra *x = extra(ctx);
	int rc;
	const int bufs[] = {B_STR_Q, B_STR_D, B_STR_S, B_STR_F, B_STR_CNT};
	const u64 sizes[] = {scratch * 8, scratch * 8, scratch * 8, scratch * 8, 8};
	for (int i = 0; i < 5; i++) {
		if ((rc = ensure(x->d[bufs[i]], sizes[i], false)) != MC2_OK) return rc;
	}
	u64 *sq = (u64 *)x->d[B_STR_Q].p, *sd = (u64 *)x->d[B_STR_D].p;
	double *ss = (double *)x->d[B_STR_S].p, *sf = (double *)x->d[B_STR_F].p;
	u64 *cnt = (u64 *)x->d[B_STR_CNT].p;
	cudaStream_t st = ctx->stream;

	// forward strand: A = {id+ >= t}, the first max_out of them straight into the output
	u64 n_fwd = 0;
	rc = run_sweep(ctx, dm, 1, t, set_q, q_begin, q_end, set_d, d_begin, d_end, upper_only, cutoff, max_out, oq, od, os, &n_fwd, n_scored);
	if (rc == MC2_OK) rc = check_err(ctx);
	if (rc != MC2_OK) return rc;
	u64 exact = x->last_exact;
	int coarse = x->last_coarse;

	// the reverse-complement rows keep the query indices, so upper_only and the length window mean the same on both strands
	if (!set_q->rc) {
		mc2_hset *r = nullptr;
		if ((rc = reverse_complement_set(ctx, set_q, &r)) != MC2_OK) return rc;
		const_cast<mc2_hset *>(set_q)->rc = r;
	}
	const mc2_hset *rcq = set_q->rc;

	// id- of the returned forward survivors: the strand and identity they report
	const u64 got_fwd = std::min<u64>(n_fwd, max_out);
	for (u64 i = 0; i < got_fwd; i += scratch) {
		const u64 m = std::min<u64>(scratch, got_fwd - i);
		rc = score_device_lists(ctx, dm, set_d, rcq, od + i, oq + i, m, sf);
		if (rc == MC2_OK) rc = launch_strand_pick(ctx, os + i, sf, ostr + i, m);
		if (rc != MC2_OK) return rc;
	}
	MC2_CUDA(cudaMemcpyAsync(cnt, &n_fwd, 8, cudaMemcpyHostToDevice, st));
	rc = fetch_err(ctx);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaStreamSynchronize(st));
	if ((rc = check_err(ctx)) != MC2_OK) return rc;

	// Reverse strand: B = {id- >= t}, query-row block by block into the scratch; B \ A = the pairs of B with id+ < t.  For
	// t <= 0 every in-window pair is in A and B adds nothing.
	if (t > 0) {
		// first block: sized from the forward survivor count (the other strand of random reads has about as many), with
		// half the scratch to spare for rows denser than average (the early rows of an upper triangle)
		const u64 all_rows = q_end - q_begin;
		const u64 rows = std::max<u64>(1, std::min<u64>(all_rows, (u64)((double)all_rows * (double)(scratch / 2) / (double)std::max<u64>(n_fwd, 1))));
		rc = sweep_row_blocks(ctx, dm, t, rcq, nullptr, q_begin, q_end, set_d, d_begin, d_end, upper_only, cutoff, scratch, rows,
				      sq, sd, ss, nullptr, nullptr, nullptr, &exact, &coarse, nullptr, [&](u64, u64, u64 nb, u64) -> int {
			if (nb == 0) return MC2_OK;
			int r = score_device_lists(ctx, dm, set_d, set_q, sd, sq, nb, sf);
			if (r == MC2_OK) r = launch_strand_append(ctx, sq, sd, ss, sf, nb, t, cnt, max_out, oq, od, os, ostr);
			if (r == MC2_OK) r = fetch_err(ctx);
			if (r != MC2_OK) return r;
			MC2_CUDA(cudaStreamSynchronize(st));
			return check_err(ctx);
		});
		if (rc != MC2_OK) return rc;
	}
	MC2_CUDA(cudaMemcpyAsync(ctx->h_slot, cnt, 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	*total = ((u64 *)ctx->h_slot)[0];
	x->last_exact = exact;
	x->last_inline = x->sum_inline;
	x->last_coarse = coarse;
	return MC2_OK;
}

int mc2_identity_pairs_both_strands(mc2_ctx *ctx, const mc2_model *model, double min_identity, const mc2_hset *set_q,
				    uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end,
				    int32_t upper_only, double cutoff, uint64_t max_out, uint64_t *out_q, uint64_t *out_d,
				    double *out_identity, int8_t *out_strand, uint64_t *n_out, uint64_t *n_scored)
{
	const std::string w("mc2_identity_pairs_both_strands");
	MC2_REQUIRE(ctx && model && set_q && set_d && n_out, w + ": NULL argument");
	MC2_REQUIRE(!std::isnan(min_identity), w + ": min_identity is NaN");
	MC2_REQUIRE(q_begin <= q_end && q_end <= set_q->n && d_begin <= d_end && d_end <= set_d->n, w + ": row range out of bounds");
	MC2_REQUIRE(set_q->k == set_d->k && set_q->eb == set_d->eb, w + ": the two sets differ in k or histogram width");
	MC2_REQUIRE(cutoff > 0, w + ": cutoff must be > 0");
	MC2_REQUIRE((q_end - q_begin) * ((d_end - d_begin + 31) / 32) < (1ULL << 32),
		    w + ": more than 2^32 (query row, 32-column block) groups in one call; split the query range");
	MC2_REQUIRE(model->dm.regression != 0, w + ": needs a regression model");
	MC2_CUDA(cudaSetDevice(ctx->device));
	*n_out = 0;
	if (n_scored) *n_scored = 0;
	CtxExtra *x = extra(ctx);
	x->last_exact = 0;
	x->last_coarse = 0;
	x->last_inline = x->sum_inline = 0;
	if (q_begin == q_end || d_begin == d_end) return MC2_OK;
	const double t = min_identity;
	const DevModel dm = identity_model(model, t);
	const u64 cap = max_out ? max_out : 1;
	int rc;
	const int bufs[] = {B_STR_OQ, B_STR_OD, B_STR_OS, B_STR_OSTR};
	const u64 sizes[] = {cap * 8, cap * 8, cap * 8, cap};
	for (int i = 0; i < 4; i++) {
		if ((rc = ensure(x->d[bufs[i]], sizes[i], false)) != MC2_OK) return rc;
	}
	u64 *oq = (u64 *)x->d[B_STR_OQ].p, *od = (u64 *)x->d[B_STR_OD].p;
	double *os = (double *)x->d[B_STR_OS].p;
	int8_t *ostr = (int8_t *)x->d[B_STR_OSTR].p;
	cudaStream_t st = ctx->stream;
	u64 total = 0;
	rc = sweep_both_strands(ctx, dm, t, set_q, q_begin, q_end, set_d, d_begin, d_end, upper_only, cutoff, max_out, oq, od, os, ostr,
				std::max<u64>(d_end - d_begin, kStrandScratch), &total, n_scored);
	if (rc != MC2_OK) return rc;
	*n_out = total;
	const u64 got = std::min<u64>(total, max_out);
	if (got) {
		if (out_q) MC2_CUDA(cudaMemcpyAsync(out_q, oq, got * 8, cudaMemcpyDeviceToHost, st));
		if (out_d) MC2_CUDA(cudaMemcpyAsync(out_d, od, got * 8, cudaMemcpyDeviceToHost, st));
		if (out_identity) MC2_CUDA(cudaMemcpyAsync(out_identity, os, got * 8, cudaMemcpyDeviceToHost, st));
		if (out_strand) MC2_CUDA(cudaMemcpyAsync(out_strand, ostr, got, cudaMemcpyDeviceToHost, st));
		MC2_CUDA(cudaStreamSynchronize(st));
	}
	return MC2_OK;
}

// One block of both strands' survivors: F = (sq, sd, ss)[0..nb) and R = (rq, rd, rs)[0..nb2) (R empty for t <= 0), sx the
// other strand's identity of one of them at a time.
struct StrandBlock {
	const u64 *sq, *sd;
	double *ss;
	int8_t *sstr;
	u64 nb;
	const u64 *rq, *rd;
	const double *rs;
	u64 nb2;
	double *sx;
};

// The strand merge and bucketing of one block on both strands (mc2_identity_topk_both_strands, mc2_identity_greedy_clusters):
// F keeps max(id+, id-) with its strand (a tie stays forward), R adds the pairs the forward sweep rejected, !(id+ >= t) on
// the same bits, on strand 1.  A (q, d) pair is then in at most one of the two, with the bits and strand
// mc2_identity_pairs_both_strands reports.  Both lists go into `rows` buckets (identity bid, row bd, strand bstr) at the
// exclusive scan off of their counts: keyed by query q - base with bd = d, or with by_d by database row d - base with bd = q.
static int bucket_both_strands(mc2_ctx *ctx, const DevModel &dm, const mc2_hset *set_q, const mc2_hset *rcq, const mc2_hset *set_d,
			       double t, const StrandBlock &b, bool by_d, u64 base, u64 rows, int exclude_self, u32 *cnt, u64 *off,
			       double *bid, u64 *bd, int8_t *bstr)
{
	cudaStream_t st = ctx->stream;
	int r = score_device_lists(ctx, dm, set_d, rcq, b.sd, b.sq, b.nb, b.sx);
	if (r == MC2_OK) r = launch_strand_pick(ctx, b.ss, b.sx, b.sstr, b.nb);
	if (r != MC2_OK) return r;
	MC2_CUDA(cudaMemsetAsync(cnt, 0, rows * 4, st));
	r = launch_topk_count_strand(ctx, b.sq, b.sd, nullptr, t, b.nb, base, exclude_self, by_d, cnt);
	if (r == MC2_OK) r = score_device_lists(ctx, dm, set_d, set_q, b.rd, b.rq, b.nb2, b.sx); // id+ of R, after F's pick used sx
	if (r == MC2_OK) r = launch_topk_count_strand(ctx, b.rq, b.rd, b.sx, t, b.nb2, base, exclude_self, by_d, cnt);
	if (r == MC2_OK) r = launch_seg_scan(ctx, cnt, rows, off);
	if (r != MC2_OK) return r;
	MC2_CUDA(cudaMemsetAsync(cnt, 0, rows * 4, st)); // now the scatter's cursors
	r = launch_topk_scatter_strand(ctx, b.sq, b.sd, b.ss, b.sstr, nullptr, t, b.nb, base, exclude_self, by_d, off, cnt, bid, bd, bstr);
	if (r == MC2_OK) r = launch_topk_scatter_strand(ctx, b.rq, b.rd, b.rs, nullptr, b.sx, t, b.nb2, base, exclude_self, by_d, off, cnt,
							bid, bd, bstr);
	return r;
}

/* ---- top-K identity search ---------------------------------------------------------------------- */
// survivors of one block of query rows that the scratch holds; a query row has at most d_end - d_begin of them
static const u64 kTopkScratch = 1ull << 22;
static const uint32_t kTopkMaxK = 1024;

// the argument checks of both top-K entry points (`w` names the caller in error messages)
static int topk_check(const std::string &w, const mc2_model *model, double min_identity, uint32_t k_best, const mc2_hset *set_q,
		      uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end,
		      int32_t exclude_self, double cutoff)
{
	MC2_REQUIRE(!std::isnan(min_identity), w + ": min_identity is NaN");
	MC2_REQUIRE(k_best >= 1 && k_best <= kTopkMaxK, w + ": k_best must be in 1..1024");
	MC2_REQUIRE(q_begin <= q_end && q_end <= set_q->n && d_begin <= d_end && d_end <= set_d->n, w + ": row range out of bounds");
	MC2_REQUIRE(set_q->k == set_d->k && set_q->eb == set_d->eb, w + ": the two sets differ in k or histogram width");
	MC2_REQUIRE(cutoff > 0, w + ": cutoff must be > 0");
	MC2_REQUIRE((q_end - q_begin) * ((d_end - d_begin + 31) / 32) < (1ULL << 32),
		    w + ": more than 2^32 (query row, 32-column block) groups in one call; split the query range");
	MC2_REQUIRE(model->dm.regression != 0, w + ": needs a regression model");
	MC2_REQUIRE(!exclude_self || set_q == set_d, w + ": exclude_self needs set_q == set_d");
	MC2_REQUIRE(q_end - q_begin <= UINT64_MAX / 16 / k_best, w + ": (q_end - q_begin) x k_best overflows");
	MC2_REQUIRE(d_end - d_begin < (1ULL << 32), w + ": the database range must hold fewer than 2^32 rows");
	return MC2_OK;
}

int mc2_identity_topk(mc2_ctx *ctx, const mc2_model *model, double min_identity, uint32_t k_best, const mc2_hset *set_q,
		      uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin, uint64_t d_end, int32_t upper_only,
		      int32_t exclude_self, double cutoff, uint64_t *out_d, double *out_identity, uint32_t *out_count,
		      uint64_t *out_n_hits, uint64_t *n_scored)
{
	const std::string w("mc2_identity_topk");
	MC2_REQUIRE(ctx && model && set_q && set_d && out_d && out_identity && out_count, w + ": NULL argument");
	int rc = topk_check(w, model, min_identity, k_best, set_q, q_begin, q_end, set_d, d_begin, d_end, exclude_self, cutoff);
	if (rc != MC2_OK) return rc;
	const u64 nq = q_end - q_begin, K = k_best;
	MC2_CUDA(cudaSetDevice(ctx->device));
	if (n_scored) *n_scored = 0;
	CtxExtra *x = extra(ctx);
	x->last_exact = 0;
	x->last_coarse = 0;
	x->last_inline = x->sum_inline = 0;
	if (nq == 0) return MC2_OK;
	if (d_begin == d_end) {
		std::fill(out_d, out_d + nq * K, UINT64_MAX);
		std::fill(out_identity, out_identity + nq * K, -1.0);
		std::fill(out_count, out_count + nq, 0u);
		if (out_n_hits) std::fill(out_n_hits, out_n_hits + nq, (uint64_t)0);
		return MC2_OK;
	}
	const DevModel dm = identity_model(model, min_identity);
	const u64 scratch = std::max<u64>(d_end - d_begin, kTopkScratch);
	const int bufs[] = {B_TOPK_Q, B_TOPK_D, B_TOPK_S, B_TOPK_BID, B_TOPK_BD, B_TOPK_CNT, B_TOPK_OFF, B_TOPK_OD, B_TOPK_OID, B_TOPK_OCNT, B_TOPK_OHITS};
	const u64 sizes[] = {scratch * 8, scratch * 8, scratch * 8, scratch * 8, scratch * 8, nq * 4, (nq + 1) * 8, nq * K * 8, nq * K * 8, nq * 4, nq * 8};
	for (int i = 0; i < 11; i++) {
		if ((rc = ensure(x->d[bufs[i]], sizes[i], false)) != MC2_OK) return rc;
	}
	u64 *sq = (u64 *)x->d[B_TOPK_Q].p, *sd = (u64 *)x->d[B_TOPK_D].p, *bd = (u64 *)x->d[B_TOPK_BD].p, *off = (u64 *)x->d[B_TOPK_OFF].p;
	double *ss = (double *)x->d[B_TOPK_S].p, *bid = (double *)x->d[B_TOPK_BID].p;
	u32 *cnt = (u32 *)x->d[B_TOPK_CNT].p;
	u64 *od = (u64 *)x->d[B_TOPK_OD].p, *ohits = (u64 *)x->d[B_TOPK_OHITS].p;
	double *oid = (double *)x->d[B_TOPK_OID].p;
	u32 *ocnt = (u32 *)x->d[B_TOPK_OCNT].p;
	cudaStream_t st = ctx->stream;

	// Every query's hits land in exactly one block, so its top K is selected once from all of them.  The first block is the
	// whole range: when the survivors fit, the call is one sweep.
	u64 exact = 0;
	uint64_t ns = 0;
	int coarse = 1;
	rc = sweep_row_blocks(ctx, dm, min_identity, set_q, nullptr, q_begin, q_end, set_d, d_begin, d_end, upper_only, cutoff, scratch,
			      nq, sq, sd, ss, nullptr, nullptr, nullptr, &exact, &coarse, &ns, [&](u64 qb, u64 qe, u64 nb, u64) -> int {
		const u64 rows = qe - qb, r0 = qb - q_begin;
		MC2_CUDA(cudaMemsetAsync(cnt, 0, rows * 4, st));
		int r = launch_topk_count(ctx, sq, sd, nb, qb, exclude_self, false, cnt);
		if (r == MC2_OK) r = launch_seg_scan(ctx, cnt, rows, off);
		if (r != MC2_OK) return r;
		MC2_CUDA(cudaMemsetAsync(cnt, 0, rows * 4, st)); // now the scatter's cursors
		r = launch_topk_scatter(ctx, sq, sd, ss, nb, qb, exclude_self, false, off, cnt, bid, bd);
		if (r == MC2_OK) r = launch_topk_select(ctx, off, bid, bd, rows, k_best, d_begin, od + r0 * K, oid + r0 * K, ocnt + r0, ohits + r0);
		return r;
	});
	if (rc != MC2_OK) return rc;
	x->last_exact = exact;
	x->last_inline = x->sum_inline;
	x->last_coarse = coarse;
	if (n_scored) *n_scored = ns;
	MC2_CUDA(cudaMemcpyAsync(out_d, od, nq * K * 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaMemcpyAsync(out_identity, oid, nq * K * 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaMemcpyAsync(out_count, ocnt, nq * 4, cudaMemcpyDeviceToHost, st));
	if (out_n_hits) MC2_CUDA(cudaMemcpyAsync(out_n_hits, ohits, nq * 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	return MC2_OK;
}

int mc2_identity_topk_both_strands(mc2_ctx *ctx, const mc2_model *model, double min_identity, uint32_t k_best,
				   const mc2_hset *set_q, uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d, uint64_t d_begin,
				   uint64_t d_end, int32_t upper_only, int32_t exclude_self, double cutoff, uint64_t *out_d,
				   double *out_identity, int8_t *out_strand, uint32_t *out_count, uint64_t *out_n_hits,
				   uint64_t *n_scored)
{
	const std::string w("mc2_identity_topk_both_strands");
	MC2_REQUIRE(ctx && model && set_q && set_d && out_d && out_identity && out_count, w + ": NULL argument");
	int rc = topk_check(w, model, min_identity, k_best, set_q, q_begin, q_end, set_d, d_begin, d_end, exclude_self, cutoff);
	if (rc != MC2_OK) return rc;
	const u64 nq = q_end - q_begin, K = k_best;
	MC2_CUDA(cudaSetDevice(ctx->device));
	if (n_scored) *n_scored = 0;
	CtxExtra *x = extra(ctx);
	x->last_exact = 0;
	x->last_coarse = 0;
	x->last_inline = x->sum_inline = 0;
	if (nq == 0) return MC2_OK;
	if (d_begin == d_end) {
		std::fill(out_d, out_d + nq * K, UINT64_MAX);
		std::fill(out_identity, out_identity + nq * K, -1.0);
		if (out_strand) std::fill(out_strand, out_strand + nq * K, (int8_t)-1);
		std::fill(out_count, out_count + nq, 0u);
		if (out_n_hits) std::fill(out_n_hits, out_n_hits + nq, (uint64_t)0);
		return MC2_OK;
	}
	const double t = min_identity;
	const DevModel dm = identity_model(model, t);
	const u64 scratch = std::max<u64>(d_end - d_begin, kTopkScratch);
	// per block: forward survivors F (q, d, identity, strand), reverse survivors R (q, d, identity; t > 0 only), the other
	// strand's identity of one of them at a time, and buckets for both (identity, d, strand)
	const bool rev = t > 0;
	const int bufs[] = {B_TOPK_Q, B_TOPK_D, B_TOPK_S, B_TK2_SSTR, B_TK2_X, B_TOPK_BID, B_TOPK_BD, B_TK2_BSTR, B_TOPK_CNT,
			    B_TOPK_OFF, B_TOPK_OD, B_TOPK_OID, B_TK2_OSTR, B_TOPK_OCNT, B_TOPK_OHITS, B_TK2_RQ, B_TK2_RD, B_TK2_RS};
	const u64 sizes[] = {scratch * 8, scratch * 8, scratch * 8, scratch, scratch * 8, 2 * scratch * 8, 2 * scratch * 8, 2 * scratch,
			     nq * 4, (nq + 1) * 8, nq * K * 8, nq * K * 8, nq * K, nq * 4, nq * 8, scratch * 8, scratch * 8, scratch * 8};
	for (int i = 0; i < (rev ? 18 : 15); i++) {
		if ((rc = ensure(x->d[bufs[i]], sizes[i], false)) != MC2_OK) return rc;
	}
	u64 *sq = (u64 *)x->d[B_TOPK_Q].p, *sd = (u64 *)x->d[B_TOPK_D].p, *bd = (u64 *)x->d[B_TOPK_BD].p, *off = (u64 *)x->d[B_TOPK_OFF].p;
	double *ss = (double *)x->d[B_TOPK_S].p, *sx = (double *)x->d[B_TK2_X].p, *bid = (double *)x->d[B_TOPK_BID].p;
	int8_t *sstr = (int8_t *)x->d[B_TK2_SSTR].p, *bstr = (int8_t *)x->d[B_TK2_BSTR].p, *ostr = (int8_t *)x->d[B_TK2_OSTR].p;
	u64 *rq = rev ? (u64 *)x->d[B_TK2_RQ].p : nullptr, *rd = rev ? (u64 *)x->d[B_TK2_RD].p : nullptr;
	double *rs = rev ? (double *)x->d[B_TK2_RS].p : nullptr;
	u32 *cnt = (u32 *)x->d[B_TOPK_CNT].p;
	u64 *od = (u64 *)x->d[B_TOPK_OD].p, *ohits = (u64 *)x->d[B_TOPK_OHITS].p;
	double *oid = (double *)x->d[B_TOPK_OID].p;
	u32 *ocnt = (u32 *)x->d[B_TOPK_OCNT].p;
	cudaStream_t st = ctx->stream;

	// the reverse-complement rows keep the query indices, so upper_only and the length window mean the same on both strands
	if (!set_q->rc) {
		mc2_hset *r = nullptr;
		if ((rc = reverse_complement_set(ctx, set_q, &r)) != MC2_OK) return rc;
		const_cast<mc2_hset *>(set_q)->rc = r;
	}
	const mc2_hset *rcq = set_q->rc;

	// Both strands of a block's rows are swept before the block is ranked, so each query's hits on both strands are selected
	// at once.  F = {id+ >= t} keeps max(id+, id-) with its strand (a tie stays forward); R = {id- >= t} adds the pairs the
	// forward sweep rejected, !(id+ >= t) on the same bits, on the reverse strand.  For t <= 0 every in-window pair is in F
	// and the reverse sweep is skipped.  A (q, d) pair is in at most one of the two, so the order stays total.
	u64 exact = 0;
	uint64_t ns = 0;
	int coarse = 1;
	rc = sweep_row_blocks(ctx, dm, t, set_q, rev ? rcq : nullptr, q_begin, q_end, set_d, d_begin, d_end, upper_only, cutoff, scratch,
			      nq, sq, sd, ss, rq, rd, rs, &exact, &coarse, &ns, [&](u64 qb, u64 qe, u64 nb, u64 nb2) -> int {
		const u64 rows = qe - qb, r0 = qb - q_begin;
		int r = reset_err(ctx);
		if (r == MC2_OK) r = bucket_both_strands(ctx, dm, set_q, rcq, set_d, t, StrandBlock{sq, sd, ss, sstr, nb, rq, rd, rs, nb2, sx},
							 false, qb, rows, exclude_self, cnt, off, bid, bd, bstr);
		if (r == MC2_OK) r = launch_topk_select_strand(ctx, off, bid, bd, bstr, rows, k_best, d_begin, od + r0 * K, oid + r0 * K,
								ostr + r0 * K, ocnt + r0, ohits + r0);
		if (r == MC2_OK) r = fetch_err(ctx);
		if (r != MC2_OK) return r;
		MC2_CUDA(cudaStreamSynchronize(st));
		return check_err(ctx);
	});
	if (rc != MC2_OK) return rc;
	x->last_exact = exact;
	x->last_inline = x->sum_inline;
	x->last_coarse = coarse;
	if (n_scored) *n_scored = ns;
	MC2_CUDA(cudaMemcpyAsync(out_d, od, nq * K * 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaMemcpyAsync(out_identity, oid, nq * K * 8, cudaMemcpyDeviceToHost, st));
	if (out_strand) MC2_CUDA(cudaMemcpyAsync(out_strand, ostr, nq * K, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaMemcpyAsync(out_count, ocnt, nq * 4, cudaMemcpyDeviceToHost, st));
	if (out_n_hits) MC2_CUDA(cudaMemcpyAsync(out_n_hits, ohits, nq * 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	return MC2_OK;
}

/* ---- identity clustering: connected components of the identity graph ------------------------------ */
// survivors of one block of query rows that each strand's scratch holds: cfg3's upper triangle at t = 0.5 (12.4 M forward
// hits) fits one block
static const u64 kComponentsScratch = 1ull << 24;

// parent array and label buffer (labels, then the component count) of a union-find over n rows, parents initialised
static int components_begin(mc2_ctx *ctx, u64 n, u32 **parent, u64 **label)
{
	CtxExtra *x = extra(ctx);
	int rc = ensure(x->d[B_CC_PARENT], n * 4, false);
	if (rc == MC2_OK) rc = ensure(x->d[B_CC_LABEL], (n + 1) * 8, false);
	if (rc != MC2_OK) return rc;
	*parent = (u32 *)x->d[B_CC_PARENT].p;
	*label = (u64 *)x->d[B_CC_LABEL].p;
	return launch_cc_init(ctx, *parent, n);
}

// flatten, then the labels and the component count to the host
static int components_end(mc2_ctx *ctx, u32 *parent, u64 *label, u64 n, u64 begin, uint64_t *out_label, uint64_t *n_components)
{
	int rc = launch_cc_flatten(ctx, parent, n, begin, label, label + n);
	if (rc != MC2_OK) return rc;
	cudaStream_t st = ctx->stream;
	MC2_CUDA(cudaMemcpyAsync(out_label, label, n * 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaMemcpyAsync(ctx->h_slot, label + n, 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	*n_components = ((u64 *)ctx->h_slot)[0];
	return MC2_OK;
}

int mc2_identity_components(mc2_ctx *ctx, const mc2_model *model, double min_identity, int32_t both_strands, const mc2_hset *set,
			    uint64_t q_begin, uint64_t q_end, uint64_t begin, uint64_t end, double cutoff, uint64_t *out_label,
			    uint64_t *n_components, uint64_t *n_scored)
{
	const std::string w("mc2_identity_components");
	MC2_REQUIRE(ctx && model && set && out_label && n_components, w + ": NULL argument");
	MC2_REQUIRE(!std::isnan(min_identity), w + ": min_identity is NaN");
	MC2_REQUIRE(begin <= q_begin && q_begin <= q_end && q_end <= end && end <= set->n, w + ": row range out of bounds");
	MC2_REQUIRE(end - begin < (1ULL << 32), w + ": the row range must hold fewer than 2^32 rows");
	MC2_REQUIRE(cutoff > 0, w + ": cutoff must be > 0");
	MC2_REQUIRE((q_end - q_begin) * ((end - begin + 31) / 32) < (1ULL << 32),
		    w + ": more than 2^32 (query row, 32-column block) groups in one call; split the query range");
	MC2_REQUIRE(model->dm.regression != 0, w + ": needs a regression model");
	MC2_CUDA(cudaSetDevice(ctx->device));
	*n_components = 0;
	if (n_scored) *n_scored = 0;
	CtxExtra *x = extra(ctx);
	x->last_exact = 0;
	x->last_coarse = 0;
	x->last_inline = x->sum_inline = 0;
	const u64 n = end - begin;
	if (n == 0) return MC2_OK;
	u32 *parent;
	u64 *label;
	int rc = components_begin(ctx, n, &parent, &label);
	if (rc != MC2_OK) return rc;
	if (q_begin < q_end) {
		const double t = min_identity;
		const DevModel dm = identity_model(model, t);
		// an edge on either strand is an edge: no strand merge, no rescoring.  For t <= 0 every in-window pair is already a
		// forward edge and the reverse sweep is skipped.
		const bool rev = both_strands && t > 0;
		const u64 scratch = std::max<u64>(n, kComponentsScratch);
		const int bufs[] = {B_TOPK_Q, B_TOPK_D, B_TOPK_S, B_TK2_RQ, B_TK2_RD, B_TK2_RS};
		for (int i = 0; i < (rev ? 6 : 3); i++) {
			if ((rc = ensure(x->d[bufs[i]], scratch * 8, false)) != MC2_OK) return rc;
		}
		u64 *sq = (u64 *)x->d[B_TOPK_Q].p, *sd = (u64 *)x->d[B_TOPK_D].p;
		double *ss = (double *)x->d[B_TOPK_S].p;
		u64 *rq = rev ? (u64 *)x->d[B_TK2_RQ].p : nullptr, *rd = rev ? (u64 *)x->d[B_TK2_RD].p : nullptr;
		double *rs = rev ? (double *)x->d[B_TK2_RS].p : nullptr;
		const mc2_hset *rcq = nullptr;
		if (rev) {
			// the reverse-complement rows keep the query indices, so upper_only and the length window mean the same on
			// both strands
			if (!set->rc) {
				mc2_hset *r = nullptr;
				if ((rc = reverse_complement_set(ctx, set, &r)) != MC2_OK) return rc;
				const_cast<mc2_hset *>(set)->rc = r;
			}
			rcq = set->rc;
		}
		// the parent array is the only state kept between blocks: each block's survivors are joined as soon as it is swept
		u64 exact = 0;
		uint64_t ns = 0;
		int coarse = 1;
		rc = sweep_row_blocks(ctx, dm, t, set, rcq, q_begin, q_end, set, begin, end, 1, cutoff, scratch, q_end - q_begin, sq, sd,
				      ss, rq, rd, rs, &exact, &coarse, &ns, [&](u64, u64, u64 nb, u64 nb2) -> int {
			int r = launch_cc_hook_pairs(ctx, sq, sd, nb, begin, parent);
			if (r == MC2_OK) r = launch_cc_hook_pairs(ctx, rq, rd, nb2, begin, parent);
			return r;
		});
		if (rc != MC2_OK) return rc;
		x->last_exact = exact;
		x->last_inline = x->sum_inline;
		x->last_coarse = coarse;
		if (n_scored) *n_scored = ns;
	}
	return components_end(ctx, parent, label, n, begin, out_label, n_components);
}

int mc2_components_merge(mc2_ctx *ctx, uint64_t begin, uint64_t end, uint32_t n_parts, const uint64_t *labels, uint64_t *out_label,
			 uint64_t *n_components)
{
	const std::string w("mc2_components_merge");
	MC2_REQUIRE(ctx && out_label && n_components, w + ": NULL argument");
	MC2_REQUIRE(n_parts >= 1, w + ": n_parts must be >= 1");
	MC2_REQUIRE(begin <= end && end - begin < (1ULL << 32), w + ": the row range must hold fewer than 2^32 rows");
	const u64 n = end - begin, m = (u64)n_parts * n;
	MC2_REQUIRE(n == 0 || labels, w + ": NULL argument");
	MC2_REQUIRE(m <= UINT64_MAX / 8, w + ": n_parts x (end - begin) overflows");
	for (u64 i = 0; i < m; i++) {
		MC2_REQUIRE(labels[i] >= begin && labels[i] < end, w + ": a label outside [begin, end)");
	}
	MC2_CUDA(cudaSetDevice(ctx->device));
	*n_components = 0;
	if (n == 0) return MC2_OK;
	CtxExtra *x = extra(ctx);
	int rc = ensure(x->d[B_TOPK_Q], m * 8, false);
	if (rc != MC2_OK) return rc;
	u64 *d_labels = (u64 *)x->d[B_TOPK_Q].p;
	MC2_CUDA(cudaMemcpyAsync(d_labels, labels, m * 8, cudaMemcpyHostToDevice, ctx->stream));
	u32 *parent;
	u64 *label;
	if ((rc = components_begin(ctx, n, &parent, &label)) != MC2_OK) return rc;
	if ((rc = launch_cc_hook_labels(ctx, d_labels, n_parts, n, begin, parent)) != MC2_OK) return rc;
	return components_end(ctx, parent, label, n, begin, out_label, n_components);
}

/* ---- identity clustering: greedy representatives in row order ------------------------------------ */
// the argument checks of mc2_identity_greedy_clusters and mc2_greedy_begin (`w` names the caller in error messages)
static int greedy_check(const std::string &w, const mc2_model *model, double min_identity, const mc2_hset *set, uint64_t begin,
			uint64_t end, double cutoff)
{
	MC2_REQUIRE(!std::isnan(min_identity), w + ": min_identity is NaN");
	MC2_REQUIRE(begin <= end && end <= set->n, w + ": row range out of bounds");
	MC2_REQUIRE(end - begin < (1ULL << 32), w + ": the row range must hold fewer than 2^32 rows");
	MC2_REQUIRE(cutoff > 0, w + ": cutoff must be > 0");
	MC2_REQUIRE((end - begin) * ((end - begin + 31) / 32) < (1ULL << 32),
		    w + ": more than 2^32 (query row, 32-column block) groups in one call; split the row range");
	MC2_REQUIRE(model->dm.regression != 0, w + ": needs a regression model");
	return MC2_OK;
}

// The device state of a greedy clustering over rows [begin, end): the rows (GreedyRows and the resolve's three round flags,
// carved from 21 n + 16 bytes), and the buckets of one block (counts / cursors, offsets, identity, query row, strand).
struct GreedyBlock {
	GreedyRows g;
	u32 *remain, *cnt;
	u64 *off, *bd;
	double *bid;
	int8_t *bstr;
	u64 begin, end;
};

// per row: identity 8, status 4, cursor 4, rep 4 bytes, the three round flags after rep, then strand 1
static void greedy_rows(char *p, u64 n, GreedyBlock *b)
{
	b->g.id = (double *)p;
	b->g.status = (u32 *)(p + 8 * n);
	b->g.cursor = (u32 *)(p + 12 * n);
	b->g.rep = (u32 *)(p + 16 * n);
	b->remain = (u32 *)(p + 20 * n);
	b->g.str = (int8_t *)(p + 20 * n + 16);
}

// One block [qb, qe) of query rows, every row below qb final: bucket(rows) puts the block's edges into the buckets of their
// larger row - qb (rows = end - qb buckets); then one cooperative launch decides the block's rows and one more brings every
// later row's best in-edge from a representative up to date.
extern "C++" {
template <typename F>
static int greedy_block(mc2_ctx *ctx, const GreedyBlock &b, u64 qb, u64 qe, F &&bucket)
{
	int r = bucket(b.end - qb);
	if (r == MC2_OK) r = launch_greedy_resolve(ctx, b.off, b.bd, qb, qe - qb, b.begin, b.g, b.remain);
	if (r == MC2_OK) r = launch_greedy_assign(ctx, b.off, b.bid, b.bd, b.bstr, qb, b.end - qb, b.begin, b.g);
	return r;
}
}

// the outputs of a finished clustering over n rows from the rows' state, through d_out (17 n + 8 bytes: rep 8, identity 8,
// strand 1 per row; the representative count after the identities)
static int greedy_outputs(mc2_ctx *ctx, const GreedyRows &g, u64 n, u64 begin, char *d_out, uint64_t *out_rep, double *out_identity,
			  int8_t *out_strand, uint64_t *n_clusters)
{
	u64 *d_rep = (u64 *)d_out, *d_reps = (u64 *)(d_out + 16 * n);
	double *d_id = (double *)(d_out + 8 * n);
	int8_t *d_str = (int8_t *)(d_out + 16 * n + 8);
	cudaStream_t st = ctx->stream;
	int rc = launch_greedy_finish(ctx, g, n, begin, d_rep, d_id, d_str, d_reps);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaMemcpyAsync(out_rep, d_rep, n * 8, cudaMemcpyDeviceToHost, st));
	if (out_identity) MC2_CUDA(cudaMemcpyAsync(out_identity, d_id, n * 8, cudaMemcpyDeviceToHost, st));
	if (out_strand) MC2_CUDA(cudaMemcpyAsync(out_strand, d_str, n, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaMemcpyAsync(ctx->h_slot, d_reps, 8, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	*n_clusters = ((u64 *)ctx->h_slot)[0];
	return MC2_OK;
}

int mc2_identity_greedy_clusters(mc2_ctx *ctx, const mc2_model *model, double min_identity, int32_t both_strands, const mc2_hset *set,
				 uint64_t begin, uint64_t end, double cutoff, uint64_t *out_rep, double *out_identity, int8_t *out_strand,
				 uint64_t *n_clusters, uint64_t *n_scored)
{
	const std::string w("mc2_identity_greedy_clusters");
	MC2_REQUIRE(ctx && model && set && out_rep && n_clusters, w + ": NULL argument");
	int rc = greedy_check(w, model, min_identity, set, begin, end, cutoff);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaSetDevice(ctx->device));
	*n_clusters = 0;
	if (n_scored) *n_scored = 0;
	CtxExtra *x = extra(ctx);
	x->last_exact = 0;
	x->last_coarse = 0;
	x->last_inline = x->sum_inline = 0;
	const u64 n = end - begin;
	if (n == 0) return MC2_OK;
	const double t = min_identity;
	const DevModel dm = identity_model(model, t);
	// Both strands: every forward survivor's id- is scored for the strand merge, so the reverse-complement set is needed for
	// any t; for t <= 0 every in-window pair is already a forward edge and the reverse sweep is skipped.
	const bool both = both_strands != 0, rev = both && t > 0;
	const u64 scratch = std::max<u64>(n, kComponentsScratch), bucket = both ? 2 * scratch : scratch;
	// per row: the state kept across blocks, the outputs, bucket counts and offsets
	const int bufs[] = {B_GR_ROWS, B_GR_OUT, B_TOPK_CNT, B_TOPK_OFF, B_TOPK_Q, B_TOPK_D, B_TOPK_S, B_TOPK_BID, B_TOPK_BD,
			    B_TK2_SSTR, B_TK2_X, B_TK2_BSTR, B_TK2_RQ, B_TK2_RD, B_TK2_RS};
	const u64 sizes[] = {21 * n + 16, 17 * n + 8, n * 4, (n + 1) * 8, scratch * 8, scratch * 8, scratch * 8, bucket * 8, bucket * 8,
			     scratch, scratch * 8, bucket, scratch * 8, scratch * 8, scratch * 8};
	for (int i = 0; i < (rev ? 15 : both ? 12 : 9); i++) {
		if ((rc = ensure(x->d[bufs[i]], sizes[i], false)) != MC2_OK) return rc;
	}
	GreedyBlock gb;
	greedy_rows((char *)x->d[B_GR_ROWS].p, n, &gb);
	gb.cnt = (u32 *)x->d[B_TOPK_CNT].p;
	gb.off = (u64 *)x->d[B_TOPK_OFF].p;
	gb.bd = (u64 *)x->d[B_TOPK_BD].p;
	gb.bid = (double *)x->d[B_TOPK_BID].p;
	gb.bstr = both ? (int8_t *)x->d[B_TK2_BSTR].p : nullptr;
	gb.begin = begin;
	gb.end = end;
	u32 *cnt = gb.cnt;
	u64 *off = gb.off, *sq = (u64 *)x->d[B_TOPK_Q].p, *sd = (u64 *)x->d[B_TOPK_D].p, *bd = gb.bd;
	double *ss = (double *)x->d[B_TOPK_S].p, *bid = gb.bid;
	double *sx = both ? (double *)x->d[B_TK2_X].p : nullptr;
	int8_t *sstr = both ? (int8_t *)x->d[B_TK2_SSTR].p : nullptr, *bstr = gb.bstr;
	u64 *rq = rev ? (u64 *)x->d[B_TK2_RQ].p : nullptr, *rd = rev ? (u64 *)x->d[B_TK2_RD].p : nullptr;
	double *rs = rev ? (double *)x->d[B_TK2_RS].p : nullptr;
	cudaStream_t st = ctx->stream;
	if ((rc = launch_greedy_init(ctx, gb.g, n)) != MC2_OK) return rc;
	const mc2_hset *rcq = nullptr;
	if (both) {
		// the reverse-complement rows keep the query indices, so upper_only and the length window mean the same on both
		// strands
		if (!set->rc) {
			mc2_hset *r = nullptr;
			if ((rc = reverse_complement_set(ctx, set, &r)) != MC2_OK) return rc;
			const_cast<mc2_hset *>(set)->rc = r;
		}
		rcq = set->rc;
	}
	// Blocks arrive in row order and an edge with the block of its smaller row, so when [qb, qe) arrives every row below qb is
	// final.
	u64 exact = 0;
	uint64_t ns = 0;
	int coarse = 1;
	rc = sweep_row_blocks(ctx, dm, t, set, rev ? rcq : nullptr, begin, end, set, begin, end, 1, cutoff, scratch, n, sq, sd, ss, rq, rd,
			      rs, &exact, &coarse, &ns, [&](u64 qb, u64 qe, u64 nb, u64 nb2) -> int {
		int r = greedy_block(ctx, gb, qb, qe, [&](u64 rows) -> int {
			if (both) {
				int r2 = reset_err(ctx);
				if (r2 == MC2_OK) r2 = bucket_both_strands(ctx, dm, set, rcq, set, t, StrandBlock{sq, sd, ss, sstr, nb, rq, rd, rs, nb2, sx},
									   true, qb, rows, 0, cnt, off, bid, bd, bstr);
				return r2;
			}
			MC2_CUDA(cudaMemsetAsync(cnt, 0, rows * 4, st));
			int r2 = launch_topk_count(ctx, sq, sd, nb, qb, 0, true, cnt);
			if (r2 == MC2_OK) r2 = launch_seg_scan(ctx, cnt, rows, off);
			if (r2 != MC2_OK) return r2;
			MC2_CUDA(cudaMemsetAsync(cnt, 0, rows * 4, st)); // now the scatter's cursors
			return launch_topk_scatter(ctx, sq, sd, ss, nb, qb, 0, true, off, cnt, bid, bd);
		});
		if (r != MC2_OK || !both) return r;
		if ((r = fetch_err(ctx)) != MC2_OK) return r;
		MC2_CUDA(cudaStreamSynchronize(st));
		return check_err(ctx);
	});
	if (rc != MC2_OK) return rc;
	x->last_exact = exact;
	x->last_inline = x->sum_inline;
	x->last_coarse = coarse;
	if (n_scored) *n_scored = ns;
	return greedy_outputs(ctx, gb.g, n, begin, (char *)x->d[B_GR_OUT].p, out_rep, out_identity, out_strand, n_clusters);
}

} // extern "C"

// A staged greedy clustering (mc2_greedy_begin .. mc2_greedy_end): the rows' state, n_parts part slots of cap records (and
// strand bytes), buckets for n_parts * cap edges, and the parts' ranges and counts (3 words each, then the bad-record flag),
// all owned by the object so that other calls may run between its stages.
struct mc2_greedy {
	DevModel dm;
	double t, cutoff;
	bool both;
	const mc2_hset *set;
	u64 begin, end, next, cap;
	u32 n_parts;
	Buf rows, out, cnt, off, bid, bd, bstr, rec, str, part;
	GreedyBlock b;
};

extern "C" {

// the default part capacity: every part of a whole-range block of cfg3's shape at t = 0.5 (12.4 M forward edges) fits
static const u64 kGreedyPartEdges = 1ull << 24;

void mc2_greedy_free(mc2_greedy *g)
{
	if (!g) return;
	Buf *bufs[] = {&g->rows, &g->out, &g->cnt, &g->off, &g->bid, &g->bd, &g->bstr, &g->rec, &g->str, &g->part};
	for (Buf *b : bufs) release(*b);
	delete g;
}

int mc2_greedy_begin(mc2_ctx *ctx, const mc2_model *model, double min_identity, int32_t both_strands, const mc2_hset *set,
		     uint64_t begin, uint64_t end, double cutoff, uint32_t n_parts, uint64_t part_capacity, mc2_greedy **out)
{
	const std::string w("mc2_greedy_begin");
	MC2_REQUIRE(ctx && model && set && out, w + ": NULL argument");
	*out = nullptr;
	int rc = greedy_check(w, model, min_identity, set, begin, end, cutoff);
	if (rc != MC2_OK) return rc;
	MC2_REQUIRE(n_parts >= 1, w + ": n_parts must be >= 1");
	const u64 n = end - begin, P = n_parts;
	const u64 cap = part_capacity ? part_capacity : std::max<u64>(n, (kGreedyPartEdges + P - 1) / P);
	MC2_REQUIRE(cap >= n, w + ": part_capacity must be >= end - begin (one query row's edges)");
	MC2_REQUIRE(cap <= UINT64_MAX / 32 / P, w + ": n_parts x part_capacity overflows");
	MC2_CUDA(cudaSetDevice(ctx->device));
	mc2_greedy *g = new (std::nothrow) mc2_greedy();
	MC2_REQUIRE(g, w + ": out of host memory");
	g->dm = identity_model(model, min_identity);
	g->t = min_identity;
	g->cutoff = cutoff;
	g->both = both_strands != 0;
	g->set = set;
	g->begin = g->next = begin;
	g->end = end;
	g->cap = cap;
	g->n_parts = n_parts;
	const u64 edges = P * cap;
	Buf *bufs[] = {&g->rows, &g->out, &g->cnt, &g->off, &g->bid, &g->bd, &g->rec, &g->part, &g->bstr, &g->str};
	const u64 sizes[] = {21 * n + 16, 17 * n + 8, n * 4 + 4, (n + 1) * 8, edges * 8, edges * 8, edges * 16, P * 24 + 8, edges, edges};
	for (int i = 0; i < (g->both ? 10 : 8) && rc == MC2_OK; i++) {
		// sized once, exactly: the object never grows
		const cudaError_t e = cudaMalloc(&bufs[i]->p, sizes[i]);
		if (e != cudaSuccess) {
			bufs[i]->p = nullptr;
			rc = cuda_fail(e, "mc2_greedy_begin: device memory", __FILE__, __LINE__);
		}
		bufs[i]->cap = sizes[i];
	}
	if (rc == MC2_OK) {
		greedy_rows((char *)g->rows.p, n, &g->b);
		g->b.cnt = (u32 *)g->cnt.p;
		g->b.off = (u64 *)g->off.p;
		g->b.bd = (u64 *)g->bd.p;
		g->b.bid = (double *)g->bid.p;
		g->b.bstr = g->both ? (int8_t *)g->bstr.p : nullptr;
		g->b.begin = begin;
		g->b.end = end;
		rc = launch_greedy_init(ctx, g->b.g, n);
	}
	if (rc == MC2_OK) {
		const cudaError_t e = cudaStreamSynchronize(ctx->stream);
		if (e != cudaSuccess) rc = cuda_fail(e, "mc2_greedy_begin", __FILE__, __LINE__);
	}
	if (rc != MC2_OK) {
		mc2_greedy_free(g);
		return rc;
	}
	*out = g;
	return MC2_OK;
}

int mc2_greedy_part_buffers(const mc2_greedy *g, uint32_t part, void **d_records, int8_t **d_strand, uint64_t *capacity)
{
	const std::string w("mc2_greedy_part_buffers");
	MC2_REQUIRE(g && d_records && capacity, w + ": NULL argument");
	MC2_REQUIRE(part < g->n_parts, w + ": part must be < n_parts");
	*d_records = (char *)g->rec.p + (u64)part * g->cap * 16;
	if (d_strand) *d_strand = g->both ? (int8_t *)g->str.p + (u64)part * g->cap : nullptr;
	*capacity = g->cap;
	return MC2_OK;
}

int mc2_greedy_sweep_part(mc2_ctx *ctx, mc2_greedy *g, uint32_t part, uint64_t q_begin, uint64_t q_end, uint64_t *n_edges,
			  uint64_t *n_scored)
{
	const std::string w("mc2_greedy_sweep_part");
	MC2_REQUIRE(ctx && g && n_edges, w + ": NULL argument");
	MC2_REQUIRE(part < g->n_parts, w + ": part must be < n_parts");
	MC2_REQUIRE(g->next <= q_begin && q_begin <= q_end && q_end <= g->end,
		    w + ": the query rows must lie in [the next undecided row, end)");
	MC2_CUDA(cudaSetDevice(ctx->device));
	*n_edges = 0;
	if (n_scored) *n_scored = 0;
	CtxExtra *x = extra(ctx);
	x->last_exact = 0;
	x->last_coarse = 0;
	x->last_inline = x->sum_inline = 0;
	cudaStream_t st = ctx->stream;
	if (q_begin == q_end) {
		// a slot is free once the stream is idle: the caller may write the next block's records into it
		MC2_CUDA(cudaStreamSynchronize(st));
		return MC2_OK;
	}
	const u64 cap = g->cap;
	int rc;
	const int bufs[] = {B_TOPK_Q, B_TOPK_D, B_TOPK_S};
	for (int i = 0; i < 3; i++) {
		if ((rc = ensure(x->d[bufs[i]], cap * 8, false)) != MC2_OK) return rc;
	}
	u64 *sq = (u64 *)x->d[B_TOPK_Q].p, *sd = (u64 *)x->d[B_TOPK_D].p;
	double *ss = (double *)x->d[B_TOPK_S].p;
	u64 total = 0;
	if (g->both) {
		// the reverse survivors of a part fit a scratch of a slot's size, as the forward ones fit the slot: the reverse sweep
		// then takes one or two blocks, as in the single call, rather than one per 2^20 survivors
		rc = sweep_both_strands(ctx, g->dm, g->t, g->set, q_begin, q_end, g->set, g->begin, g->end, 1, g->cutoff, cap, sq, sd, ss,
					(int8_t *)g->str.p + (u64)part * cap, cap, &total, n_scored);
	} else {
		rc = run_sweep(ctx, g->dm, 1, g->t, g->set, q_begin, q_end, g->set, g->begin, g->end, 1, g->cutoff, cap, sq, sd, ss, &total,
			       n_scored);
		if (rc == MC2_OK) rc = check_err(ctx);
	}
	if (rc != MC2_OK) return rc;
	*n_edges = total;
	if (total <= cap) {
		if ((rc = launch_greedy_pack(ctx, sq, sd, ss, total, g->begin, (GreedyEdge *)g->rec.p + (u64)part * cap)) != MC2_OK) return rc;
	}
	MC2_CUDA(cudaStreamSynchronize(st));
	return MC2_OK;
}

int mc2_greedy_add_block(mc2_ctx *ctx, mc2_greedy *g, uint64_t qb, uint64_t qe, const uint64_t *part_q_begin,
			 const uint64_t *part_q_end, const uint64_t *part_edges)
{
	const std::string w("mc2_greedy_add_block");
	MC2_REQUIRE(ctx && g && part_q_begin && part_q_end && part_edges, w + ": NULL argument");
	MC2_REQUIRE(qb == g->next, w + ": the block must start at the next undecided row");
	MC2_REQUIRE(qb <= qe && qe <= g->end, w + ": the block must end at or before end");
	const u64 P = g->n_parts;
	std::vector<u64> h(3 * P);
	u64 at = qb, stride = 0;
	for (u64 p = 0; p < P; p++) {
		MC2_REQUIRE(part_q_begin[p] == at && part_q_begin[p] <= part_q_end[p], w + ": the part ranges must tile [qb, qe) in part order");
		MC2_REQUIRE(part_edges[p] <= g->cap, w + ": a part's edge count exceeds the part capacity");
		at = part_q_end[p];
		h[3 * p] = part_q_begin[p];
		h[3 * p + 1] = part_q_end[p];
		h[3 * p + 2] = part_edges[p];
		stride = std::max<u64>(stride, part_edges[p]);
	}
	MC2_REQUIRE(at == qe, w + ": the part ranges must tile [qb, qe) in part order");
	MC2_CUDA(cudaSetDevice(ctx->device));
	if (qb == qe) return MC2_OK;
	cudaStream_t st = ctx->stream;
	u64 *d_part = (u64 *)g->part.p;
	u32 *bad = (u32 *)(d_part + 3 * P);
	GreedyParts src{(const GreedyEdge *)g->rec.p, g->both ? (const int8_t *)g->str.p : nullptr, d_part, P, stride, g->cap, g->begin,
			g->end, bad};
	const GreedyBlock &b = g->b;
	const u64 rows = g->end - qb;
	// The records came through the caller's exchange: the count pass checks every one before anything else is written, and
	// a bad one leaves the object as it was.
	MC2_CUDA(cudaMemcpyAsync(d_part, h.data(), P * 24, cudaMemcpyHostToDevice, st));
	MC2_CUDA(cudaMemsetAsync(bad, 0, 4, st));
	MC2_CUDA(cudaMemsetAsync(b.cnt, 0, rows * 4, st));
	int rc = launch_greedy_parts_count(ctx, src, qb, b.cnt);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaMemcpyAsync(ctx->h_slot, bad, 4, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	MC2_REQUIRE(*(u32 *)ctx->h_slot == 0, w + ": a part slot holds a record outside its part's query range or outside (r, end)");
	src.bad = nullptr;
	rc = greedy_block(ctx, b, qb, qe, [&](u64 n_rows) -> int {
		int r = launch_seg_scan(ctx, b.cnt, n_rows, b.off);
		if (r != MC2_OK) return r;
		MC2_CUDA(cudaMemsetAsync(b.cnt, 0, n_rows * 4, st)); // now the scatter's cursors
		return launch_greedy_parts_scatter(ctx, src, qb, b.off, b.cnt, b.bid, b.bd, b.bstr);
	});
	if (rc != MC2_OK) return rc;
	// the slots are read: the caller may write the next block's records once this returns
	MC2_CUDA(cudaStreamSynchronize(st));
	g->next = qe;
	return MC2_OK;
}

int mc2_greedy_end(mc2_ctx *ctx, mc2_greedy *g, uint64_t *out_rep, double *out_identity, int8_t *out_strand, uint64_t *n_clusters)
{
	const std::string w("mc2_greedy_end");
	MC2_REQUIRE(ctx && g && out_rep && n_clusters, w + ": NULL argument");
	MC2_REQUIRE(g->next == g->end, w + ": rows remain undecided: add the blocks up to end first");
	MC2_CUDA(cudaSetDevice(ctx->device));
	*n_clusters = 0;
	const u64 n = g->end - g->begin;
	if (n == 0) return MC2_OK;
	return greedy_outputs(ctx, g->b.g, n, g->begin, (char *)g->out.p, out_rep, out_identity, out_strand, n_clusters);
}

int mc2_debug_last_sweep(mc2_ctx *ctx, uint64_t *n_exact, int32_t *coarse, uint64_t *n_inline)
{
	MC2_REQUIRE(ctx && n_exact && coarse, "mc2_debug_last_sweep: NULL argument");
	const CtxExtra *x = extra(ctx);
	*n_exact = x->last_exact;
	*coarse = x->last_coarse;
	if (n_inline) *n_inline = x->last_inline;
	return MC2_OK;
}

int mc2_bench_issue_rate(mc2_ctx *ctx, int iters, double *warp_instr_per_s)
{
	MC2_REQUIRE(ctx && warp_instr_per_s && iters > 0, "mc2_bench_issue_rate: bad argument");
	MC2_CUDA(cudaSetDevice(ctx->device));
	CtxExtra *x = extra(ctx);
	int rc = ensure(x->d[B_MISC], (size_t)ctx->sm_count * 4 * 256 * 4 + 64, false); if (rc) return rc;
	u64 wi = 0;
	rc = launch_issue_probe(ctx, iters, (u32 *)x->d[B_MISC].p, &wi); // warm-up (clocks, instruction cache)
	if (rc != MC2_OK) return rc;
	float ms = 0;
	for (int rep = 0; rep < 3; rep++) { // best of three
		MC2_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
		rc = launch_issue_probe(ctx, iters, (u32 *)x->d[B_MISC].p, &wi);
		if (rc != MC2_OK) return rc;
		MC2_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
		MC2_CUDA(cudaEventSynchronize(ctx->ev1));
		float t = 0;
		MC2_CUDA(cudaEventElapsedTime(&t, ctx->ev0, ctx->ev1));
		if (rep == 0 || t < ms) ms = t;
	}
	*warp_instr_per_s = ms > 0 ? (double)wi / (ms * 1e-3) : 0.0;
	return MC2_OK;
}

int mc2_debug_tile_reductions(mc2_ctx *ctx, const mc2_hset *set_q, uint64_t q_begin, uint64_t q_end, const mc2_hset *set_d,
			      uint64_t d_begin, uint64_t d_end, int32_t need, uint32_t *out_dot, uint32_t *out_emd, uint32_t *out_sad)
{
	MC2_REQUIRE(ctx && set_q && set_d, "mc2_debug_tile_reductions: NULL argument");
	MC2_REQUIRE(q_begin <= q_end && q_end <= set_q->n && d_begin <= d_end && d_end <= set_d->n, "mc2_debug_tile_reductions: row range out of bounds");
	MC2_REQUIRE(tile_sweep_shape_ok(set_q, set_d), "mc2_debug_tile_reductions: needs uint8 / uint16 sets of whole 1 KiB slabs whose rows fit the tile form");
	MC2_REQUIRE((need & 7) != 0 && (need & ~7) == 0, "mc2_debug_tile_reductions: need is a mask of 1 (sad), 2 (dot), 4 (emd)");
	MC2_CUDA(cudaSetDevice(ctx->device));
	const u64 cells = (q_end - q_begin) * (d_end - d_begin);
	if (cells == 0) return MC2_OK;
	CtxExtra *x = extra(ctx);
	int rc = ensure(x->d[B_SCORE], cells * 4, false); if (rc) return rc;
	rc = ensure(x->d[B_DIST], cells * 4, false); if (rc) return rc;
	rc = ensure(x->d[B_CACHE], cells * 4, false); if (rc) return rc;
	rc = ensure(x->d[B_MISC], 64, false); if (rc) return rc;
	MC2_CUDA(cudaMemsetAsync(x->d[B_MISC].p, 0, 64, ctx->stream));
	rc = reset_err(ctx);
	DevModel dm;
	memset(&dm, 0, sizeof dm);
	if (rc == MC2_OK)
		rc = launch_tile_sweep(ctx, dm, need, set_q, q_begin, q_end, set_d, d_begin, d_end, 0, 1.0, 0, nullptr, nullptr, nullptr,
				       (u64 *)x->d[B_MISC].p, (u32 *)x->d[B_SCORE].p, (u32 *)x->d[B_DIST].p, (u32 *)x->d[B_CACHE].p, 0, 0.0);
	if (rc == MC2_OK) rc = fetch_err(ctx);
	if (rc != MC2_OK) return rc;
	cudaStream_t st = ctx->stream;
	if (out_dot && (need & 2)) MC2_CUDA(cudaMemcpyAsync(out_dot, x->d[B_SCORE].p, cells * 4, cudaMemcpyDeviceToHost, st));
	if (out_emd && (need & 4)) MC2_CUDA(cudaMemcpyAsync(out_emd, x->d[B_DIST].p, cells * 4, cudaMemcpyDeviceToHost, st));
	if (out_sad && (need & 1)) MC2_CUDA(cudaMemcpyAsync(out_sad, x->d[B_CACHE].p, cells * 4, cudaMemcpyDeviceToHost, st));
	MC2_CUDA(cudaStreamSynchronize(st));
	return check_err(ctx);
}

int mc2_distance(mc2_ctx *ctx, const mc2_pairs *pairs, uint64_t *out)
{
	MC2_REQUIRE(ctx && pairs && out, "mc2_distance: NULL argument");
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	CtxExtra *x = extra(ctx);
	PairArgs a;
	int rc = fill_pair_args(ctx, pairs, a, x);
	if (rc != MC2_OK) return rc;
	const u64 m = pairs->n_pairs;
	if (m == 0) return MC2_OK;
	rc = ensure(x->d[B_MISC], m * 8 + 64, false); if (rc) return rc;
	rc = launch_distance(ctx, a, (u64 *)x->d[B_MISC].p);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaMemcpyAsync(out, x->d[B_MISC].p, m * 8, cudaMemcpyDeviceToHost, ctx->stream));
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	return MC2_OK;
}

static int mean_closest_impl(mc2_ctx *ctx, const mc2_hset *set, const uint64_t *members, uint64_t n, const double *mean_in,
			     int64_t *best, double *best_dist, double *mean_out, double *dist_out);

int mc2_mean_closest(mc2_ctx *ctx, const mc2_hset *set, const uint64_t *members, uint64_t n, int64_t *best, double *best_dist,
		     double *mean_out, double *dist_out)
{
	return mean_closest_impl(ctx, set, members, n, nullptr, best, best_dist, mean_out, dist_out);
}

int mc2_closest(mc2_ctx *ctx, const mc2_hset *set, const uint64_t *members, uint64_t n, const double *mean, int64_t *best,
		double *best_dist, double *dist_out)
{
	MC2_REQUIRE(mean != nullptr, "mc2_closest: mean is NULL");
	return mean_closest_impl(ctx, set, members, n, mean, best, best_dist, nullptr, dist_out);
}

static int mean_closest_impl(mc2_ctx *ctx, const mc2_hset *set, const uint64_t *members, uint64_t n, const double *mean_in,
			     int64_t *best, double *best_dist, double *mean_out, double *dist_out)
{
	MC2_REQUIRE(ctx && set && members && best && best_dist, "mc2_mean_closest: NULL argument");
	MC2_REQUIRE(n > 0, "mc2_mean_closest: empty member list (the reference throws \"N cannot be 0\")");
	for (u64 j = 0; j < n; j++) {
		MC2_REQUIRE(members[j] < set->n, "mc2_mean_closest: member row out of range");
	}
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	CtxExtra *x = extra(ctx);
	const u64 N = set->N;
	int rc = ensure(x->d[B_IA], n * 8, false); if (rc) return rc;
	rc = ensure(x->d[B_SCORE], N * 8, false); if (rc) return rc;   // column sums
	rc = ensure(x->d[B_CACHE], N * 8, false); if (rc) return rc;   // mean
	rc = ensure(x->d[B_DIST], n * 8, false); if (rc) return rc;    // distances
	cudaStream_t st = ctx->stream;
	if ((rc = h2d(ctx, x->d[B_IA].p, members, n * 8)) != MC2_OK) return rc;
	if (mean_in && (rc = h2d(ctx, x->d[B_CACHE].p, mean_in, N * 8)) != MC2_OK) return rc;
	rc = launch_mean_closest(ctx, set, (const u64 *)x->d[B_IA].p, n, (u64 *)x->d[B_SCORE].p, (double *)x->d[B_CACHE].p,
				 (double *)x->d[B_DIST].p, ctx->d_slot, mean_in != nullptr);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaMemcpyAsync(ctx->h_slot, ctx->d_slot, 16, cudaMemcpyDeviceToHost, st));
	if (mean_out && (rc = d2h(ctx, mean_out, x->d[B_CACHE].p, N * 8)) != MC2_OK) return rc;
	if (dist_out && (rc = d2h(ctx, dist_out, x->d[B_DIST].p, n * 8)) != MC2_OK) return rc;
	if ((rc = sync_stage(ctx)) != MC2_OK) return rc;
	*best = ((long long *)ctx->h_slot)[0];
	*best_dist = ((double *)ctx->h_slot)[1];
	return MC2_OK;
}

/* ---- batched update / merge stage ---------------------------------------------------------------- */
// scores the pair list (ia into set_a, ib into set_b) with the length window and leaves dist / close / skipped on the device
static int score_on_device(mc2_ctx *ctx, const mc2_model *model, const mc2_pairs *p, PairArgs &a)
{
	CtxExtra *x = extra(ctx);
	int rc = fill_pair_args(ctx, p, a, x);
	if (rc != MC2_OK) return rc;
	const u64 m = p->n_pairs;
	rc = ensure(x->d[B_DIST], m * 8, false); if (rc) return rc;
	rc = ensure(x->d[B_CLOSE], m, false); if (rc) return rc;
	rc = ensure(x->d[B_SKIP], m, false); if (rc) return rc;
	a.dist = (double *)x->d[B_DIST].p;
	a.close = (uint8_t *)x->d[B_CLOSE].p;
	a.skipped = (uint8_t *)x->d[B_SKIP].p;
	rc = reset_err(ctx);
	if (rc == MC2_OK) rc = launch_pair_score(ctx, model->dm, a);
	return rc;
}

int mc2_update_centers(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *centers, uint64_t n_centers, const mc2_hset *set_m,
		       const uint64_t *member_off, const uint64_t *members, double id, int64_t *next, uint64_t *n_good)
{
	MC2_REQUIRE(ctx && model && centers && set_m && (n_centers == 0 || (member_off && next)), "mc2_update_centers: NULL argument");
	MC2_REQUIRE(n_centers <= centers->n, "mc2_update_centers: more centers than staged rows");
	if (n_centers == 0) return MC2_OK;
	// round(score) != 0 (Trainer.cpp:135) is the kernel's close flag round(score) > 0 as long as score > -0.5
	if (model->dm.bias < -0.5 || model->dm.regression) {
		set_error("mc2_update_centers: needs a classifier with bias >= -0.5");
		return MC2_ERR_UNSUPPORTED;
	}
	MC2_REQUIRE(member_off[0] == 0, "mc2_update_centers: member_off[0] must be 0");
	for (u64 c = 0; c < n_centers; c++) {
		MC2_REQUIRE(member_off[c] <= member_off[c + 1], "mc2_update_centers: member_off must be non-decreasing");
	}
	const u64 m = member_off[n_centers];
	MC2_REQUIRE(m == 0 || members, "mc2_update_centers: members is NULL");
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	if (m == 0) {
		for (u64 c = 0; c < n_centers; c++) {
			next[c] = -1;
			if (n_good) n_good[c] = 0;
		}
		return MC2_OK;
	}
	std::vector<uint64_t> ia(m);
	for (u64 c = 0; c < n_centers; c++) {
		for (u64 p = member_off[c]; p < member_off[c + 1]; p++) {
			ia[p] = c;
		}
	}
	mc2_pairs p;
	memset(&p, 0, sizeof p);
	p.set_a = centers; // classify(center, member), Trainer.cpp:133
	p.set_b = set_m;
	p.n_pairs = m;
	p.ia = ia.data();
	p.ib = members;
	p.len_filter = 1;
	p.anchor_is_b = 0;
	p.cutoff = id;
	PairArgs a;
	int rc = score_on_device(ctx, model, &p, a);
	if (rc != MC2_OK) return rc;
	CtxExtra *x = extra(ctx);
	const u64 N = set_m->N;
	// scratch: [member_off | next | n_good] and the per-center means, chunked so the means stay below 256 MiB
	u64 chunk = (256ull << 20) / (N * 8);
	chunk = chunk < 1 ? 1 : (chunk > n_centers ? n_centers : chunk);
	rc = ensure(x->d[B_MISC], (3 * n_centers + 1) * 8, false); if (rc) return rc;
	rc = ensure(x->d[B_RAW], chunk * N * 8, false); if (rc) return rc;
	u64 *d_off = (u64 *)x->d[B_MISC].p;
	long long *d_next = (long long *)(d_off + n_centers + 1);
	u64 *d_ng = (u64 *)(d_next + n_centers);
	bool staged = false;
	rc = h2d(ctx, d_off, member_off, (n_centers + 1) * 8, &staged);
	if (rc != MC2_OK) return rc;
	for (u64 c0 = 0; c0 < n_centers && rc == MC2_OK; c0 += chunk) {
		const u64 cnt = n_centers - c0 < chunk ? n_centers - c0 : chunk;
		rc = launch_update_batch(ctx, set_m, d_off, a.ib, a.close, a.skipped, c0, cnt, (double *)x->d[B_RAW].p, d_next, d_ng);
	}
	if (rc == MC2_OK) rc = fetch_err(ctx);
	if (rc != MC2_OK) return rc;
	static_assert(sizeof(int64_t) == sizeof(long long), "int64_t layout");
	MC2_CUDA(cudaMemcpyAsync(next, d_next, n_centers * 8, cudaMemcpyDeviceToHost, ctx->stream));
	if (n_good) MC2_CUDA(cudaMemcpyAsync(n_good, d_ng, n_centers * 8, cudaMemcpyDeviceToHost, ctx->stream));
	if ((rc = sync_stage(ctx)) != MC2_OK) return rc;
	return check_err(ctx);
}

int mc2_merge_centers(mc2_ctx *ctx, const mc2_model *model, const mc2_hset *centers, uint64_t n_centers, int64_t delta, double id,
		      int64_t *out)
{
	MC2_REQUIRE(ctx && model && centers && (n_centers == 0 || out), "mc2_merge_centers: NULL argument");
	MC2_REQUIRE(n_centers <= centers->n && delta >= 0, "mc2_merge_centers: bad center count or delta");
	if (model->dm.regression || model->dm.bias >= 0.5 || model->dm.bias < -0.5) { // see mc2_merge
		set_error("mc2_merge_centers: needs a classifier with -0.5 <= bias < 0.5");
		return MC2_ERR_UNSUPPORTED;
	}
	if (n_centers == 0) return MC2_OK;
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	std::vector<uint64_t> off(n_centers + 1), ia, ib;
	for (u64 c = 0; c < n_centers; c++) {
		off[c] = ia.size();
		const u64 last = (u64)delta < n_centers - 1 - c ? c + (u64)delta : n_centers - 1; // min(size-1, c+delta)
		for (u64 i = c + 1; i <= last; i++) {
			ia.push_back(i); // compute(*cen, *p): the other center first (Trainer.cpp:93)
			ib.push_back(c);
		}
	}
	off[n_centers] = ia.size();
	const u64 m = ia.size();
	if (m == 0) {
		for (u64 c = 0; c < n_centers; c++) out[c] = 0;
		return MC2_OK;
	}
	mc2_pairs p;
	memset(&p, 0, sizeof p);
	p.set_a = centers;
	p.set_b = centers;
	p.n_pairs = m;
	p.ia = ia.data();
	p.ib = ib.data();
	p.len_filter = 1;
	p.anchor_is_b = 1; // the window comes from the current center's length (Trainer.cpp:82-83, 91)
	p.cutoff = id;
	PairArgs a;
	int rc = score_on_device(ctx, model, &p, a);
	if (rc != MC2_OK) return rc;
	CtxExtra *x = extra(ctx);
	rc = ensure(x->d[B_MISC], (2 * n_centers + 1) * 8, false); if (rc) return rc;
	u64 *d_off = (u64 *)x->d[B_MISC].p;
	long long *d_out = (long long *)(d_off + n_centers + 1);
	bool staged = false;
	rc = h2d(ctx, d_off, off.data(), (n_centers + 1) * 8, &staged);
	if (rc == MC2_OK) rc = launch_merge_batch(ctx, a.dist, a.skipped, a.close, d_off, n_centers, d_out);
	if (rc == MC2_OK) rc = fetch_err(ctx);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaMemcpyAsync(out, d_out, n_centers * 8, cudaMemcpyDeviceToHost, ctx->stream));
	if ((rc = sync_stage(ctx)) != MC2_OK) return rc;
	for (u64 c = 0; c < n_centers; c++) {
		out[c] = out[c] < 0 ? 0 : (int64_t)(c + 1) + out[c];
	}
	return check_err(ctx);
}

/* ---- device-timed bench helpers ---------------------------------------------------------------- */
int mc2_bench_score_pairs(mc2_ctx *ctx, const mc2_model *model, const mc2_pairs *pairs, int iters, int flush_l2,
			  float *avg_ms, uint64_t *n_close)
{
	MC2_REQUIRE(ctx && model && pairs && avg_ms && iters > 0, "mc2_bench_score_pairs: bad argument");
	MC2_CUDA(cudaSetDevice(ctx->device));
	drop_stale_stage(ctx);
	CtxExtra *x = extra(ctx);
	PairArgs a;
	int rc = fill_pair_args(ctx, pairs, a, x);
	if (rc != MC2_OK) return rc;
	const u64 m = pairs->n_pairs;
	rc = ensure(x->d[B_SCORE], m * 8, false); if (rc) return rc;
	rc = ensure(x->d[B_CLOSE], m, false); if (rc) return rc;
	rc = ensure(x->d[B_MISC], 64, false); if (rc) return rc;
	a.score = (double *)x->d[B_SCORE].p;
	a.close = (uint8_t *)x->d[B_CLOSE].p;
	a.n_close = (u64 *)x->d[B_MISC].p;
	rc = reset_err(ctx);
	if (rc != MC2_OK) return rc;
	double total = 0;
	for (int it = 0; it < iters; it++) {
		if (flush_l2) {
			rc = mc2_ctx_flush_l2(ctx, 256u << 20);
			if (rc != MC2_OK) return rc;
		}
		MC2_CUDA(cudaMemsetAsync(a.n_close, 0, 8, ctx->stream));
		MC2_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
		rc = launch_pair_score(ctx, model->dm, a);
		if (rc != MC2_OK) return rc;
		MC2_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
		MC2_CUDA(cudaEventSynchronize(ctx->ev1));
		float ms = 0;
		MC2_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
		total += ms;
	}
	*avg_ms = (float)(total / iters);
	rc = fetch_err(ctx);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaMemcpyAsync(ctx->h_slot, a.n_close, 8, cudaMemcpyDeviceToHost, ctx->stream));
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	if (n_close) *n_close = *(u64 *)ctx->h_slot;
	return check_err(ctx);
}

int mc2_bench_count_kmers(mc2_ctx *ctx, const mc2_seqs *seqs, int k, int elem_bytes, int iters, int flush_l2,
			  float *avg_ms)
{
	MC2_REQUIRE(ctx && seqs && avg_ms && iters > 0, "mc2_bench_count_kmers: bad argument");
	int rc = check_k_eb(k, elem_bytes);
	if (rc != MC2_OK) return rc;
	MC2_CUDA(cudaSetDevice(ctx->device));
	mc2_hset *h = nullptr;
	rc = alloc_hset(ctx, seqs->n, k, elem_bytes, &h);
	if (rc != MC2_OK) return rc;
	double total = 0;
	rc = reset_err(ctx);
	for (int it = 0; it < iters && rc == MC2_OK; it++) {
		if (flush_l2) rc = mc2_ctx_flush_l2(ctx, 256u << 20);
		if (rc != MC2_OK) break;
		cudaEventRecord(ctx->ev0, ctx->stream);
		rc = launch_count(ctx, seqs, k, elem_bytes, h, 1);
		cudaEventRecord(ctx->ev1, ctx->stream);
		cudaEventSynchronize(ctx->ev1);
		float ms = 0;
		cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
		total += ms;
	}
	mc2_hset_free(h);
	if (rc != MC2_OK) return rc;
	*avg_ms = (float)(total / iters);
	return MC2_OK;
}

} // extern "C"
