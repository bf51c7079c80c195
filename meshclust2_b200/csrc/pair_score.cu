// pair_score.cu — K2: pair features + GLM score + cutoff, gather / one-vs-many form (sm_100a).
//
// Replaces, for whole batches of pairs, the per-pair chain of the reference
//   Feature<T>::compute  (src/predict/Feature.h:197-201, Feature.cpp:136-171)
//   Feature<T>::operator() combos (Feature.h:205-239)
//   Trainer<T>::classify / Predictor<T>::p_close / p_predict (Trainer.cpp:112-120, Predictor.cpp:284-333)
// One warp walks one pair's two histogram rows with coalesced 16-byte loads and produces the three exact
// integer reductions every "fast" single derives from (SURVEY.md §8 a7):
//     S_sad = sum |p-q|   (VABSDIFF4.U8.ACC, 4 bins / instruction)      -> manhattan, intersection, kulczynski2
//     S_dot = sum p*q     (IDP.4A, 4 bins / instruction)                -> euclidean, simratio, normalized_vectors, pearson
//     S_emd = sum |cumP-cumQ| (per-lane prefix via IDP.4A with +1/-1 byte masks, warp scan, VABSDIFF accumulate)
// The per-pair fp64 epilogue (singles -> normalise -> combos -> w.x -> logistic -> cutoff) runs one pair per
// lane after every 32 pairs, so it costs 1/32 of a warp-serial epilogue.
// HBM-bound by design: algorithmic bytes per pair = N*w (streamed row) + side-band, see DESIGN.md.
#include "mc2_internal.cuh"
#include "pair_eval.cuh"
#include <math_constants.h>
#include <cstring>

namespace mc2 {

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 vabsdiff4_acc(u32 a, u32 b, u32 c)
{
	u32 d;
	asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
	return d;
}
__device__ __forceinline__ int dp4a_us(u32 a, u32 b_s8, int c)
{
	int d;
	asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b_s8), "r"(c));
	return d;
}
__device__ __forceinline__ u32 dp2a_lo_uu(u32 a, u32 b, u32 c)
{
	u32 d;
	asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
	return d;
}
__device__ __forceinline__ u32 dp2a_hi_uu(u32 a, u32 b, u32 c)
{
	u32 d;
	asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
	return d;
}
__device__ __forceinline__ int dp2a_lo_us(u32 a, u32 b_s8, int c)
{
	int d;
	asm("dp2a.lo.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b_s8), "r"(c));
	return d;
}
__device__ __forceinline__ uint4 ldg_stream(const void *p)
{
	// streamed once: do not keep in L1
	uint4 r;
	asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
		     : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
		     : "l"(p));
	return r;
}
__device__ __forceinline__ uint4 ldg_keep(const void *p)
{
	return __ldg(reinterpret_cast<const uint4 *>(p));
}

// exact warp sum of a u64 per lane through three 24-bit limbs and the REDUX unit
__device__ __forceinline__ u64 warp_sum_u64(u64 v)
{
	u32 lo = (u32)(v & 0xFFFFFFu);
	u32 mid = (u32)((v >> 24) & 0xFFFFFFu);
	u32 hi = (u32)(v >> 48);
	u64 s = __reduce_add_sync(0xffffffffu, lo);
	// most totals fit the low limbs; the ballot keeps the extra REDUX off the common path
	if (__any_sync(0xffffffffu, (mid | hi) != 0)) {
		s += (u64)__reduce_add_sync(0xffffffffu, mid) << 24;
		s += (u64)__reduce_add_sync(0xffffffffu, hi) << 48;
	}
	return s;
}
__device__ __forceinline__ double warp_sum_f64(double v)
{
#pragma unroll
	for (int d = 16; d > 0; d >>= 1) {
		v += __shfl_xor_sync(0xffffffffu, v, d);
	}
	return v;
}
__device__ __forceinline__ s64 shfl_up_s64(s64 v, int d)
{
	return __shfl_up_sync(0xffffffffu, v, d);
}

// accumulators reproducing the reference's type-dependent arithmetic for 32/64-bit histograms (SURVEY E2-E4)
struct RedW {
	int man;
	u64 euc, nv_sum, nv_d1, nv_d2, smin, inter2, emd, norm2;
	double dpq, dpp, dqq, jeff, js;
};


__device__ int raw_single_narrow(int code, u64 N, const RedN &r, const Side &p, const Side &q, double *out)
{
	switch (code) {
	case SC_MANHATTAN: { // Feature.cpp:858-871 (int accumulator)
		u64 sad = p.sum + q.sum - 2 * r.smin;
		*out = (double)(int)sad;
		return 0;
	}
	case SC_EUCLIDEAN: // Feature.cpp:1112-1124
		*out = sqrt((double)(p.sumsq + q.sumsq - 2 * r.dot));
		return 0;
	case SC_NORMALIZED_VECTORS: // Feature.cpp:1170-1184 (u64 product, wraps like the reference)
		*out = (double)r.dot / sqrt((double)(p.sumsq * q.sumsq));
		return 0;
	case SC_PEARSON:
		*out = pearson_exact(N, r.dot, p, q);
		return 0;
	case SC_INTERSECTION: // Feature.cpp:763-777
		*out = (double)(2 * r.smin) / (double)(p.mag + q.mag);
		return 0;
	case SC_EMD: // Feature.cpp:1504-1518
		*out = (double)r.emd;
		return 0;
	case SC_LENGTHD: // Feature.cpp:873-887 (throws 123 on a zero length)
		if (p.len == 0 || q.len == 0) {
			return 1;
		}
		*out = (double)(p.len > q.len ? p.len - q.len : q.len - p.len);
		return 0;
	case SC_KULCZYNSKI2: { // Feature.cpp:681-695
		double ap = (double)p.mag / (double)N;
		double aq = (double)q.mag / (double)N;
		double coeff = (double)N * (ap + aq) / (2 * ap * aq);
		*out = coeff * (double)r.smin;
		return 0;
	}
	case SC_SIMRATIO: { // Feature.cpp:828-841
		double dot = (double)r.dot;
		u64 norm2 = p.sumsq + q.sumsq - 2 * r.dot;
		*out = dot / (dot + sqrt((double)norm2));
		return 0;
	}
	case SC_JEFFEREY: // Feature.cpp:1230-1263
		*out = r.jeff;
		return 0;
	case SC_JENSEN_SHANNON: // Feature.cpp:983-1009
		*out = r.js / 2;
		return 0;
	}
	return 2;
}

__device__ int raw_single_wide(int code, u64 N, const RedW &r, const Side &p, const Side &q, double *out)
{
	switch (code) {
	case SC_MANHATTAN:
		*out = (double)r.man;
		return 0;
	case SC_EUCLIDEAN:
		*out = sqrt((double)r.euc);
		return 0;
	case SC_NORMALIZED_VECTORS:
		*out = (double)r.nv_sum / sqrt((double)(r.nv_d1 * r.nv_d2));
		return 0;
	case SC_PEARSON: { // fp64 sums of products; the reference's own loop is fp64 too
		double dap = (double)p.mag / (double)N;
		double daq = (double)q.mag / (double)N;
		double n = (double)N;
		double dot = r.dpq - dap * (double)q.sum - daq * (double)p.sum + n * dap * daq;
		double np = r.dpp - 2 * dap * (double)p.sum + n * dap * dap;
		double nq = r.dqq - 2 * daq * (double)q.sum + n * daq * daq;
		*out = dot / sqrt(np * nq);
		return 0;
	}
	case SC_INTERSECTION:
		*out = (double)r.inter2 / (double)(p.mag + q.mag);
		return 0;
	case SC_EMD:
		*out = (double)r.emd;
		return 0;
	case SC_LENGTHD:
		if (p.len == 0 || q.len == 0) {
			return 1;
		}
		*out = (double)(p.len > q.len ? p.len - q.len : q.len - p.len);
		return 0;
	case SC_KULCZYNSKI2: {
		double ap = (double)p.mag / (double)N;
		double aq = (double)q.mag / (double)N;
		double coeff = (double)N * (ap + aq) / (2 * ap * aq);
		*out = coeff * (double)r.smin;
		return 0;
	}
	case SC_SIMRATIO: {
		double dot = (double)r.nv_sum;
		*out = dot / (dot + sqrt((double)r.norm2));
		return 0;
	}
	case SC_JEFFEREY:
		*out = r.jeff;
		return 0;
	case SC_JENSEN_SHANNON:
		*out = r.js / 2;
		return 0;
	}
	return 2;
}


// normalise (Feature.cpp:136-154), combos (Feature.h:205-239), GLM sum, logistic + bias (Predictor.cpp:316-320)
// returns a bit mask: 1 = the reference would throw, 2 = internal (unknown single code)
template <typename RED, bool WIDE>
__device__ int eval_pair(const DevModel &dm, u64 N, const RED &r, const Side &first, const Side &second, double *raw_out,
			 double *cache_out, double &score, double &d0, int &close, bool lazy = false)
{
	if constexpr (!WIDE) {
		if (dm.fast_epi && raw_out == nullptr && cache_out == nullptr) {
			return eval_pair_fast(dm, N, r, first, second, lazy, score, d0, close);
		}
	}
	double cache[MC2_MAX_SINGLES];
	int bad = 0;
#pragma unroll 1
	for (int i = 0; i < dm.n_singles; i++) {
		double v = 0;
		int rc;
		if constexpr (WIDE) {
			rc = raw_single_wide(dm.code[i], N, r, first, second, &v);
		} else {
			rc = raw_single_narrow(dm.code[i], N, r, first, second, &v);
		}
		bad |= rc;
		if (raw_out) {
			raw_out[i] = v;
		}
		double nv = (v - dm.smin[i]) / (dm.smax[i] - dm.smin[i]);
		if (isnan(nv)) {
			bad |= 1;
		}
		cache[i] = dm.is_sim[i] ? nv : 1 - nv;
		if (cache_out) {
			cache_out[i] = cache[i];
		}
	}
	double sum = dm.weight[0];
	d0 = 0;
#pragma unroll 1
	for (int c = 0; c < dm.n_combos; c++) {
		double d;
		const int *ix = dm.idx[c];
		switch (dm.kind[c]) {
		case MC2_COMBO_XY: {
			double prod = 1;
			for (int t = 0; t < dm.nidx[c]; t++) {
				prod *= cache[ix[t]];
			}
			d = prod;
			break;
		}
		case MC2_COMBO_X2Y2: {
			double prod = 1;
			for (int t = 0; t < dm.nidx[c]; t++) {
				prod *= cache[ix[t]] * cache[ix[t]];
			}
			d = prod;
			break;
		}
		case MC2_COMBO_XY2:
			d = cache[ix[0]] * cache[ix[1]] * cache[ix[1]];
			break;
		default: // MC2_COMBO_X2Y
			d = cache[ix[0]] * cache[ix[0]] * cache[ix[1]];
			break;
		}
		if (c == 0) {
			d0 = d;
		}
		sum += dm.weight[c + 1] * d;
	}
	if (dm.regression) { // Predictor::p_predict, Predictor.cpp:284-300
		score = sum < 0 ? 0 : (sum > 1 ? 1 : sum);
		close = 0;
	} else {
		score = 1.0 / (1 + exp(-sum)) + dm.bias;
		close = round(score) > 0;
	}
	return bad;
}

template <typename RED, bool WIDE>
__device__ void finish_pair(const DevModel &dm, const PairArgs &a, u64 j, u64 N, const RED &r, const Side &first,
			    const Side &second)
{
	double score, d0;
	int close;
	const u64 S = (u64)dm.n_singles;
	int bad = eval_pair<RED, WIDE>(dm, N, r, first, second, a.raw ? a.raw + j * S : nullptr,
				       a.cache ? a.cache + j * S : nullptr, score, d0, close, a.score == nullptr);
	if (bad) {
		atomicOr(a.err, bad & 1 ? 1 : 2);
	}
	if (a.score) {
		a.score[j] = score;
	}
	if (a.dist) {
		a.dist[j] = d0;
	}
	if (a.close) {
		a.close[j] = (uint8_t)close;
	}
	if (a.skipped) {
		a.skipped[j] = 0;
	}
	if (a.n_close && close) {
		atomicAdd(a.n_close, 1ULL);
	}
}

__device__ __forceinline__ void write_skipped(const PairArgs &a, u64 j)
{
	if (a.score) {
		a.score[j] = CUDART_NAN;
	}
	if (a.dist) {
		a.dist[j] = CUDART_NAN;
	}
	if (a.close) {
		a.close[j] = 0;
	}
	if (a.skipped) {
		a.skipped[j] = 1;
	}
}

// rows + length prefilter for pair j (Trainer.cpp:39-48 / 82-91 / 126-130: u64 truncation of len*cutoff, len/cutoff)
__device__ __forceinline__ bool resolve_pair(const PairArgs &a, u64 j, u64 &ra, u64 &rb)
{
	ra = a.ia ? a.ia[j] : a.a_begin + (a.a_bc ? 0 : j);
	rb = a.ib ? a.ib[j] : a.b_begin + (a.b_bc ? 0 : j);
	if (a.len_filter) {
		u64 la = a.sbA.len[ra], lb = a.sbB.len[rb];
		u64 anchor = a.anchor_is_b ? lb : la;
		u64 other = a.anchor_is_b ? la : lb;
		u64 min_len = (u64)((double)anchor * a.cutoff);
		u64 max_len = (u64)((double)anchor / a.cutoff);
		if (other < min_len || other > max_len) {
			return false;
		}
	}
	return true;
}

// ------------------------------------------------------------------------------------------------
// fast path: 8/16-bit bins, rows a multiple of 1 KiB, bin sums < 2^26.
// A warp walks a row in 1 KiB slabs; lane l owns the 32 CONTIGUOUS bytes [32l, 32l+32) of the slab (one 256-bit
// load, the warp reads 1 KiB contiguous), so the EMD prefix needs ONE warp scan per slab:
//   tot_l   = sum_lane(p) - sum_lane(q)                 (IDP with all-ones / all-minus-ones byte masks)
//   off_l   = exclusive warp scan of tot + carry        (5 SHFL.UP with predicated add)
//   c_{i+1} = c_i + p_i - q_i  starting at off_l        (PRMT interleave + IDP with +1/-1 masks, 2 bins per dependent step)
//   emd    += |c_i|                                      (VABSDIFF with accumulate)
// ------------------------------------------------------------------------------------------------
struct Row8 {
	u32 w[8];
};

__device__ __forceinline__ Row8 ld_row_stream(const void *p)
{
	Row8 r;
	asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
		     : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
		     : "l"(p));
	return r;
}
__device__ __forceinline__ Row8 ld_row_keep(const void *p)
{
	Row8 r;
	asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
		     : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
		     : "l"(p));
	return r;
}

// inclusive scan step: x += shfl_up(x, d) where the source lane exists
__device__ __forceinline__ void scan_step(int &x, int d)
{
	asm volatile("{\n\t.reg .s32 t;\n\t.reg .pred p;\n\tshfl.sync.up.b32 t|p, %0, %1, 0x0, 0xffffffff;\n\t@p add.s32 %0, %0, t;\n\t}"
		     : "+r"(x)
		     : "r"(d));
}
__device__ __forceinline__ int warp_excl_scan(int tot, int &warp_total)
{
	int x = tot;
	scan_step(x, 1);
	scan_step(x, 2);
	scan_step(x, 4);
	scan_step(x, 8);
	scan_step(x, 16);
	warp_total = __shfl_sync(0xffffffffu, x, 31);
	return x - tot;
}

// sum over the lane's 32 bytes of q, as the (negative) constant the scan needs; hoisted when q is the fixed query
template <typename T>
__device__ __forceinline__ int lane_sum(const Row8 &q)
{
	u32 s = 0;
#pragma unroll
	for (int w = 0; w < 8; w++) {
		if (sizeof(T) == 1) {
			s = __dp4a(q.w[w], 0x01010101u, s);
		} else {
			s = dp2a_lo_uu(q.w[w], 0x0101u, s);
		}
	}
	return (int)s;
}

// one 1 KiB slab: per-lane partial sums; `carry` is the running cumP-cumQ at the start of the slab
template <typename T, int NEED>
__device__ __forceinline__ void slab_reduce(const Row8 &p, const Row8 &q, int qsum, int &carry, u32 &a_min, u32 &a_dot_lo,
					    u32 &a_dot_hi, u32 &a_emd)
{
	if (NEED & NEED_MIN) {
#pragma unroll
		for (int w = 0; w < 8; w++) {
			if (sizeof(T) == 1) {
				a_min = vabsdiff4_acc(p.w[w], q.w[w], a_min);   // sum |p-q| (converted to S_min by the caller)
			} else {
				a_min = dp2a_lo_uu(__vminu2(p.w[w], q.w[w]), 0x0101u, a_min);
			}
		}
	}
	if (NEED & NEED_DOT) {
#pragma unroll
		for (int w = 0; w < 8; w++) {
			if (sizeof(T) == 1) {
				a_dot_lo = __dp4a(p.w[w], q.w[w], a_dot_lo);
			} else {
				u32 qp = __byte_perm(q.w[w], q.w[w], 0x3120); // q0.lo q1.lo q0.hi q1.hi
				a_dot_lo = dp2a_lo_uu(p.w[w], qp, a_dot_lo);
				a_dot_hi = dp2a_hi_uu(p.w[w], qp, a_dot_hi);
			}
		}
	}
	if (NEED & NEED_EMD) {
		int tot = lane_sum<T>(p) - qsum;
		int wt;
		int c = warp_excl_scan(tot, wt) + carry;
		carry += wt;
		u32 e = a_emd;
#pragma unroll
		for (int w = 0; w < 8; w++) {
			if (sizeof(T) == 1) {
				u32 w01 = __byte_perm(p.w[w], q.w[w], 0x5140); // p0 q0 p1 q1
				u32 w23 = __byte_perm(p.w[w], q.w[w], 0x7362); // p2 q2 p3 q3
				int l0 = dp4a_us(w01, 0x0000FF01u, c);
				int l1 = dp4a_us(w01, 0xFF01FF01u, c);
				int l2 = dp4a_us(w23, 0x0000FF01u, l1);
				int l3 = dp4a_us(w23, 0xFF01FF01u, l1);
				c = l3;
				e = __sad(l0, 0, e);
				e = __sad(l1, 0, e);
				e = __sad(l2, 0, e);
				e = __sad(l3, 0, e);
			} else {
				u32 w0 = __byte_perm(p.w[w], q.w[w], 0x5410); // p0 (16 bit) | q0 (16 bit)
				u32 w1 = __byte_perm(p.w[w], q.w[w], 0x7632); // p1 | q1
				int l0 = dp2a_lo_us(w0, 0xFF01u, c);
				int l1 = dp2a_lo_us(w1, 0xFF01u, l0);
				c = l1;
				e = __sad(l0, 0, e);
				e = __sad(l1, 0, e);
			}
		}
		a_emd = e;
	}
}

#define MC2_SLAB_PREFETCH 8 // multi-slab rows: L2 prefetch distance in 1 KiB slabs
// whole row pair, any number of slabs; q rows come through L1 (hot when q is the broadcast side)
template <typename T, int NEED>
__device__ __forceinline__ RedN reduce_rows_fast(const T *__restrict__ P, const T *__restrict__ Q, u32 slabs, int lane,
						 bool q_hot)
{
	u64 t_min = 0, t_dot = 0, t_emd = 0;
	int carry = 0;
	const char *pp = reinterpret_cast<const char *>(P) + lane * 32;
	const char *qq = reinterpret_cast<const char *>(Q) + lane * 32;
	Row8 pv = ld_row_stream(pp);
	Row8 qv = q_hot ? ld_row_keep(qq) : ld_row_stream(qq);
#pragma unroll 1
	for (u32 s = 0; s < slabs; s++) {
		Row8 pn = pv, qn = qv;
		if (s + 1 < slabs) { // next slab in flight during this slab's ALU work
			pn = ld_row_stream(pp + (size_t)(s + 1) * 1024);
			qn = q_hot ? ld_row_keep(qq + (size_t)(s + 1) * 1024) : ld_row_stream(qq + (size_t)(s + 1) * 1024);
		}
		if (s + MC2_SLAB_PREFETCH < slabs) { // and the slabs further ahead on their way from HBM into L2
			asm volatile("prefetch.global.L2 [%0];" ::"l"(pp + (size_t)(s + MC2_SLAB_PREFETCH) * 1024));
			if (!q_hot) {
				asm volatile("prefetch.global.L2 [%0];" ::"l"(qq + (size_t)(s + MC2_SLAB_PREFETCH) * 1024));
			}
		}
		u32 a_min = 0, lo = 0, hi = 0, e = 0;
		slab_reduce<T, NEED>(pv, qv, (NEED & NEED_EMD) ? lane_sum<T>(qv) : 0, carry, a_min, lo, hi, e);
		t_min += a_min;
		t_dot += (u64)lo + ((u64)hi << 8);
		t_emd += e;
		pv = pn;
		qv = qn;
	}
	RedN r;
	r.smin = (NEED & NEED_MIN) ? warp_sum_u64(t_min) : 0;
	r.dot = (NEED & NEED_DOT) ? warp_sum_u64(t_dot) : 0;
	r.emd = (NEED & NEED_EMD) ? warp_sum_u64(t_emd) : 0;
	r.jeff = r.js = 0;
	return r;
}

// ------------------------------------------------------------------------------------------------
// single-slab rows (k=5 uint8: 1 KiB, the BASELINE shape) against a FIXED row q (the query of a candidate scan, or the
// query row of one sweep group).  Everything that depends only on q is hoisted into registers once:
//   q.w[8]   the lane's 32 bins (for the dot / min terms)
//   bq[32]   the lane-local inclusive prefix sums of q, so that  |cumP_i - cumQ_i| = |(off + prefixP_i) - bq_i|
//            is ONE VABSDIFF whose operands are an IDP result and a register: no byte interleave (PRMT) at all.
// Per streamed row and lane: 8 IDP (dot) + 8 IDP (lane total of p) + 32 IDP (prefixes) on the full-rate FMA pipe,
// 32 VABSDIFF on the half-rate ALU pipe, one 5-step warp scan, one REDUX per needed sum.
// ------------------------------------------------------------------------------------------------
struct FixedQ {
	Row8 q;
	int bq[32];
	int qsum;
	int qoff; // sum of the fixed row's bins below this lane's chunk (from lane_off), used when LOFF
};

template <int NEED>
__device__ __forceinline__ void fixed_q_setup(FixedQ &f, const void *row, int lane)
{
	f.q = ld_row_keep(reinterpret_cast<const char *>(row) + lane * 32);
	int base = 0;
#pragma unroll
	for (int w = 0; w < 8; w++) {
		if (NEED & NEED_EMD) {
			f.bq[4 * w + 0] = (int)__dp4a(f.q.w[w], 0x00000001u, (u32)base);
			f.bq[4 * w + 1] = (int)__dp4a(f.q.w[w], 0x00000101u, (u32)base);
			f.bq[4 * w + 2] = (int)__dp4a(f.q.w[w], 0x00010101u, (u32)base);
			f.bq[4 * w + 3] = (int)__dp4a(f.q.w[w], 0x01010101u, (u32)base);
			base = f.bq[4 * w + 3];
		}
	}
	f.qsum = base;
	f.qoff = 0;
}

template <int NEED>
__device__ __forceinline__ void reduce_row1(const Row8 &p, const FixedQ &f, u32 &smin, u32 &dot, u32 &emd)
{
	u32 a_min = 0, a_dot = 0, e = 0;
	if (NEED & NEED_MIN) {
#pragma unroll
		for (int w = 0; w < 8; w++) {
			a_min = vabsdiff4_acc(p.w[w], f.q.w[w], a_min); // sum |p-q| (converted to S_min by the caller)
		}
	}
	if (NEED & NEED_DOT) {
		u32 d0 = 0, d1 = 0; // two chains for ILP
#pragma unroll
		for (int w = 0; w < 8; w += 2) {
			d0 = __dp4a(p.w[w], f.q.w[w], d0);
			d1 = __dp4a(p.w[w + 1], f.q.w[w + 1], d1);
		}
		a_dot = d0 + d1;
	}
	if (NEED & NEED_EMD) {
		u32 t0 = 0, t1 = 0;
#pragma unroll
		for (int w = 0; w < 8; w += 2) {
			t0 = __dp4a(p.w[w], 0x01010101u, t0);
			t1 = __dp4a(p.w[w + 1], 0x01010101u, t1);
		}
		int wt;
		int base = warp_excl_scan((int)(t0 + t1) - f.qsum, wt);
		u32 e0 = 0, e1 = 0;
#pragma unroll
		for (int w = 0; w < 8; w++) {
			int a0 = (int)__dp4a(p.w[w], 0x00000001u, (u32)base);
			int a1 = (int)__dp4a(p.w[w], 0x00000101u, (u32)base);
			int a2 = (int)__dp4a(p.w[w], 0x00010101u, (u32)base);
			int a3 = (int)__dp4a(p.w[w], 0x01010101u, (u32)base);
			base = a3;
			e0 = __sad(a0, f.bq[4 * w + 0], e0);
			e1 = __sad(a1, f.bq[4 * w + 1], e1);
			e0 = __sad(a2, f.bq[4 * w + 2], e0);
			e1 = __sad(a3, f.bq[4 * w + 3], e1);
		}
		e = e0 + e1;
	}
	// N*w = 1 KiB: every warp total fits 32 bits (dot <= 2^26, emd <= 2^28), one REDUX each
	smin = (NEED & NEED_MIN) ? __reduce_add_sync(0xffffffffu, a_min) : 0;
	dot = (NEED & NEED_DOT) ? __reduce_add_sync(0xffffffffu, a_dot) : 0;
	emd = (NEED & NEED_EMD) ? __reduce_add_sync(0xffffffffu, e) : 0;
}

// two streamed rows against the same fixed row, written side by side so the two dependency chains (lane totals ->
// warp scan -> prefix chain -> |.| accumulation -> REDUX) interleave and hide each other's latencies
template <int NEED, bool LOFF>
__device__ __forceinline__ void reduce_row2(const Row8 &pa, const Row8 &pb, int offa, int offb, const FixedQ &f, u32 (&oa)[3],
					    u32 (&ob)[3])
{
	u32 mina = 0, minb = 0, dota = 0, dotb = 0, ea = 0, eb = 0;
	if (NEED & NEED_MIN) {
#pragma unroll
		for (int w = 0; w < 8; w++) {
			mina = vabsdiff4_acc(pa.w[w], f.q.w[w], mina);
			minb = vabsdiff4_acc(pb.w[w], f.q.w[w], minb);
		}
	}
	if (NEED & NEED_DOT) {
#pragma unroll
		for (int w = 0; w < 8; w++) {
			dota = __dp4a(pa.w[w], f.q.w[w], dota);
			dotb = __dp4a(pb.w[w], f.q.w[w], dotb);
		}
	}
	if (NEED & NEED_EMD) {
		int basea, baseb;
		if (LOFF) {
			// cumP - cumQ at the lane boundary comes from the precomputed lane offsets: no lane totals, no warp scan
			basea = offa - f.qoff;
			baseb = offb - f.qoff;
		} else {
			u32 ta = 0, tb = 0;
#pragma unroll
			for (int w = 0; w < 8; w++) {
				ta = __dp4a(pa.w[w], 0x01010101u, ta);
				tb = __dp4a(pb.w[w], 0x01010101u, tb);
			}
			int xa = (int)ta - f.qsum, xb = (int)tb - f.qsum;
			const int ta0 = xa, tb0 = xb;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				scan_step(xa, d);
				scan_step(xb, d);
			}
			basea = xa - ta0;
			baseb = xb - tb0;
		}
#pragma unroll
		for (int w = 0; w < 8; w++) {
			int a0 = (int)__dp4a(pa.w[w], 0x00000001u, (u32)basea);
			int b0 = (int)__dp4a(pb.w[w], 0x00000001u, (u32)baseb);
			int a1 = (int)__dp4a(pa.w[w], 0x00000101u, (u32)basea);
			int b1 = (int)__dp4a(pb.w[w], 0x00000101u, (u32)baseb);
			int a2 = (int)__dp4a(pa.w[w], 0x00010101u, (u32)basea);
			int b2 = (int)__dp4a(pb.w[w], 0x00010101u, (u32)baseb);
			int a3 = (int)__dp4a(pa.w[w], 0x01010101u, (u32)basea);
			int b3 = (int)__dp4a(pb.w[w], 0x01010101u, (u32)baseb);
			basea = a3;
			baseb = b3;
			ea = __sad(a0, f.bq[4 * w + 0], ea);
			eb = __sad(b0, f.bq[4 * w + 0], eb);
			ea = __sad(a1, f.bq[4 * w + 1], ea);
			eb = __sad(b1, f.bq[4 * w + 1], eb);
			ea = __sad(a2, f.bq[4 * w + 2], ea);
			eb = __sad(b2, f.bq[4 * w + 2], eb);
			ea = __sad(a3, f.bq[4 * w + 3], ea);
			eb = __sad(b3, f.bq[4 * w + 3], eb);
		}
	}
	oa[0] = (NEED & NEED_MIN) ? __reduce_add_sync(0xffffffffu, mina) : 0;
	ob[0] = (NEED & NEED_MIN) ? __reduce_add_sync(0xffffffffu, minb) : 0;
	oa[1] = (NEED & NEED_DOT) ? __reduce_add_sync(0xffffffffu, dota) : 0;
	ob[1] = (NEED & NEED_DOT) ? __reduce_add_sync(0xffffffffu, dotb) : 0;
	oa[2] = (NEED & NEED_EMD) ? __reduce_add_sync(0xffffffffu, ea) : 0;
	ob[2] = (NEED & NEED_EMD) ? __reduce_add_sync(0xffffffffu, eb) : 0;
}

// predicated 256-bit streaming load: the destination keeps its old contents when pred is false, so the register
// ring below never needs a copy that would wait on a load still in flight
__device__ __forceinline__ void ld_row_stream_if(Row8 &r, const void *p, int pred)
{
	asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.s32 q, %9, 0;\n\t"
		     "@q ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n\t}"
		     : "+r"(r.w[0]), "+r"(r.w[1]), "+r"(r.w[2]), "+r"(r.w[3]), "+r"(r.w[4]), "+r"(r.w[5]), "+r"(r.w[6]), "+r"(r.w[7])
		     : "l"(p), "r"(pred));
}

__device__ __forceinline__ void ld_u16_if(int &v, const unsigned short *p, int pred)
{
	asm volatile("{\n\t.reg .pred q;\n\t.reg .u16 t;\n\tsetp.ne.s32 q, %2, 0;\n\t@q ld.global.nc.u16 t, [%1];\n\t@q cvt.u32.u16 %0, t;\n\t}"
		     : "+r"(v)
		     : "l"(p), "r"(pred));
}

// stream the rows of up to 32 pairs (bit mask `active`, row index of pair i held by lane i in `rs`, or consecutive rows
// first_row + i when contig) against the fixed row, two rows per step.  Two buffer pairs alternate by loop unrolling
// (no register copies): while one pair of rows is reduced the next pair is in flight.
// PF > 0 (HBM-streaming callers): while rows pi..pi+3 are reduced, the rows PF ahead are pulled into L2 with
// prefetch.global.L2 — of this group, or past its end of the group this warp takes next (pf_next) — so the register ring's
// loads find them on chip; one instruction per row and lane, no registers held.
template <int NEED, bool LOFF, int PF = 0>
__device__ __forceinline__ void scan_group(const unsigned char *S, const unsigned short *loff, u64 row_bytes, unsigned active,
					   u64 rs, bool contig, u64 first_row, const FixedQ &f, int lane, u32 &my_min, u32 &my_dot,
					   u32 &my_emd, const unsigned char *pf_next = nullptr)
{
	auto next_idx = [&]() -> int {
		int pi = active ? __ffs(active) - 1 : -1;
		active &= active ? active - 1 : 0;
		return pi;
	};
	auto fetch = [&](Row8 &r, int &off, int pi) {
		// the shuffle must be executed by the whole warp: clamp the source lane instead of predicating it
		u64 x = contig ? first_row + (u64)(pi < 0 ? 0 : pi) : __shfl_sync(0xffffffffu, rs, pi < 0 ? 0 : pi);
		ld_row_stream_if(r, S + x * row_bytes + lane * 32, pi >= 0);
		if (LOFF && (NEED & NEED_EMD)) {
			ld_u16_if(off, loff + x * 32 + lane, pi >= 0);
		}
	};
	auto reduce = [&](const Row8 &ra, int oa_, int ia, const Row8 &rb, int ob_, int ib) {
		u32 oa[3], ob[3];
		reduce_row2<NEED, LOFF>(ra, rb, oa_, ob_, f, oa, ob); // an absent second row (ib < 0) reduces stale data that nobody keeps
		if (lane == ia) {
			my_min = oa[0];
			my_dot = oa[1];
			my_emd = oa[2];
		}
		if (lane == ib) {
			my_min = ob[0];
			my_dot = ob[1];
			my_emd = ob[2];
		}
	};
	Row8 a0 = {}, b0 = {}, a1 = {}, b1 = {};
	int fa0 = 0, fb0 = 0, fa1 = 0, fb1 = 0; // lane offsets of the four buffered rows
	if (contig && active == 0xffffffffu) {
		// the common case — 32 consecutive rows, none filtered: plain counted loop, no mask / ffs / predicate traffic
		const unsigned char *rp = S + first_row * row_bytes + lane * 32;
		const unsigned short *op = loff + first_row * 32 + lane;
		auto get = [&](Row8 &r, int &off, int pi) {
			r = ld_row_stream(rp + (size_t)pi * row_bytes);
			if (LOFF && (NEED & NEED_EMD)) {
				off = (int)__ldg(op + pi * 32);
			}
		};
		get(a0, fa0, 0);
		get(b0, fb0, 1);
		get(a1, fa1, 2);
		get(b1, fb1, 3);
		// the prefetch is unconditional: the last trip re-reads rows 0..3 of the group (L2 hits, results unused) instead
		// of predicating the loads (~6 predicated register moves per pair) or peeling a second copy of the body (the
		// kernel is instruction-cache sensitive: stall_no_instruction grew from 0.4 to 1.0 per issue with the copy)
#pragma unroll 1
		for (int pi = 0; pi < 32; pi += 4) {
			if (PF > 0) {
				const int t = pi + PF;
				const unsigned char *p = t < 32 ? rp + (size_t)t * row_bytes : pf_next + (size_t)(t - 32) * row_bytes;
#pragma unroll
				for (int u = 0; u < 4; u++) {
					asm volatile("prefetch.global.L2 [%0];" ::"l"(p + (size_t)u * row_bytes));
				}
			}
			reduce(a0, fa0, pi, b0, fb0, pi + 1);
			get(a0, fa0, (pi + 4) & 31);
			get(b0, fb0, (pi + 5) & 31);
			reduce(a1, fa1, pi + 2, b1, fb1, pi + 3);
			get(a1, fa1, (pi + 6) & 31);
			get(b1, fb1, (pi + 7) & 31);
		}
		return;
	}
	int ia0 = next_idx();
	if (ia0 < 0) {
		return;
	}
	int ib0 = next_idx();
	fetch(a0, fa0, ia0);
	fetch(b0, fb0, ib0);
	int ia1 = next_idx(), ib1 = next_idx();
	fetch(a1, fa1, ia1);
	fetch(b1, fb1, ib1);
	while (true) {
		reduce(a0, fa0, ia0, b0, fb0, ib0);
		if (ia1 < 0) {
			break;
		}
		ia0 = next_idx();
		ib0 = next_idx();
		fetch(a0, fa0, ia0);
		fetch(b0, fb0, ib0);
		reduce(a1, fa1, ia1, b1, fb1, ib1);
		if (ia0 < 0) {
			break;
		}
		ia1 = next_idx();
		ib1 = next_idx();
		fetch(a1, fa1, ia1);
		fetch(b1, fb1, ib1);
	}
}

#define MC2_PAIR_PREFETCH_ROWS 8 // one-vs-many: L2 prefetch distance in rows (0 = off)
#define MC2_PAIR_CTAS_PER_SM 4 // resident 128-thread CTAs of the one-vs-many (1 KiB rows) form
template <typename T, int NEED, bool ONE, bool LOFF>
__global__ void __launch_bounds__(ONE ? 128 : 256, ONE ? MC2_PAIR_CTAS_PER_SM : 2) pair_fast_kernel(const __grid_constant__ DevModel dm, const __grid_constant__ PairArgs a)
{
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	const u64 warp_id = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
	const u32 slabs = (u32)(a.N * sizeof(T) / 1024);
	const T *A = reinterpret_cast<const T *>(a.binsA);
	const T *B = reinterpret_cast<const T *>(a.binsB);
	// pairs per warp group: 32 (one epilogue lane each) unless the batch is too small to occupy the GPU that way; the
	// fixed-row (ONE) form always takes 32 consecutive rows
	const u32 G = (ONE || a.group <= 0) ? 32u : (u32)a.group;
	const u64 groups = (a.n_pairs + G - 1) / G;
	// the streamed side is the one that is not broadcast; the broadcast row stays resident
	const bool a_hot = a.a_bc && !a.ia;
	const bool b_hot = a.b_bc && !a.ib;
	constexpr bool fixed_q = ONE; // host picks ONE when slabs == 1, T = u8 and one side is a broadcast row
	FixedQ fq;
	if constexpr (fixed_q) { // one-vs-many: the query row and its prefix sums live in registers for the whole kernel
		const T *qrow = a_hot ? A + a.a_begin * a.N : B + a.b_begin * a.N;
		fixed_q_setup<NEED>(fq, qrow, lane);
		if (LOFF) {
			fq.qoff = a_hot ? a.loffA[a.a_begin * 32 + lane] : a.loffB[a.b_begin * 32 + lane];
		}
	}
	for (u64 g = warp_id; g < groups; g += warps_total) {
		const u64 j = g * G + lane;
		const bool valid = (u32)lane < G && j < a.n_pairs;
		u64 ra = 0, rb = 0;
		bool go = valid && resolve_pair(a, j, ra, rb);
		RedN mine;
		mine.smin = mine.dot = mine.emd = 0;
		mine.jeff = mine.js = 0;
		unsigned active = __ballot_sync(0xffffffffu, go);
		if constexpr (fixed_q) {
			const unsigned char *S = reinterpret_cast<const unsigned char *>(a_hot ? B : A);
			const bool contig = a_hot ? (a.ib == nullptr) : (a.ia == nullptr);
			const u64 first_row = (a_hot ? a.b_begin : a.a_begin) + g * 32;
			u32 m0 = 0, m1 = 0, m2 = 0;
			// rows to prefetch past this group's end: the group this warp takes next (or this one again at the very end)
			const u64 g_next = g + warps_total < groups ? g + warps_total : g;
			const unsigned char *pf_next = S + ((a_hot ? a.b_begin : a.a_begin) + g_next * 32) * 1024 + lane * 32;
			scan_group<NEED, LOFF, MC2_PAIR_PREFETCH_ROWS>(S, a_hot ? a.loffB : a.loffA, 1024, active, a_hot ? rb : ra, contig,
									      first_row, fq, lane, m0, m1, m2, pf_next);
			mine.smin = m0;
			mine.dot = m1;
			mine.emd = m2;
		} else {
			while (active) {
				int pi = __ffs(active) - 1;
				active &= active - 1;
				u64 xa = __shfl_sync(0xffffffffu, ra, pi);
				u64 xb = __shfl_sync(0xffffffffu, rb, pi);
				RedN r;
				if (a_hot) { // stream B, keep A
					r = reduce_rows_fast<T, NEED>(B + xb * a.N, A + xa * a.N, slabs, lane, true);
				} else {
					r = reduce_rows_fast<T, NEED>(A + xa * a.N, B + xb * a.N, slabs, lane, b_hot);
				}
				if (lane == pi) {
					mine = r;
				}
			}
		}
		if (go) {
			Side sa = load_side(a.sbA, ra), sb = load_side(a.sbB, rb);
			if constexpr (sizeof(T) == 1) {
				// u8 path accumulated sum|p-q|; S_min = (sumP + sumQ - sad) / 2
				if (NEED & NEED_MIN) {
					mine.smin = (sa.sum + sb.sum - mine.smin) >> 1;
				}
			}
			finish_pair<RedN, false>(dm, a, j, a.N, mine, sa, sb);
		} else if (valid) {
			write_skipped(a, j);
		}
	}
}

// ------------------------------------------------------------------------------------------------
// generic path: any width, any N, log features; lane-interleaved bins, 64-bit accumulators.
// Reproduces the reference's type-dependent integer arithmetic for 32/64-bit bins.
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void reduce_rows_generic(const T *__restrict__ P, const T *__restrict__ Q, u64 N, int lane,
						    int need, u64 magP, u64 magQ, RedN &rn, RedW &rw)
{
	constexpr bool WIDE = sizeof(T) > 2;
	u64 smin = 0, dot = 0, emd = 0;
	int man = 0;
	u64 euc = 0, d1 = 0, d2 = 0, inter2 = 0, norm2 = 0;
	double dpq = 0, dpp = 0, dqq = 0, jeff = 0, js = 0;
	s64 carry = 0;
	for (u64 base = 0; base < N; base += 32) {
		u64 i = base + lane;
		bool in = i < N;
		T p = in ? P[i] : (T)0;
		T q = in ? Q[i] : (T)0;
		smin += p < q ? p : q;
		if constexpr (WIDE) {
			// same expressions as Feature.cpp so the usual arithmetic conversions (and wrap-around) match
			man += p > q ? p - q : q - p;                       // :864-867
			euc += (p - q) * (p - q);                           // :1120-1121
			dot += p * q;                                       // :1179 / :837
			d1 += p * p;                                        // :1180
			d2 += q * q;                                        // :1181
			inter2 += 2 * (p < q ? p : q);                      // :773
			long long diff = p - q;                             // :836 (intmax_t from the T-typed difference)
			norm2 += diff * diff;                               // :838
			dpq += (double)p * (double)q;
			dpp += (double)p * (double)p;
			dqq += (double)q * (double)q;
		} else {
			dot += (u32)p * (u32)q;
		}
		if (need & NEED_EMD) { // Feature.cpp:1504-1518
			s64 d = (s64)((u64)p - (u64)q);
			s64 x = d;
#pragma unroll
			for (int s = 1; s < 32; s <<= 1) {
				s64 y = shfl_up_s64(x, s);
				if (lane >= s) {
					x += y;
				}
			}
			s64 c = x + carry;
			if (in) {
				emd += (u64)(c < 0 ? -c : c);
			}
			carry += __shfl_sync(0xffffffffu, x, 31);
		}
		if ((need & NEED_LOG) && in) {
			double pp = (double)p / (double)magP;
			double pq = (double)q / (double)magQ;
			double diff = pp - pq;
			jeff += diff * log(pp / pq);                        // :1240-1260
			double avg = 0.5 * (pp + pq);
			js += pp * log(pp / avg) + pq * log(pq / avg);      // :994-1006
		}
	}
	if constexpr (WIDE) {
		rw.man = __reduce_add_sync(0xffffffffu, man);
		rw.euc = warp_sum_u64(euc);
		rw.nv_sum = warp_sum_u64(dot);
		rw.nv_d1 = warp_sum_u64(d1);
		rw.nv_d2 = warp_sum_u64(d2);
		rw.smin = warp_sum_u64(smin);
		rw.inter2 = warp_sum_u64(inter2);
		rw.emd = warp_sum_u64(emd);
		rw.norm2 = warp_sum_u64(norm2);
		rw.dpq = warp_sum_f64(dpq);
		rw.dpp = warp_sum_f64(dpp);
		rw.dqq = warp_sum_f64(dqq);
		rw.jeff = (need & NEED_LOG) ? warp_sum_f64(jeff) : 0;
		rw.js = (need & NEED_LOG) ? warp_sum_f64(js) : 0;
	} else {
		rn.smin = warp_sum_u64(smin);
		rn.dot = warp_sum_u64(dot);
		rn.emd = warp_sum_u64(emd);
		rn.jeff = (need & NEED_LOG) ? warp_sum_f64(jeff) : 0;
		rn.js = (need & NEED_LOG) ? warp_sum_f64(js) : 0;
	}
}

template <typename T>
__global__ void __launch_bounds__(256) pair_generic_kernel(const __grid_constant__ DevModel dm, const __grid_constant__ PairArgs a)
{
	constexpr bool WIDE = sizeof(T) > 2;
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	const u64 warp_id = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
	const T *A = reinterpret_cast<const T *>(a.binsA);
	const T *B = reinterpret_cast<const T *>(a.binsB);
	const u32 G = a.group <= 0 ? 32u : (u32)a.group;
	const u64 groups = (a.n_pairs + G - 1) / G;
	for (u64 g = warp_id; g < groups; g += warps_total) {
		const u64 j = g * G + lane;
		const bool valid = (u32)lane < G && j < a.n_pairs;
		u64 ra = 0, rb = 0;
		bool go = valid && resolve_pair(a, j, ra, rb);
		RedN mn;
		RedW mw;
		mn.smin = mn.dot = mn.emd = 0;
		mn.jeff = mn.js = 0;
		mw = RedW();
		unsigned active = __ballot_sync(0xffffffffu, go);
		while (active) {
			int pi = __ffs(active) - 1;
			active &= active - 1;
			u64 xa = __shfl_sync(0xffffffffu, ra, pi);
			u64 xb = __shfl_sync(0xffffffffu, rb, pi);
			u64 magA = a.sbA.mag[xa], magB = a.sbB.mag[xb];
			RedN rn;
			RedW rw;
			reduce_rows_generic<T>(A + xa * a.N, B + xb * a.N, a.N, lane, dm.need, magA, magB, rn, rw);
			if (lane == pi) {
				if constexpr (WIDE) {
					mw = rw;
				} else {
					mn = rn;
				}
			}
		}
		if (go) {
			Side sa = load_side(a.sbA, ra), sb = load_side(a.sbB, rb);
			if constexpr (WIDE) {
				finish_pair<RedW, true>(dm, a, j, a.N, mw, sa, sb);
			} else {
				finish_pair<RedN, false>(dm, a, j, a.N, mn, sa, sb);
			}
		} else if (valid) {
			write_skipped(a, j);
		}
	}
}

// ------------------------------------------------------------------------------------------------
// DivergencePoint<T>::distance (DivergencePoint.cpp:70-82): thin kernel, warp per pair
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) distance_kernel(const __grid_constant__ PairArgs a, u64 *out)
{
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	const u64 warp_id = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
	const T *A = reinterpret_cast<const T *>(a.binsA);
	const T *B = reinterpret_cast<const T *>(a.binsB);
	for (u64 j = warp_id; j < a.n_pairs; j += warps_total) {
		u64 ra = a.ia ? a.ia[j] : a.a_begin + (a.a_bc ? 0 : j);
		u64 rb = a.ib ? a.ib[j] : a.b_begin + (a.b_bc ? 0 : j);
		const T *P = A + ra * a.N, *Q = B + rb * a.N;
		u64 s = 0;
		for (u64 i = lane; i < a.N; i += 32) {
			T p = P[i], q = Q[i];
			s += p < q ? p : q;
		}
		s = warp_sum_u64(s);
		if (lane == 0) {
			u64 dist = s * 2;
			u64 mag = a.sbA.mag[ra] + a.sbB.mag[rb];
			double frac = (double)dist / (double)mag;
			out[j] = (u64)(10000.0 * (1.0 - frac * frac));
		}
	}
}

// ------------------------------------------------------------------------------------------------
// argmax / any-close reductions for get_close and merge (single CTA, inputs are 9 bytes per candidate)
// mode 0 (get_close): best = first position with the maximum dist among non-skipped; init (-1, -1); is_min = !any(close)
// mode 1 (merge):     best = last position p (sequential `best.second > dist ? best : (i,dist)`) among close ones, init (0, DBL_MIN)
// ------------------------------------------------------------------------------------------------
struct ArgOut {
	long long best;
	double best_dist;
	int is_min;
	int has; // mode 1: a close candidate was found
};

// flags_out (may be NULL): the close flags copied next to the result so that one device->host copy returns both
// Block b reduces candidates [b * chunk, min(n, (b + 1) * chunk)) into out[b] (absolute positions); one block with
// chunk >= n is the whole reduction, several blocks leave partial records for argmax_combine_kernel.
__global__ void __launch_bounds__(1024) argmax_kernel(const double *dist, const uint8_t *skipped, const uint8_t *close, u64 n,
						      int mode, ArgOut *out, uint8_t *flags_out, u64 chunk)
{
	if (flags_out) {
		for (u64 i = threadIdx.x; i < n; i += blockDim.x) {
			flags_out[i] = close[i];
		}
	}
	const u64 i_begin = (u64)blockIdx.x * chunk, i_end = i_begin + chunk < n ? i_begin + chunk : n;
	out += blockIdx.x;
	__shared__ double s_d[32];
	__shared__ long long s_i[32];
	__shared__ int s_any[32];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	double bd = mode == 0 ? -1.0 : 2.2250738585072014e-308;
	long long bi = mode == 0 ? -1 : 0;
	bool has = false; // mode 1: whether bi was set by a candidate
	int any = 0;
	for (u64 i = i_begin + threadIdx.x; i < i_end; i += blockDim.x) {
		if (skipped[i]) {
			continue;
		}
		double d = dist[i];
		any |= close[i];
		if (mode == 0) {
			if (d > bd) { // strict: the first maximum in sequence order wins
				bd = d;
				bi = (long long)i;
			}
		} else if (close[i]) {
			// sequential semantics: replace unless best.second > dist  => later ties win
			if (!(bd > d)) {
				bd = d;
				bi = (long long)i;
				has = true;
			}
		}
	}
	// combine: mode 0 prefers larger dist then smaller index; mode 1 prefers larger dist then larger index
	auto better = [&](double d2, long long i2, bool h2) {
		if (mode == 0) {
			if (i2 < 0) {
				return false;
			}
			return bi < 0 || d2 > bd || (d2 == bd && i2 < bi);
		}
		if (!h2) {
			return false;
		}
		return !has || d2 > bd || (d2 == bd && i2 > bi);
	};
	for (int s = 16; s > 0; s >>= 1) {
		double d2 = __shfl_xor_sync(0xffffffffu, bd, s);
		long long i2 = __shfl_xor_sync(0xffffffffu, bi, s);
		int h2 = __shfl_xor_sync(0xffffffffu, (int)has, s);
		any |= __shfl_xor_sync(0xffffffffu, any, s);
		if (better(d2, i2, h2 != 0)) {
			bd = d2;
			bi = i2;
			has = h2 != 0;
		}
	}
	if (lane == 0) {
		s_d[warp] = bd;
		s_i[warp] = has || mode == 0 ? bi : -2;
		s_any[warp] = any;
	}
	__syncthreads();
	if (warp == 0) {
		int nw = blockDim.x >> 5;
		bd = lane < nw ? s_d[lane] : (mode == 0 ? -1.0 : 2.2250738585072014e-308);
		long long raw = lane < nw ? s_i[lane] : (mode == 0 ? -1 : -2);
		has = mode == 1 && raw != -2;
		bi = mode == 1 && raw == -2 ? 0 : raw;
		any = lane < nw ? s_any[lane] : 0;
		for (int s = 16; s > 0; s >>= 1) {
			double d2 = __shfl_xor_sync(0xffffffffu, bd, s);
			long long i2 = __shfl_xor_sync(0xffffffffu, bi, s);
			int h2 = __shfl_xor_sync(0xffffffffu, (int)has, s);
			any |= __shfl_xor_sync(0xffffffffu, any, s);
			if (better(d2, i2, h2 != 0)) {
				bd = d2;
				bi = i2;
				has = h2 != 0;
			}
		}
		if (lane == 0) {
			out->best = bi;
			out->best_dist = bd;
			out->is_min = !any;
			out->has = mode == 0 ? (bi >= 0) : (int)has;
		}
	}
}

// partial records of consecutive candidate ranges, in range order -> the result (same tie rules as above: mode 0 keeps
// the earlier range on ties, mode 1 the later one)
__global__ void argmax_combine_kernel(const ArgOut *parts, int n_parts, int mode, ArgOut *out)
{
	if (threadIdx.x != 0) {
		return;
	}
	double bd = mode == 0 ? -1.0 : 2.2250738585072014e-308;
	long long bi = mode == 0 ? -1 : 0;
	bool has = false;
	int any = 0;
	for (int b = 0; b < n_parts; b++) {
		const ArgOut p = parts[b];
		any |= !p.is_min;
		if (!p.has) {
			continue;
		}
		if (mode == 0 ? (!has || p.best_dist > bd) : (!has || !(bd > p.best_dist))) {
			bd = p.best_dist;
			bi = p.best;
			has = true;
		}
	}
	out->best = bi;
	out->best_dist = bd;
	out->is_min = !any;
	out->has = (int)has;
}

// ------------------------------------------------------------------------------------------------
// query-vs-database sweep with fused length prefilter, cutoff and survivor compaction
// (fastcar work(), src/fastcar/FC_Runner.cpp:427-470).  A warp takes one query row r and 32 consecutive
// database rows; the query row stays hot in L1, database rows stream (from L2 when the set fits its 126 MB).
// ------------------------------------------------------------------------------------------------
struct SweepArgs {
	u64 q0, q1, d0, d1;
	int upper_only;
	double cutoff;
	u64 max_out;
	u64 *out_q, *out_d;
	double *out_score;
	u64 *counters; // [0] survivors, [1] scored pairs
	int identity;  // 0: survivors are the classifier's close pairs; 1 (regression models): pairs whose score >= min_identity
	double min_identity;
};

#define MC2_SWEEP_SPAN 4 // 32-column blocks per (query row) group in the 1 KiB-row sweep
#define MC2_SWEEP_CTAS_PER_SM 5 // resident 128-thread CTAs of the 1 KiB-row sweep: 96 registers; measured 4: 922 ms, 5: 898 ms, 6: slower (spills)
template <typename T, int NEED, bool FAST, bool ONE, bool LOFF>
__global__ void __launch_bounds__(ONE ? 128 : 256, ONE ? MC2_SWEEP_CTAS_PER_SM : 2) sweep_kernel(const __grid_constant__ DevModel dm, const __grid_constant__ PairArgs a,
						    const __grid_constant__ SweepArgs g)
{
	constexpr bool WIDE = sizeof(T) > 2;
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	const u64 warp_id = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
	const u32 slabs = (u32)(a.N * sizeof(T) / 1024);
	const T *Dm = reinterpret_cast<const T *>(a.binsA); // database = first argument of close(pts[i], query)
	const T *Qm = reinterpret_cast<const T *>(a.binsB);
	// a group = one query row x SPAN consecutive 32-column blocks: the 1 KiB form keeps the query row and its 32 prefix
	// sums in registers across the span, so their set-up (one row load + 32 IDP) is paid once per 128 pairs
	constexpr u32 SPAN = ONE ? MC2_SWEEP_SPAN : 1;
	const u64 cblocks = (g.d1 - g.d0 + 31) / 32;
	const u32 cspans32 = (u32)((cblocks + SPAN - 1) / SPAN);
	const u64 groups = (g.q1 - g.q0) * (u64)cspans32; // host guarantees groups < 2^32 per launch
	for (u64 grp = warp_id; grp < groups; grp += warps_total) {
		const u32 gr = (u32)grp / cspans32, gs = (u32)grp - gr * cspans32;
		const u64 r = g.q0 + gr;
		FixedQ fq;
		bool fq_ready = false;
#pragma unroll 1
		for (u32 h = 0; h < SPAN; h++) {
		const u64 gc = (u64)gs * SPAN + h;
		if (gc >= cblocks) {
			break;
		}
		const u64 cfirst = g.d0 + gc * 32;
		if (g.upper_only && cfirst + 31 <= r) {
			continue; // whole block at or below the diagonal
		}
		const u64 c = cfirst + lane;
		bool go = c < g.d1 && (!g.upper_only || c > r);
		if (go) { // FC_Runner.cpp:435-444: size_t truncation, window on the database length
			u64 lq = a.sbB.len[r], lc = a.sbA.len[c];
			u64 begin_length = (u64)((double)lq * g.cutoff);
			u64 end_length = (u64)((double)lq / g.cutoff);
			go = lc >= begin_length && lc <= end_length;
		}
		RedN mn;
		RedW mw;
		mn.smin = mn.dot = mn.emd = 0;
		mn.jeff = mn.js = 0;
		mw = RedW();
		unsigned active = __ballot_sync(0xffffffffu, go);
		const unsigned scored = active;
		if constexpr (FAST) {
			if constexpr (ONE) { // slabs == 1 && T == u8, picked by the host
				// the query row r and its prefix sums sit in registers for the whole 32-candidate group
				if (!fq_ready) {
					fixed_q_setup<NEED>(fq, Qm + r * a.N, lane);
					if (LOFF) {
						fq.qoff = a.loffB[r * 32 + lane];
					}
					fq_ready = true;
				}
				u32 m0 = 0, m1 = 0, m2 = 0;
				// the register ring: at the bench size (100 MB set, ~90 % L2 hits) it beat a ringless / 5-CTA variant by
				// 2.4 %; on a fully L2-resident 20 MB set it was the other way round by the same margin
				scan_group<NEED, LOFF>(reinterpret_cast<const unsigned char *>(Dm), a.loffA, 1024, active, c, true, cfirst,
							     fq, lane, m0, m1, m2);
				mn.smin = m0;
				mn.dot = m1;
				mn.emd = m2;
			} else {
				while (active) {
					int pi = __ffs(active) - 1;
					active &= active - 1;
					u64 xc = __shfl_sync(0xffffffffu, c, pi);
					RedN rr = reduce_rows_fast<T, NEED>(Dm + xc * a.N, Qm + r * a.N, slabs, lane, true);
					if (lane == pi) {
						mn = rr;
					}
				}
			}
		} else {
			while (active) {
				int pi = __ffs(active) - 1;
				active &= active - 1;
				u64 xc = __shfl_sync(0xffffffffu, c, pi);
				RedN rn;
				RedW rw;
				reduce_rows_generic<T>(Dm + xc * a.N, Qm + r * a.N, a.N, lane, dm.need, a.sbA.mag[xc], a.sbB.mag[r], rn, rw);
				if (lane == pi) {
					mn = rn;
					mw = rw;
				}
			}
		}
		int close = 0;
		double score = 0, d0;
		if (go) {
			Side sd = load_side(a.sbA, c), sq = load_side(a.sbB, r);
			int bad;
			if constexpr (WIDE) {
				bad = eval_pair<RedW, true>(dm, a.N, mw, sd, sq, nullptr, nullptr, score, d0, close);
			} else {
				if (FAST && sizeof(T) == 1 && (NEED & NEED_MIN)) {
					mn.smin = (sd.sum + sq.sum - mn.smin) >> 1;
				}
				bad = FAST ? eval_pair_fast(dm, a.N, mn, sd, sq, true, score, d0, close) // host routes !fast_epi models to FAST=false
					   : eval_pair<RedN, false>(dm, a.N, mn, sd, sq, nullptr, nullptr, score, d0, close, true);
			}
			if (bad) {
				atomicOr(a.err, bad & 1 ? 1 : 2);
			}
			if (g.identity) {
				close = score >= g.min_identity;
			}
		}
		unsigned cm = __ballot_sync(0xffffffffu, close);
		u64 base = 0;
		if (lane == 0) {
			if (cm) {
				base = atomicAdd(g.counters, (u64)__popc(cm));
			}
			if (scored) {
				atomicAdd(g.counters + 1, (u64)__popc(scored));
			}
		}
		base = __shfl_sync(0xffffffffu, base, 0);
		if (close) {
			u64 idx = base + __popc(cm & ((1u << lane) - 1));
			if (idx < g.max_out) {
				g.out_q[idx] = r;
				g.out_d[idx] = c;
				g.out_score[idx] = score;
			}
		}
		} // span
	}
}

// ------------------------------------------------------------------------------------------------
// Wide rows (several 1 KiB slabs, e.g. k = 8 uint16 = 128 KiB): the sweep with the QUERY ROW IN SHARED MEMORY.
// In sweep_kernel every (query, candidate) pair pulls both rows through L2 -> SM: 2 x 128 KiB per pair although only the
// candidate row comes from HBM.  Here a CTA owns one query row, copies it once into its shared memory (128 KB of the SM's
// 227 KB) and its 16 warps stream candidate rows against it: L2 -> SM traffic halves, HBM traffic is unchanged (one
// candidate row per pair), slabs further ahead are prefetched into L2.
// ------------------------------------------------------------------------------------------------
template <typename T, int NEED>
__device__ __forceinline__ RedN reduce_rows_smemq(const T *__restrict__ P, const unsigned char *qs, u32 slabs, int lane)
{
	u64 t_min = 0, t_dot = 0, t_emd = 0;
	int carry = 0;
	const char *pp = reinterpret_cast<const char *>(P) + lane * 32;
	const unsigned char *qq = qs + lane * 32;
	Row8 pv = ld_row_stream(pp);
#pragma unroll 1
	for (u32 s = 0; s < slabs; s++) {
		Row8 pn = pv;
		if (s + 1 < slabs) {
			pn = ld_row_stream(pp + (size_t)(s + 1) * 1024);
		}
		if (s + MC2_SLAB_PREFETCH < slabs) {
			asm volatile("prefetch.global.L2 [%0];" ::"l"(pp + (size_t)(s + MC2_SLAB_PREFETCH) * 1024));
		}
		Row8 qv;
		const uint4 q0 = *reinterpret_cast<const uint4 *>(qq + (size_t)s * 1024);
		const uint4 q1 = *reinterpret_cast<const uint4 *>(qq + (size_t)s * 1024 + 16);
		qv.w[0] = q0.x; qv.w[1] = q0.y; qv.w[2] = q0.z; qv.w[3] = q0.w;
		qv.w[4] = q1.x; qv.w[5] = q1.y; qv.w[6] = q1.z; qv.w[7] = q1.w;
		u32 a_min = 0, lo = 0, hi = 0, e = 0;
		slab_reduce<T, NEED>(pv, qv, (NEED & NEED_EMD) ? lane_sum<T>(qv) : 0, carry, a_min, lo, hi, e);
		t_min += a_min;
		t_dot += (u64)lo + ((u64)hi << 8);
		t_emd += e;
		pv = pn;
	}
	RedN r;
	r.smin = (NEED & NEED_MIN) ? warp_sum_u64(t_min) : 0;
	r.dot = (NEED & NEED_DOT) ? warp_sum_u64(t_dot) : 0;
	r.emd = (NEED & NEED_EMD) ? warp_sum_u64(t_emd) : 0;
	r.jeff = r.js = 0;
	return r;
}

template <typename T, int NEED>
__global__ void __launch_bounds__(512, 1) sweep_wide_kernel(const __grid_constant__ DevModel dm, const __grid_constant__ PairArgs a,
							    const __grid_constant__ SweepArgs g)
{
	extern __shared__ __align__(16) unsigned char qs[];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
	const u64 row_bytes = a.N * sizeof(T);
	const u32 slabs = (u32)(row_bytes / 1024);
	const T *Dm = reinterpret_cast<const T *>(a.binsA); // database = first argument of close(pts[i], query)
	const T *Qm = reinterpret_cast<const T *>(a.binsB);
	u64 scored = 0;
	for (u64 r = g.q0 + blockIdx.x; r < g.q1; r += gridDim.x) {
		__syncthreads(); // the previous query row is no longer being read
		const uint4 *src = reinterpret_cast<const uint4 *>(Qm + r * a.N);
		for (u32 i = threadIdx.x; i < row_bytes / 16; i += blockDim.x) {
			reinterpret_cast<uint4 *>(qs)[i] = __ldg(src + i);
		}
		__syncthreads();
		const Side sq = load_side(a.sbB, r);
		// FC_Runner.cpp:435-444: size_t truncation, window on the database length
		const u64 begin_length = (u64)((double)sq.len * g.cutoff), end_length = (u64)((double)sq.len / g.cutoff);
		u64 c0 = g.d0;
		if (g.upper_only && r + 1 > c0) {
			c0 = r + 1;
		}
		for (u64 c = c0 + warp; c < g.d1; c += nwarps) {
			const u64 lc = a.sbA.len[c];
			if (lc < begin_length || lc > end_length) {
				continue; // warp-uniform
			}
			scored++;
			RedN mn = reduce_rows_smemq<T, NEED>(Dm + c * a.N, qs, slabs, lane);
			if (lane == 0) {
				const Side sd = load_side(a.sbA, c);
				if (sizeof(T) == 1 && (NEED & NEED_MIN)) {
					mn.smin = (sd.sum + sq.sum - mn.smin) >> 1;
				}
				double score = 0, d0v;
				int close = 0;
				const int bad = eval_pair_fast(dm, a.N, mn, sd, sq, true, score, d0v, close);
				if (bad) {
					atomicOr(a.err, bad & 1 ? 1 : 2);
				}
				if (g.identity) {
					close = score >= g.min_identity;
				}
				if (close) {
					const u64 idx = atomicAdd(g.counters, 1ULL);
					if (idx < g.max_out) {
						g.out_q[idx] = r;
						g.out_d[idx] = c;
						g.out_score[idx] = score;
					}
				}
			}
		}
	}
	if (lane == 0 && scored) {
		atomicAdd(g.counters + 1, scored);
	}
}

// ------------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------------
static int grid_for(mc2_ctx *ctx, u64 n_pairs, int warps_per_cta, int ctas_per_sm, int group = 32)
{
	u64 groups = (n_pairs + group - 1) / group;
	u64 want = (groups + warps_per_cta - 1) / warps_per_cta;
	u64 cap = (u64)ctx->sm_count * ctas_per_sm;
	u64 g = want < cap ? want : cap;
	return (int)(g ? g : 1);
}

template <typename T, bool ONE, bool LOFF = false>
static void launch_fast_need(int need, int grid, cudaStream_t st, const DevModel &dm, const PairArgs &a)
{
	switch (need & 7) {
#define CASE(n)                                                         \
	case n:                                                         \
		pair_fast_kernel<T, n, ONE, LOFF><<<grid, ONE ? 128 : 256, 0, st>>>(dm, a); \
		break;
		CASE(0)
		CASE(1)
		CASE(2)
		CASE(3)
		CASE(4)
		CASE(5)
		CASE(6)
		CASE(7)
#undef CASE
	}
}

int launch_pair_score(mc2_ctx *ctx, const DevModel &dm, const PairArgs &a_in)
{
	if (a_in.n_pairs == 0) {
		return MC2_OK;
	}
	PairArgs a = a_in;
	const u64 row_bytes = a.N * (u64)a.eb;
	// a warp handles `group` pairs one after the other; when rows are wide (many 1 KiB slabs each) and the batch is small,
	// 32 pairs per warp leaves most of the GPU idle (5 000 pairs of 128 KiB rows = 157 busy warps): shrink the group until
	// there are about two warps' worth of groups per resident warp slot
	{
		const u64 slots = (u64)ctx->sm_count * 16;
		int group = 32;
		while (group > 1 && row_bytes > 1024 && (a.n_pairs + group - 1) / group < 2 * slots) {
			group >>= 1;
		}
		a.group = group;
	}
	const bool fast = a.eb <= 2 && row_bytes % 1024 == 0 && !(dm.need & NEED_LOG) && a.max_sum < (1ULL << 26);
	prof_begin(ctx, 2);
	if (fast) {
		int grid = grid_for(ctx, a.n_pairs, 8, 8, a.group);
		const int grid_one = grid_for(ctx, a.n_pairs, 4, MC2_PAIR_CTAS_PER_SM * 4); // 128-thread CTAs, four waves
		const bool one = a.eb == 1 && row_bytes == 1024 && ((a.a_bc && !a.ia) || (a.b_bc && !a.ib));
		if (one && a.loffA && a.loffB && (dm.need & NEED_EMD)) {
			launch_fast_need<uint8_t, true, true>(dm.need, grid_one, ctx->stream, dm, a);
		} else if (one) {
			launch_fast_need<uint8_t, true>(dm.need, grid_one, ctx->stream, dm, a);
		} else if (a.eb == 1) {
			launch_fast_need<uint8_t, false>(dm.need, grid, ctx->stream, dm, a);
		} else {
			launch_fast_need<uint16_t, false>(dm.need, grid, ctx->stream, dm, a);
		}
	} else {
		int grid = grid_for(ctx, a.n_pairs, 8, 8, a.group);
		switch (a.eb) {
		case 1: pair_generic_kernel<uint8_t><<<grid, 256, 0, ctx->stream>>>(dm, a); break;
		case 2: pair_generic_kernel<uint16_t><<<grid, 256, 0, ctx->stream>>>(dm, a); break;
		case 4: pair_generic_kernel<uint32_t><<<grid, 256, 0, ctx->stream>>>(dm, a); break;
		case 8: pair_generic_kernel<unsigned long long><<<grid, 256, 0, ctx->stream>>>(dm, a); break;
		default: set_error("elem_bytes must be 1, 2, 4 or 8"); return MC2_ERR_ARG;
		}
	}
	prof_end(ctx);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_argmax(mc2_ctx *ctx, const double *dist, const uint8_t *skipped, const uint8_t *close, u64 n, int mode, void *d_out,
		  uint8_t *d_flags_out)
{
	prof_begin(ctx, 4);
	if (n < 32768 || d_flags_out) {
		argmax_kernel<<<1, 1024, 0, ctx->stream>>>(dist, skipped, close, n, mode, reinterpret_cast<ArgOut *>(d_out), d_flags_out, n);
	} else {
		// long scans (10^5 .. 10^6 candidates): up to 96 blocks leave partial records in the result slot's spare bytes
		// (d_out is the context's 4 KB slot; the result and the error word use its first 128 bytes)
		const u64 chunk = n / 96 + 1 > 8192 ? n / 96 + 1 : 8192;
		const int parts = (int)((n + chunk - 1) / chunk);
		ArgOut *d_parts = reinterpret_cast<ArgOut *>(reinterpret_cast<char *>(d_out) + 128);
		argmax_kernel<<<parts, 1024, 0, ctx->stream>>>(dist, skipped, close, n, mode, d_parts, nullptr, chunk);
		argmax_combine_kernel<<<1, 32, 0, ctx->stream>>>(d_parts, parts, mode, reinterpret_cast<ArgOut *>(d_out));
		ctx->launches++;
	}
	prof_end(ctx);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_distance(mc2_ctx *ctx, const PairArgs &a, u64 *d_out)
{
	if (a.n_pairs == 0) {
		return MC2_OK;
	}
	u64 want = (a.n_pairs + 7) / 8;
	u64 cap = (u64)ctx->sm_count * 8;
	int grid = (int)(want < cap ? want : cap);
	switch (a.eb) {
	case 1: distance_kernel<uint8_t><<<grid, 256, 0, ctx->stream>>>(a, d_out); break;
	case 2: distance_kernel<uint16_t><<<grid, 256, 0, ctx->stream>>>(a, d_out); break;
	case 4: distance_kernel<uint32_t><<<grid, 256, 0, ctx->stream>>>(a, d_out); break;
	case 8: distance_kernel<unsigned long long><<<grid, 256, 0, ctx->stream>>>(a, d_out); break;
	default: set_error("elem_bytes must be 1, 2, 4 or 8"); return MC2_ERR_ARG;
	}
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

template <typename T, bool ONE, bool LOFF = false>
static void launch_sweep_fast(int need, int grid, cudaStream_t st, const DevModel &dm, const PairArgs &a, const SweepArgs &g)
{
	switch (need & 7) {
#define CASE(n)                                                               \
	case n:                                                               \
		sweep_kernel<T, n, true, ONE, LOFF><<<grid, ONE ? 128 : 256, 0, st>>>(dm, a, g); \
		break;
		CASE(0)
		CASE(1)
		CASE(2)
		CASE(3)
		CASE(4)
		CASE(5)
		CASE(6)
		CASE(7)
#undef CASE
	}
}

template <typename T>
static void launch_sweep_wide(int need, int grid, size_t smem, cudaStream_t st, const DevModel &dm, const PairArgs &a, const SweepArgs &g)
{
	switch (need & 7) {
#define CASE(n)                                                                                                  \
	case n:                                                                                                  \
		cudaFuncSetAttribute(sweep_wide_kernel<T, n>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
		sweep_wide_kernel<T, n><<<grid, 512, smem, st>>>(dm, a, g);                                       \
		break;
		CASE(0)
		CASE(1)
		CASE(2)
		CASE(3)
		CASE(4)
		CASE(5)
		CASE(6)
		CASE(7)
#undef CASE
	}
}

int launch_all_pairs(mc2_ctx *ctx, const DevModel &dm, const mc2_hset *q, u64 q0, u64 q1, const mc2_hset *d, u64 d0, u64 d1,
		     int upper_only, double cutoff, u64 max_out, u64 *d_out_q, u64 *d_out_d, double *d_out_score,
		     u64 *d_counters, int identity, double min_identity)
{
	// uint8 / uint16 rows of whole 1 KiB slabs with a model the fast epilogue covers: 64 x 256 pair tiles
	// (tile_sweep.cu).  Its operand pass may still find the rows unfit (a uint16 bin above 255, a bin below the
	// pseudo-count): nothing has been written then, and the row-streaming kernels below take the call.
	if (tile_sweep_supported(dm, q, d, identity)) {
		const int rc = launch_tile_sweep(ctx, dm, dm.need & 7, q, q0, q1, d, d0, d1, upper_only, cutoff, max_out, d_out_q, d_out_d,
						 d_out_score, d_counters, nullptr, nullptr, nullptr, identity, min_identity);
		if (rc != MC2_ERR_UNSUPPORTED) {
			return rc;
		}
	}
	PairArgs a;
	memset(&a, 0, sizeof a);
	a.binsA = d->bins;
	a.binsB = q->bins;
	a.sbA = Sideband{d->mag, d->sum, d->sumsq, d->len};
	a.sbB = Sideband{q->mag, q->sum, q->sumsq, q->len};
	a.N = q->N;
	a.eb = q->eb;
	a.err = ctx->d_err;
	a.max_sum = q->max_sum > d->max_sum ? q->max_sum : d->max_sum;
	if ((dm.need & NEED_EMD) && ensure_lane_off(ctx, d) == MC2_OK && ensure_lane_off(ctx, q) == MC2_OK) {
		a.loffA = d->lane_off_valid ? d->lane_off : nullptr;
		a.loffB = q->lane_off_valid ? q->lane_off : nullptr;
	}
	SweepArgs g;
	g.q0 = q0;
	g.q1 = q1;
	g.d0 = d0;
	g.d1 = d1;
	g.upper_only = upper_only;
	g.cutoff = cutoff;
	g.max_out = max_out;
	g.out_q = d_out_q;
	g.out_d = d_out_d;
	g.out_score = d_out_score;
	g.counters = d_counters;
	g.identity = identity;
	g.min_identity = min_identity;
	const u64 groups = (q1 - q0) * ((d1 - d0 + 31) / 32);
	u64 want = (groups + 7) / 8, cap = (u64)ctx->sm_count * 8;
	int grid = (int)(want < cap ? want : cap);
	// 1 KiB rows: 128-thread CTAs, four waves of the resident set (groups differ in cost: diagonal, length window)
	const u64 groups_one = (q1 - q0) * ((((d1 - d0 + 31) / 32) + MC2_SWEEP_SPAN - 1) / MC2_SWEEP_SPAN);
	const u64 want_one = (groups_one + 3) / 4, cap_one = (u64)ctx->sm_count * MC2_SWEEP_CTAS_PER_SM * 4;
	const int grid_one = (int)(want_one < cap_one ? want_one : cap_one);
	const u64 row_bytes = a.N * (u64)a.eb;
	const bool fast = a.eb <= 2 && row_bytes % 1024 == 0 && !(dm.need & NEED_LOG) && a.max_sum < (1ULL << 26) && dm.fast_epi;
	prof_begin(ctx, 3);
	if (fast) {
		if (a.eb == 1 && row_bytes == 1024 && a.loffA && a.loffB && (dm.need & NEED_EMD)) {
			launch_sweep_fast<uint8_t, true, true>(dm.need, grid_one, ctx->stream, dm, a, g);
		} else if (a.eb == 1 && row_bytes == 1024) {
			launch_sweep_fast<uint8_t, true>(dm.need, grid_one, ctx->stream, dm, a, g);
		} else if (row_bytes <= 200 * 1024) {
			// wide rows that fit shared memory: one CTA per query row, query row on chip (see sweep_wide_kernel)
			const u64 nq = q1 - q0, capw = (u64)ctx->sm_count * 8;
			const int gridw = (int)(nq < capw ? nq : capw);
			if (a.eb == 1) {
				launch_sweep_wide<uint8_t>(dm.need, gridw, (size_t)row_bytes, ctx->stream, dm, a, g);
			} else {
				launch_sweep_wide<uint16_t>(dm.need, gridw, (size_t)row_bytes, ctx->stream, dm, a, g);
			}
		} else if (a.eb == 1) {
			launch_sweep_fast<uint8_t, false>(dm.need, grid, ctx->stream, dm, a, g);
		} else {
			launch_sweep_fast<uint16_t, false>(dm.need, grid, ctx->stream, dm, a, g);
		}
	} else {
		switch (a.eb) {
		case 1: sweep_kernel<uint8_t, 0, false, false, false><<<grid, 256, 0, ctx->stream>>>(dm, a, g); break;
		case 2: sweep_kernel<uint16_t, 0, false, false, false><<<grid, 256, 0, ctx->stream>>>(dm, a, g); break;
		case 4: sweep_kernel<uint32_t, 0, false, false, false><<<grid, 256, 0, ctx->stream>>>(dm, a, g); break;
		case 8: sweep_kernel<unsigned long long, 0, false, false, false><<<grid, 256, 0, ctx->stream>>>(dm, a, g); break;
		default: set_error("elem_bytes must be 1, 2, 4 or 8"); return MC2_ERR_ARG;
		}
	}
	prof_end(ctx);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

// ------------------------------------------------------------------------------------------------
// Resident scan server (see ScanMailbox in mc2_internal.cuh): Trainer<T>::get_close (src/cluster/Trainer.cpp:23-71) for
// small candidate lists without a launch per call.  One CTA of 16 warps; a warp scores one candidate at a time with the
// same row reduction and the same fp64 epilogue as pair_fast_kernel, the CTA reduces the first maximum of the first
// combo value over the in-window candidates (strict >, initial -1: Trainer.cpp:52-56) and the close marks.
// The server leaves after MC2_SCAN_IDLE_NS without a request, so nothing that waits for an idle device (cudaFree,
// cudaMalloc) waits longer than that.
// ------------------------------------------------------------------------------------------------
#define MC2_SCAN_IDLE_NS 300000ull
__device__ __forceinline__ unsigned long long ld_sys_u64(const volatile unsigned long long *p)
{
	unsigned long long v;
	asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ unsigned long long global_ns()
{
	unsigned long long t;
	asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
	return t;
}

template <typename T>
__global__ void __launch_bounds__(512, 1) scan_server_kernel(const __grid_constant__ DevModel dm, ScanMailbox *mb, u64 first_seq)
{
	__shared__ unsigned long long s_hdr[64];      // the request header
	__shared__ unsigned long long s_cand[MC2_SCAN_CAP];
	__shared__ double s_dist[MC2_SCAN_CAP];
	__shared__ unsigned char s_flag[MC2_SCAN_CAP]; // 1 close, 2 skipped / not scored
	__shared__ double s_bd[16];
	__shared__ long long s_bi[16];
	__shared__ int s_any[16], s_err, s_go;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	constexpr int NW = 16;
	u64 last = first_seq - 1;
	for (;;) {
		if (warp == 0) {
			// every poll fetches the whole header with one coalesced read (16 bytes per lane); it is taken when its six
			// sequence copies agree
			const unsigned long long t0 = global_ns();
			int go = 0;
			for (;;) {
				unsigned long long vx, vy;
				asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(vx), "=l"(vy) : "l"(&mb->w[2 * lane]) : "memory");
				const unsigned long long s0 = __shfl_sync(0xffffffffu, vx, 0);
				const bool whole = __shfl_sync(0xffffffffu, vy, 7) == s0 && __shfl_sync(0xffffffffu, vy, 11) == s0 &&
						   __shfl_sync(0xffffffffu, vy, 15) == s0 && __shfl_sync(0xffffffffu, vy, 23) == s0 &&
						   __shfl_sync(0xffffffffu, vy, 31) == s0;
				if (s0 != last && whole) {
					s_hdr[2 * lane] = vx;
					s_hdr[2 * lane + 1] = vy;
					go = 1;
					break;
				}
				if (__shfl_sync(0xffffffffu, vy, 3) != 0 || global_ns() - t0 > MC2_SCAN_IDLE_NS) {
					break;
				}
			}
			if (lane == 0) {
				s_go = go;
				s_err = 0;
			}
		}
		__syncthreads();
		if (!s_go) {
			break;
		}
		last = s_hdr[0];
		const u64 q_row = s_hdr[1];
		const u32 n = (u32)(s_hdr[6] & 0xFFFFFFFFull);
		const bool has_list = (s_hdr[6] >> 32) & 1, ovr = (s_hdr[6] >> 33) & 1;
		const double cutoff = __longlong_as_double((long long)s_hdr[5]);
		if (has_list) {
			if ((s_hdr[6] >> 34) & 1) { // the ids travel in the header, two 32-bit row numbers per word
				if (threadIdx.x < n) {
					const unsigned long long wv = s_hdr[scan_id_word((int)threadIdx.x >> 1)];
					s_cand[threadIdx.x] = (threadIdx.x & 1) ? (wv >> 32) : (wv & 0xFFFFFFFFull);
				}
			} else {
				for (u32 j = threadIdx.x; j < n; j += blockDim.x) {
					s_cand[j] = ld_sys_u64(&mb->cand[j]);
				}
			}
			__syncthreads();
		}
		const u64 N = s_hdr[14];
		const u32 slabs = (u32)(N * sizeof(T) / 1024);
		const T *Q = reinterpret_cast<const T *>(s_hdr[8]) + q_row * N;
		const T *C = reinterpret_cast<const T *>(s_hdr[9]);
		const u64 *magQ = reinterpret_cast<const u64 *>(s_hdr[10]), *sumQ = reinterpret_cast<const u64 *>(s_hdr[11]);
		const u64 *sumsqQ = reinterpret_cast<const u64 *>(s_hdr[12]), *lenQ = reinterpret_cast<const u64 *>(s_hdr[13]);
		const u64 *magC = reinterpret_cast<const u64 *>(s_hdr[16]), *sumC = reinterpret_cast<const u64 *>(s_hdr[17]);
		const u64 *sumsqC = reinterpret_cast<const u64 *>(s_hdr[18]), *lenC = reinterpret_cast<const u64 *>(s_hdr[19]);
		Side sq;
		sq.mag = ovr ? s_hdr[2] : magQ[q_row];
		sq.len = ovr ? s_hdr[3] : lenQ[q_row];
		sq.sum = sumQ[q_row];
		sq.sumsq = sumsqQ[q_row];
		// length window on the candidate, anchored at the query (Trainer.cpp:39-48: u64 truncation)
		const u64 min_len = (u64)((double)sq.len * cutoff), max_len = (u64)((double)sq.len / cutoff);
		// a warp reduces its (up to 32) candidates one after the other, keeping candidate i's sums in lane i; then the
		// lanes run the fp64 epilogue side by side
		const u32 chunk = (n + NW - 1) / NW;
		const u32 first = (u32)warp * chunk;
		RedN mine;
		mine.smin = mine.dot = mine.emd = 0;
		mine.jeff = mine.js = 0;
		// lane i owns candidate first + i: its row index and side-band are requested now, all loads in flight together
		// (one dependent round trip to memory instead of three)
		u64 my_c = 0, my_len = 0;
		Side sc;
		sc.mag = sc.sum = sc.sumsq = sc.len = 0;
		const bool mine_valid = (u32)lane < chunk && first + lane < n;
		if (mine_valid) {
			my_c = has_list ? s_cand[first + lane] : s_hdr[4] + first + lane;
			my_len = lenC[my_c];
			sc.mag = magC[my_c];
			sc.sum = sumC[my_c];
			sc.sumsq = sumsqC[my_c];
			sc.len = my_len;
		}
		const bool my_go = mine_valid && my_len >= min_len && my_len <= max_len;
		const unsigned go_mask = __ballot_sync(0xffffffffu, my_go);
		if (my_go && chunk > 1) {
			// the warp reduces its candidates one after the other: pull all their rows towards L2 now, so only the first
			// one pays the trip to HBM
			const char *row = reinterpret_cast<const char *>(C + my_c * N);
			const u32 bytes = (u32)(N * sizeof(T)) < 4096u ? (u32)(N * sizeof(T)) : 4096u;
			for (u32 o = 0; o < bytes; o += 128) {
				asm volatile("prefetch.global.L2 [%0];" ::"l"(row + o));
			}
		}
		if (slabs == 1) {
			// 1 KiB rows: the query's slab and its lane sum are loaded once, and the next wanted candidate's row is
			// requested before the current one is reduced
			const Row8 qv = ld_row_keep(reinterpret_cast<const char *>(Q) + lane * 32);
			const int qsum = lane_sum<T>(qv);
			unsigned todo = go_mask;
			Row8 cur = qv;
			if (todo) {
				const u64 c0 = __shfl_sync(0xffffffffu, my_c, __ffs(todo) - 1);
				cur = ld_row_stream(reinterpret_cast<const char *>(C + c0 * N) + lane * 32);
			}
			while (todo) {
				const int i = __ffs(todo) - 1;
				todo &= todo - 1;
				Row8 nxt = cur;
				if (todo) {
					const u64 c1 = __shfl_sync(0xffffffffu, my_c, __ffs(todo) - 1);
					nxt = ld_row_stream(reinterpret_cast<const char *>(C + c1 * N) + lane * 32);
				}
				int carry = 0;
				u32 a_min = 0, lo = 0, hi = 0, e = 0;
				slab_reduce<T, 7>(cur, qv, qsum, carry, a_min, lo, hi, e);
				RedN r;
				r.smin = warp_sum_u64(a_min);
				r.dot = warp_sum_u64((u64)lo + ((u64)hi << 8));
				r.emd = warp_sum_u64(e);
				r.jeff = r.js = 0;
				if (lane == i) {
					mine = r;
				}
				cur = nxt;
			}
		} else {
			for (u32 i = 0; i < chunk && first + i < n; i++) {
				const u64 c = __shfl_sync(0xffffffffu, my_c, (int)i);
				if ((go_mask >> i) & 1) {
					const RedN r = reduce_rows_fast<T, 7>(C + c * N, Q, slabs, lane, true);
					if (lane == (int)i) {
						mine = r;
					}
				}
			}
		}
		if ((u32)lane < chunk && first + lane < n) {
			const u32 j = first + lane;
			if (my_go) {
				if (sizeof(T) == 1) {
					mine.smin = (sc.sum + sq.sum - mine.smin) >> 1; // 8-bit rows reduce sum |p-q|
				}
				double score, d0;
				int close;
				const int bad = eval_pair_fast(dm, N, mine, sc, sq, true, score, d0, close); // compute(candidate, query)
				if (bad) {
					atomicOr(&s_err, bad & 1 ? 1 : 2);
				}
				s_dist[j] = d0;
				s_flag[j] = close ? 1 : 0;
			} else {
				s_dist[j] = 0;
				s_flag[j] = 2;
			}
		}
		__syncthreads();
		// first maximum over the scored candidates (strict >, initial -1), any close
		double bd = -1.0;
		long long bi = -1;
		int any = 0;
		for (u32 j = threadIdx.x; j < n; j += blockDim.x) {
			const unsigned char f = s_flag[j];
			if (f & 2) {
				continue;
			}
			any |= f & 1;
			const double d = s_dist[j];
			if (d > bd) {
				bd = d;
				bi = (long long)j;
			}
		}
		for (int o = 16; o > 0; o >>= 1) {
			const double d2 = __shfl_xor_sync(0xffffffffu, bd, o);
			const long long i2 = __shfl_xor_sync(0xffffffffu, bi, o);
			any |= __shfl_xor_sync(0xffffffffu, any, o);
			if (i2 >= 0 && (bi < 0 || d2 > bd || (d2 == bd && i2 < bi))) {
				bd = d2;
				bi = i2;
			}
		}
		if (lane == 0) {
			s_bd[warp] = bd;
			s_bi[warp] = bi;
			s_any[warp] = any;
		}
		__syncthreads();
		// the answer: ONE 64-byte line written by one store instruction of eight lanes, the sequence number closing each of
		// its two 32-byte halves (the host takes the line when both agree), so no fence and no second write sit between the
		// result and its publication.  The marks of up to 192 candidates travel in the line as a bit mask; longer lists
		// go to the byte array first, fenced system-wide before the line is written.
		if (n > MC2_SCAN_MARKS_INLINE) {
			bool wrote = false;
			for (u32 w = threadIdx.x; w < (n + 7) / 8; w += blockDim.x) {
				unsigned long long v = 0;
				for (u32 b = 0; b < 8 && w * 8 + b < n; b++) {
					v |= (unsigned long long)(s_flag[w * 8 + b] & 1) << (8 * b);
				}
				reinterpret_cast<unsigned long long *>(mb->marks)[w] = v;
				wrote = true;
			}
			if (wrote) {
				__threadfence_system();
			}
			__syncthreads();
		}
		if (warp == 0) {
			bd = -1.0;
			bi = -1;
			any = 0;
			for (int w = 0; w < NW; w++) {
				any |= s_any[w];
				if (s_bi[w] >= 0 && (bi < 0 || s_bd[w] > bd || (s_bd[w] == bd && s_bi[w] < bi))) {
					bd = s_bd[w];
					bi = s_bi[w];
				}
			}
			unsigned long long v = 0;
			if (lane == 0) {
				v = (unsigned long long)bi;
			} else if (lane == 1) {
				v = (unsigned long long)__double_as_longlong(bi >= 0 ? bd : -1.0);
			} else if (lane == 2) {
				v = (unsigned long long)(any ? 0 : 1) | ((unsigned long long)(unsigned)s_err << 32);
			} else if (lane == 3 || lane == 7) {
				v = last;
			}
			// mark bits: six ballots over the first 192 flags, two per 64-bit word, kept by lanes 4..6
#pragma unroll
			for (int h = 0; h < 6; h++) {
				const u32 j = (u32)h * 32 + (u32)lane;
				const unsigned bits = __ballot_sync(0xffffffffu, j < n && j < MC2_SCAN_MARKS_INLINE && (s_flag[j] & 1));
				if (lane == 4 + (h >> 1)) {
					v |= (unsigned long long)bits << (32 * (h & 1));
				}
			}
			if (lane < 8) {
				mb->r[lane] = v;
			}
		}
		__syncthreads(); // s_flag / s_bd are rewritten by the next request
	}
	if (threadIdx.x == 0) {
		mb->running = 0;
		__threadfence_system();
	}
}

int launch_scan_server(mc2_ctx *ctx, const DevModel &dm, int eb, u64 first_seq)
{
	if (eb == 1) {
		scan_server_kernel<uint8_t><<<1, 512, 0, ctx->server_stream>>>(dm, ctx->mb, first_seq);
	} else {
		scan_server_kernel<uint16_t><<<1, 512, 0, ctx->server_stream>>>(dm, ctx->mb, first_seq);
	}
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

// exclusive prefix of the bin sums at the 32 lane boundaries of every 1 KiB uint8 row (see mc2_hset::lane_off)
__global__ void __launch_bounds__(256) lane_off_kernel(const unsigned char *__restrict__ bins, u64 n, unsigned short *__restrict__ out)
{
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	for (u64 r = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += warps_total) {
		Row8 p = ld_row_keep(bins + r * 1024 + lane * 32);
		int tot = lane_sum<uint8_t>(p), wt;
		int off = warp_excl_scan(tot, wt);
		out[r * 32 + lane] = (unsigned short)off;
	}
}

int ensure_lane_off(mc2_ctx *ctx, const mc2_hset *hc)
{
	mc2_hset *h = const_cast<mc2_hset *>(hc);
	if (h->eb != 1 || h->N != 1024 || h->max_sum >= 65536 || h->n == 0) {
		h->lane_off_valid = 0;
		return MC2_OK;
	}
	if (h->lane_off_valid) {
		return MC2_OK;
	}
	if (!h->lane_off) {
		MC2_CUDA(cudaMalloc((void **)&h->lane_off, h->n * 64));
	}
	u64 want = (h->n + 7) / 8, cap = (u64)ctx->sm_count * 8;
	int grid = (int)(want < cap ? want : cap);
	prof_begin(ctx, 5);
	lane_off_kernel<<<grid, 256, 0, ctx->stream>>>((const unsigned char *)h->bins, h->n, h->lane_off);
	prof_end(ctx);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	h->lane_off_valid = 1;
	return MC2_OK;
}

} // namespace mc2
