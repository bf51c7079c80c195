// kmer_count.cu — K1: batched k-mer histograms (sm_100a).
//
// Replaces, for a whole batch of sequences, the reference chain
//   Loader<T>::get_point            src/clutil/Loader.cpp:138-179
//   Loader<T>::fill_table           src/clutil/Loader.cpp:42-86
//   KmerHashTable::hash / wholesaleIncrementNoOverflow   src/nonltr/KmerHashTable.cpp:108-160, 236-256
//   DivergencePoint ctor (mag)      src/clutil/DivergencePoint.cpp:99-110
// hist[h] = min(max(T), init + #occurrences of k-mer h inside the segments), order independent, so the
// sequential rolling hash becomes: one thread per 16-base packed word, the k-mer index is a funnel shift
// of two consecutive big-endian 2-bit words, counts go to a shared-memory u32 histogram with atomics and
// are narrowed (saturating) to T on the way out, fused with the side-band sums K2 needs.
#include "mc2_internal.cuh"
#include <cstdlib>

namespace mc2 {

// ------------------------------------------------------------------------------------------------
// pack: 1 byte/base codes -> 2 bits/base, big-endian inside each 32-bit word (base j of a sequence sits in
// word j/16 at bits [31-2(j%16)-1, 31-2(j%16)]), validating that every in-segment byte is a code 0..3
// (KmerHashTable.cpp:138-149 throws InvalidInputException otherwise).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) pack_kernel(const char *__restrict__ codes, const u64 *__restrict__ seq_off,
						   const u64 *__restrict__ word_off, const int *__restrict__ segs,
						   const u64 *__restrict__ seg_off, u64 n, u32 *__restrict__ packed, int *err)
{
	for (u64 s = blockIdx.x; s < n; s += gridDim.x) {
		const u64 b0 = seq_off[s];
		const u64 len = seq_off[s + 1] - b0;
		const u64 w0 = word_off[s];
		const u64 nw = word_off[s + 1] - w0;
		const u64 sg0 = seg_off[s], sg1 = seg_off[s + 1];
		const unsigned char *src = reinterpret_cast<const unsigned char *>(codes) + b0;
		for (u64 w = threadIdx.x; w < nw; w += blockDim.x) {
			u32 word = 0;
			u32 badmask = 0;
			const u64 j0 = w * 16;
#pragma unroll
			for (int t = 0; t < 16; t++) {
				u64 j = j0 + t;
				u32 c = j < len ? src[j] : 0;
				badmask |= (c > 3 ? 1u : 0u) << t;
				word |= (c & 3u) << (30 - 2 * t);
			}
			packed[w0 + w] = word;
			if (badmask) {
				// only bytes inside a segment matter; binary search the (sorted, disjoint) segment list
				for (int t = 0; t < 16; t++) {
					if (!(badmask >> t & 1)) {
						continue;
					}
					long long j = (long long)(j0 + t);
					u64 lo = sg0, hi = sg1;
					while (lo < hi) {
						u64 mid = (lo + hi) >> 1;
						if (segs[2 * mid + 1] < j) {
							lo = mid + 1;
						} else {
							hi = mid;
						}
					}
					if (lo < sg1 && segs[2 * lo] <= j && j <= segs[2 * lo + 1]) {
						atomicOr(err, 4);
					}
				}
			}
		}
	}
}

int launch_pack(mc2_ctx *ctx, const char *d_codes, const u64 *d_seq_off, mc2_seqs *s)
{
	if (s->n == 0) {
		return MC2_OK;
	}
	u64 cap = (u64)ctx->sm_count * 16;
	int grid = (int)(s->n < cap ? s->n : cap);
	prof_begin(ctx, 0);
	pack_kernel<<<grid, 128, 0, ctx->stream>>>(d_codes, d_seq_off, s->word_off, s->segs, s->seg_off, s->n, s->packed,
						      ctx->d_err);
	prof_end(ctx);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

// ------------------------------------------------------------------------------------------------
// counting
// ------------------------------------------------------------------------------------------------
struct CountArgs {
	const u32 *packed;
	const u64 *word_off;
	const int *segs;
	const u64 *seg_off;
	u64 n;
	u64 seq_begin;  // first sequence of this launch (global path batches)
	int k;
	int eb;
	u64 N;
	u64 init;
	void *bins;
	u64 *mag, *sum, *sumsq, *len, *mers1;
	double *stddev;
	int *novf;
	u32 *maxc;
	u32 *gscratch;  // global path: [batch x N] u32 counts, zeroed
};

// group = the threads cooperating on one sequence: a warp (WARP=true, several sequences per CTA) or the CTA
template <bool WARP>
__device__ __forceinline__ void group_sync()
{
	if (WARP) {
		__syncwarp();
	} else {
		__syncthreads();
	}
}
template <bool WARP>
__device__ __forceinline__ int group_or(int v)
{
	if (WARP) {
		return __any_sync(0xffffffffu, v);
	}
	return __syncthreads_or(v);
}

__device__ __forceinline__ u64 block_sum_u64(u64 v, u64 *sh)
{
	// CTA-wide sum; sh: 32 u64
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
	for (int d = 16; d > 0; d >>= 1) {
		v += __shfl_xor_sync(0xffffffffu, v, d);
	}
	__syncthreads();
	if (lane == 0) {
		sh[warp] = v;
	}
	__syncthreads();
	u64 t = 0;
	for (int w = 0; w < (int)(blockDim.x >> 5); w++) {
		t += sh[w];
	}
	return t;
}
__device__ __forceinline__ u64 warp_sum_u64_shfl(u64 v)
{
#pragma unroll
	for (int d = 16; d > 0; d >>= 1) {
		v += __shfl_xor_sync(0xffffffffu, v, d);
	}
	return v;
}

template <bool WARP>
__device__ __forceinline__ u64 group_sum(u64 v, u64 *sh)
{
	if (WARP) {
		return warp_sum_u64_shfl(v);
	}
	return block_sum_u64(v, sh);
}
template <bool WARP>
__device__ __forceinline__ u32 group_max(u32 v, u64 *sh)
{
	v = __reduce_max_sync(0xffffffffu, v);
	if (WARP) {
		return v;
	}
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	__syncthreads();
	if (lane == 0) {
		sh[warp] = v;
	}
	__syncthreads();
	u32 t = 0;
	for (int w = 0; w < (int)(blockDim.x >> 5); w++) {
		t = max(t, (u32)sh[w]);
	}
	return t;
}

// count one sequence's k-mers into `hist` (shared or global u32 counters) and its 1-mers; returns per-thread partials.
// All position arithmetic is 32-bit (the reference's positions are int).  Words whose 16 k-mer starts are all inside the
// segment take a branch-free 16-way unrolled path (2 shifts + 1 atomic per k-mer); only the (at most two) edge words of a
// segment loop over their valid positions.  Per-increment overflow tracking (the atomic's return value) is needed only
// for multi-segment sequences with a narrow T: with one segment "some increment met a saturated bin" is exactly
// "some final count exceeds max(T)", which the narrowing pass sees anyway.
// one k-mer occurrence; returns the bin's previous count.  P16: two 16-bit bins per 32-bit shared word (k = 8 in 128 KB);
// the host only picks it when no sequence has 65 536 or more k-mers, so a half can never carry into its neighbour.
template <bool P16>
__device__ __forceinline__ u32 hist_add(u32 *hist, u32 idx)
{
	if (P16) {
		const u32 sh = (idx & 1u) * 16u;
		return (atomicAdd(&hist[idx >> 1], 1u << sh) >> sh) & 0xFFFFu;
	}
	return atomicAdd(&hist[idx], 1u);
}

template <bool WARP, bool GLOBAL, bool P16 = false>
__device__ __forceinline__ void count_sequence(const CountArgs &a, u64 seq, u32 *hist, int gt, int gs, u64 tmax, u32 (&m1)[4],
					       u64 &eff_len, int &novf, bool &ovf_from_bins)
{
	const u64 w0 = a.word_off[seq];
	const int nw = (int)(a.word_off[seq + 1] - w0);
	const u32 *pk = a.packed + w0;
	const int k = a.k;
	const int sh_r = 32 - 2 * k;
	const u64 sg0 = a.seg_off[seq], sg1 = a.seg_off[seq + 1];
	// per-segment overflow counts need the atomics' old values -- except in the packed 16-bit form with 16-bit (or wider)
	// output bins, where the launcher has checked that init + the longest sequence cannot reach 65 535: nothing saturates
	const bool track = (sg1 - sg0 > 1) && tmax < 0xFFFFFFFFull && !(P16 && tmax >= 0xFFFFull);
	const u32 ovf_at = tmax < 0xFFFFFFFFull && tmax >= a.init ? (u32)(tmax - a.init) : 0xFFFFFFFFu; // old >= ovf_at <=> saturated
	m1[0] = m1[1] = m1[2] = m1[3] = 0;
	eff_len = 0;
	novf = 0;
	ovf_from_bins = !track;
	for (u64 sg = sg0; sg < sg1; sg++) {
		const int s0 = a.segs[2 * sg], e0 = a.segs[2 * sg + 1];
		eff_len += (u64)(e0 - s0 + 1);
		const int last = e0 - k + 1; // last k-mer start; k-mers counted only if the segment holds >= k bases
		const bool do_k = (e0 - s0 + 1 >= k);
		int ovf = 0;
		for (int w = (s0 >> 4) + gt; w <= (e0 >> 4); w += gs) {
			const u32 cur = pk[w];
			const u32 nxt = (w + 1 < nw) ? pk[w + 1] : 0u;
			const int j0 = w << 4;
			// 1-mers over [s0, e0] (the k=1 table, Loader.cpp:144,150): 3 popcounts, A by difference
			{
				const int lo_t = max(0, s0 - j0), hi_t = min(15, e0 - j0);
				// valid fields mask on the low bit of each 2-bit field; field t sits at bits (31-2t, 30-2t)
				u32 vm = 0x55555555u & (0xFFFFFFFFu >> (2 * lo_t));
				vm &= hi_t >= 15 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> (2 * (hi_t + 1)));
				const u32 lo = cur & vm, hi = (cur >> 1) & vm;
				const u32 nT = __popc(hi & lo), nCT = __popc(lo), nGT = __popc(hi);
				m1[3] += nT;
				m1[1] += nCT - nT;
				m1[2] += nGT - nT;
				m1[0] += (u32)(hi_t - lo_t + 1) - nCT - nGT + nT;
			}
			if (!do_k) {
				continue;
			}
			const int t0 = max(0, s0 - j0), t1 = min(15, last - j0);
			if (t0 == 0 && t1 == 15) {
				if (track) {
#pragma unroll
					for (int t = 0; t < 16; t++) {
						u32 old = hist_add<P16>(hist, __funnelshift_l(nxt, cur, 2 * t) >> sh_r);
						ovf |= old >= ovf_at;
					}
				} else {
#pragma unroll
					for (int t = 0; t < 16; t++) {
						hist_add<P16>(hist, __funnelshift_l(nxt, cur, 2 * t) >> sh_r);
					}
				}
			} else {
				for (int t = t0; t <= t1; t++) {
					u32 old = hist_add<P16>(hist, __funnelshift_l(nxt, cur, 2 * t) >> sh_r);
					ovf |= old >= ovf_at;
				}
			}
		}
		// one -1 return per overflowing segment (Loader.cpp:54-56); needs every increment of the segment done
		if (track && group_or<WARP>(ovf)) {
			novf++;
		}
	}
	(void)GLOBAL;
}

// narrow counts -> T with saturation, 4 bins per thread per step; accumulate side-band partials
template <typename T>
__device__ __forceinline__ void emit4(const u32 *cnt4, u64 init, u64 tmax, T *dst, u64 &sum, u64 &sumsq, u32 &mx)
{
	T v[4];
#pragma unroll
	for (int i = 0; i < 4; i++) {
		u64 x = init + (u64)cnt4[i];
		x = x > tmax ? tmax : x;
		v[i] = (T)x;
		sum += x;
		sumsq += x * x;
		mx = max(mx, cnt4[i]);
	}
	if constexpr (sizeof(T) == 1) {
		*reinterpret_cast<uchar4 *>(dst) = make_uchar4(v[0], v[1], v[2], v[3]);
	} else if constexpr (sizeof(T) == 2) {
		*reinterpret_cast<ushort4 *>(dst) = make_ushort4(v[0], v[1], v[2], v[3]);
	} else if constexpr (sizeof(T) == 4) {
		*reinterpret_cast<uint4 *>(dst) = make_uint4(v[0], v[1], v[2], v[3]);
	} else {
		reinterpret_cast<ulonglong2 *>(dst)[0] = make_ulonglong2(v[0], v[1]);
		reinterpret_cast<ulonglong2 *>(dst)[1] = make_ulonglong2(v[2], v[3]);
	}
}

// 8-bit fast narrowing: everything in 32 bits (init <= 255, at most 4096 bins per group in shared memory)
__device__ __forceinline__ void emit4_u8(const uint4 &c, u32 init, uint8_t *dst, u32 &sum, u32 &sumsq, u32 &mx)
{
	const u32 v0 = min(c.x + init, 255u), v1 = min(c.y + init, 255u), v2 = min(c.z + init, 255u), v3 = min(c.w + init, 255u);
	const u32 packed = v0 | (v1 << 8) | (v2 << 16) | (v3 << 24);
	*reinterpret_cast<u32 *>(dst) = packed;
	sum = __dp4a(packed, 0x01010101u, sum);
	sumsq = __dp4a(packed, packed, sumsq);
	mx = max(mx, max(max(c.x, c.y), max(c.z, c.w)));
}

template <typename T, bool WARP, bool GLOBAL, bool P16 = false>
__global__ void __launch_bounds__(P16 ? 1024 : 256) count_kernel(const __grid_constant__ CountArgs a)
{
	extern __shared__ __align__(16) u32 sh_hist[];
	__shared__ u64 sh_red[32];
	const int warps = blockDim.x >> 5;
	const int gt = WARP ? (threadIdx.x & 31) : threadIdx.x;
	const int gs = WARP ? 32 : blockDim.x;
	const u64 group = WARP ? (u64)blockIdx.x * warps + (threadIdx.x >> 5) : blockIdx.x;
	const u64 groups = WARP ? (u64)gridDim.x * warps : gridDim.x;
	const u64 tmax = sizeof(T) == 8 ? ~0ULL : ((1ULL << (8 * sizeof(T))) - 1);
	const u64 N = a.N;
	u32 *hist = GLOBAL ? nullptr : (WARP ? sh_hist + (u64)(threadIdx.x >> 5) * N : sh_hist);
	// WARP mode: every warp of the CTA iterates the same number of times (no CTA-wide barriers are used)
	for (u64 seq = a.seq_begin + group; seq < a.n; seq += groups) {
		if (!WARP && !GLOBAL) {
			// pull the next sequence's packed words into L2 while this one is counted: 128 B per thread
			const u64 nx = seq + groups;
			if (nx < a.n) {
				const u64 line = a.word_off[nx] + (u64)gt * 32;
				if (line < a.word_off[nx + 1]) {
					asm volatile("prefetch.global.L2 [%0];" ::"l"(a.packed + line));
				}
			}
		}
		if (GLOBAL) {
			hist = a.gscratch + (seq - a.seq_begin) * N; // zeroed by the host before the launch
		} else {
			for (u64 b = gt * 4; b < (P16 ? N / 2 : N); b += (u64)gs * 4) {
				*reinterpret_cast<uint4 *>(hist + b) = make_uint4(0, 0, 0, 0);
			}
			group_sync<WARP>();
		}
		u32 m1[4];
		u64 eff_len;
		int novf;
		bool ovf_from_bins;
		count_sequence<WARP, GLOBAL, P16>(a, seq, hist, gt, gs, tmax, m1, eff_len, novf, ovf_from_bins);
		if (GLOBAL) {
			__threadfence();
		}
		group_sync<WARP>();
		// narrow + side-band
		u64 sum = 0, sumsq = 0;
		u32 mx = 0;
		T *dst = reinterpret_cast<T *>(a.bins) + seq * N;
		u64 t0, t1, t2, t3;
		if (WARP && sizeof(T) == 1 && a.init <= 255) {
			// warp-private shared histogram of <= 4096 bins: all partial sums fit 32 bits, one REDUX each
			u32 s32 = 0, q32 = 0;
			const u32 init32 = (u32)a.init;
			for (u32 b = (u32)gt * 4; b < (u32)N; b += 128) {
				emit4_u8(*reinterpret_cast<const uint4 *>(hist + b), init32, reinterpret_cast<uint8_t *>(dst) + b, s32, q32, mx);
			}
			sum = __reduce_add_sync(0xffffffffu, s32);
			sumsq = __reduce_add_sync(0xffffffffu, q32);
			mx = __reduce_max_sync(0xffffffffu, mx);
			t0 = __reduce_add_sync(0xffffffffu, m1[0]);
			t1 = __reduce_add_sync(0xffffffffu, m1[1]);
			t2 = __reduce_add_sync(0xffffffffu, m1[2]);
			t3 = __reduce_add_sync(0xffffffffu, m1[3]);
		} else {
			if constexpr (P16 && sizeof(T) == 2) {
				// packed counts -> packed bins: no bin can saturate (see count_sequence), so count + init is one 32-bit add
				// per two bins and 8 bins leave as one 16-byte store
				const u32 init2 = (u32)a.init * 0x10001u;
				u32 s32 = 0, mx2 = 0;
				for (u32 b = (u32)gt * 8; b < (u32)N; b += (u32)gs * 8) {
					const uint4 c = *reinterpret_cast<const uint4 *>(hist + (b >> 1));
					const u32 v[4] = {c.x + init2, c.y + init2, c.z + init2, c.w + init2};
					*reinterpret_cast<uint4 *>(dst + b) = make_uint4(v[0], v[1], v[2], v[3]);
					mx2 = __vmaxu2(mx2, __vmaxu2(__vmaxu2(c.x, c.y), __vmaxu2(c.z, c.w)));
#pragma unroll
					for (int i = 0; i < 4; i++) {
						const u32 lo = v[i] & 0xFFFFu, hi = v[i] >> 16;
						s32 = __dp2a_lo(v[i], 0x0101u, s32); // both halves, one instruction; < 2^23 per thread
						sumsq += (u64)(lo * lo) + (u64)(hi * hi);
					}
				}
				sum = s32;
				mx = max(mx2 & 0xFFFFu, mx2 >> 16);
			} else if constexpr (P16) { // 4 shared words = 8 bins per thread and step
				for (u64 b = (u64)gt * 8; b < N; b += (u64)gs * 8) {
					const uint4 c = *reinterpret_cast<const uint4 *>(hist + (b >> 1));
					u32 lo4[4] = {c.x & 0xFFFFu, c.x >> 16, c.y & 0xFFFFu, c.y >> 16};
					u32 hi4[4] = {c.z & 0xFFFFu, c.z >> 16, c.w & 0xFFFFu, c.w >> 16};
					emit4<T>(lo4, a.init, tmax, dst + b, sum, sumsq, mx);
					emit4<T>(hi4, a.init, tmax, dst + b + 4, sum, sumsq, mx);
				}
			} else {
				for (u64 b = (u64)gt * 4; b < N; b += (u64)gs * 4) {
					uint4 c = GLOBAL ? __ldcg(reinterpret_cast<const uint4 *>(hist + b)) : *reinterpret_cast<const uint4 *>(hist + b);
					u32 c4[4] = {c.x, c.y, c.z, c.w};
					emit4<T>(c4, a.init, tmax, dst + b, sum, sumsq, mx);
				}
			}
			sum = group_sum<WARP>(sum, sh_red);
			sumsq = group_sum<WARP>(sumsq, sh_red);
			mx = group_max<WARP>(mx, sh_red);
			t0 = group_sum<WARP>(m1[0], sh_red);
			t1 = group_sum<WARP>(m1[1], sh_red);
			t2 = group_sum<WARP>(m1[2], sh_red);
			t3 = group_sum<WARP>(m1[3], sh_red);
		}
		if (ovf_from_bins && eff_len > 0) { // single segment: it overflowed iff some final count exceeds max(T)
			novf = (tmax < 0xFFFFFFFFull && a.init + (u64)mx > tmax) ? 1 : 0;
		}
		if (gt == 0) {
			a.mag[seq] = sum;
			a.sum[seq] = sum;
			a.sumsq[seq] = sumsq;
			a.len[seq] = eff_len;
			a.mers1[4 * seq + 0] = 1 + t0;
			a.mers1[4 * seq + 1] = 1 + t1;
			a.mers1[4 * seq + 2] = 1 + t2;
			a.mers1[4 * seq + 3] = 1 + t3;
			a.novf[seq] = novf;
			a.maxc[seq] = mx;
			// Loader.cpp:162-171: sqrt(sum((p_i - mag/N)^2)/N) == sqrt(N*sumsq - sum^2)/N, exact integer numerator
			unsigned __int128 num = (unsigned __int128)N * sumsq - (unsigned __int128)sum * sum;
			double numd = (double)(u64)(num >> 64) * 18446744073709551616.0 + (double)(u64)num;
			a.stddev[seq] = sqrt(numd) / (double)N;
		}
		group_sync<WARP>();
	}
}

// ------------------------------------------------------------------------------------------------
// count_warp_kernel — the short-read shape (warp per sequence, u8 / u16 bins, at most 4096 bins, init <= 255), written for
// instruction count: count_kernel above spends ~1 200 warp-instructions on a 1 kb read, most of them outside the counting
// loop.  Here
//   * the warp-private histogram sits on a boundary of its own size, so a bin's shared address is
//     (funnel-shifted word & mask) | base: one 64-bit funnel shift, one LOP3 and the reduction per k-mer occurrence;
//   * words whose 16 k-mer starts all lie in the segment take the unrolled path; the at most 30 starts in the two edge
//     words of the segment are spread over the lanes instead of being looped over by one lane;
//   * the narrowing pass re-zeroes the histogram it reads, all partial sums fit 32 bits (one REDUX each);
//   * the next sequence's offsets, segment and first 64 packed words are loaded while the current one is narrowed;
//   * the eleven side-band values leave through two lane-specialised stores.
// Sequences with several segments (N runs) fall back to count_sequence() inside the same warp loop.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sts_zero4(u32 addr)
{
	asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(addr), "r"(0u) : "memory");
}
__device__ __forceinline__ uint4 lds4(u32 addr)
{
	uint4 v;
	asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
	return v;
}
__device__ __forceinline__ void reds_inc(u32 addr)
{
	asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(1u) : "memory");
}
// low 32 bits of (hi:lo) >> r, r in 0..63
__device__ __forceinline__ u32 shr64_lo(u32 hi, u32 lo, int r)
{
	return (u32)((((u64)hi << 32) | lo) >> r);
}

#define MC2_K1_MIN_CTAS 4 // CTAs of 8 warps per SM the register budget must allow (4 -> 64 registers; 5 and 6 measured no faster)
template <typename T>
__global__ void __launch_bounds__(256, MC2_K1_MIN_CTAS) count_warp_kernel(const __grid_constant__ CountArgs a)
{
	static_assert(sizeof(T) <= 2, "count_warp_kernel: u8 / u16 bins only");
	extern __shared__ __align__(16) u32 sh_hist[];
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, warps = blockDim.x >> 5;
	const u32 N = (u32)a.N, hbytes = N * 4u;
	const u32 sh0 = (u32)__cvta_generic_to_shared(sh_hist);
	const u32 hbase = ((sh0 + hbytes - 1u) & ~(hbytes - 1u)) + (u32)wid * hbytes; // the launch reserves one histogram of slack
	u32 *hist = sh_hist + ((hbase - sh0) >> 2);
	const u32 amask = hbytes - 4u; // (N - 1) << 2
	const int k = a.k;
	const int r0 = 62 - 2 * k; // (cur:nxt) >> (r0 - 2t) puts the k-mer starting at base t of cur on bits [2, 2k + 2)
	const u32 init = (u32)a.init;
	const u64 tmax = sizeof(T) == 1 ? 0xFFull : 0xFFFFull;
	const double rcpN = 1.0 / (double)N;
	const u32 n = (u32)a.n;
	// lane-specialised side-band stores: lanes 0..8 one 64-bit value each, lanes 9..10 one 32-bit value each
	u64 *p64 = lane == 0 ? a.mag : lane == 1 ? a.sum : lane == 2 ? a.sumsq : lane == 3 ? a.len
		 : lane < 8 ? a.mers1 + (lane - 4) : reinterpret_cast<u64 *>(a.stddev);
	const u32 stride64 = (lane >= 4 && lane < 8) ? 4u : 1u;
	u32 *p32 = lane == 9 ? reinterpret_cast<u32 *>(a.novf) : a.maxc;

	for (u32 b = (u32)lane * 16u; b < hbytes; b += 512u) {
		sts_zero4(hbase + b);
	}
	__syncwarp();
	const u32 groups = gridDim.x * (u32)warps; // the launcher keeps n below 2^32
	u32 seq = blockIdx.x * (u32)warps + (u32)wid;
	if (seq >= n) {
		return;
	}
	u64 w0 = a.word_off[seq], sg0 = a.seg_off[seq];
	u32 nw = (u32)(a.word_off[seq + 1] - w0), nseg = (u32)(a.seg_off[seq + 1] - sg0);
	int2 se = nseg ? *reinterpret_cast<const int2 *>(a.segs + 2 * sg0) : make_int2(0, -1);
	u32 rw0 = (u32)lane < nw ? a.packed[w0 + lane] : 0u, rw1 = (u32)lane + 32u < nw ? a.packed[w0 + 32 + lane] : 0u;
	for (;;) {
		const u32 nseq = seq + groups;
		const bool more = nseq < n && nseq > seq;
		u64 n_w0 = 0, n_w1 = 0, n_sg0 = 0, n_sg1 = 0;
		if (more) {
			n_w0 = a.word_off[nseq];
			n_w1 = a.word_off[nseq + 1];
			n_sg0 = a.seg_off[nseq];
			n_sg1 = a.seg_off[nseq + 1];
		}
		// ---- count
		u32 cC = 0, cG = 0, cT = 0; // per-lane 1-mer partials (A follows from the effective length)
		u64 eff_len = 0;
		int novf = 0;
		bool ovf_from_bins = true;
		const u32 *pk = a.packed + w0;
		if (nseg == 1 && se.x == 0 && nw <= 64u) {
			// the common shape: one segment from base 0, at most 64 words, i.e. exactly the two words this lane already
			// holds (word `lane` and word `lane + 32`); neighbours come from shuffles, nothing is loaded or looped over
			const int e0 = se.y;
			eff_len = (u64)(e0 + 1);
			const int last = e0 - k + 1;
			const int wl = last >= 0 ? (last + 1) >> 4 : 0; // words below wl have all 16 starts <= last
			const u32 first_b = __shfl_sync(0xffffffffu, rw1, 0);
			u32 nxt0 = __shfl_down_sync(0xffffffffu, rw0, 1);
			u32 nxt1 = __shfl_down_sync(0xffffffffu, rw1, 1);
			nxt0 = lane == 31 ? first_b : nxt0;
			nxt1 = lane == 31 ? 0u : nxt1;
			// 1-mers: fields 0 .. e0 - 16w of word w (none when negative, all when >= 15)
			u32 nCT = 0, nGT = 0, nT = 0;
#pragma unroll
			for (int h = 0; h < 2; h++) {
				const u32 cur = h ? rw1 : rw0;
				const int rem = e0 - ((lane + 32 * h) << 4);
				const int shn = min(max(2 * rem + 2, 0), 32);
				const u32 vm = 0x55555555u & ~(u32)(0xFFFFFFFFull >> shn);
				const u32 lo = cur & vm, hi = (cur >> 1) & vm;
				nT += __popc(hi & lo);
				nCT += __popc(lo);
				nGT += __popc(hi);
			}
			if (lane < wl) {
#pragma unroll
				for (int t = 0; t < 16; t++) {
					reds_inc((shr64_lo(rw0, nxt0, r0 - 2 * t) & amask) | hbase);
				}
			}
			if (lane + 32 < wl) {
#pragma unroll
				for (int t = 0; t < 16; t++) {
					reds_inc((shr64_lo(rw1, nxt1, r0 - 2 * t) & amask) | hbase);
				}
			}
			// the < 16 starts of word wl, one per lane
			{
				const u32 src_c = wl < 32 ? rw0 : rw1, src_n = wl + 1 < 32 ? rw0 : rw1;
				const u32 ec = __shfl_sync(0xffffffffu, src_c, wl & 31);
				u32 en = __shfl_sync(0xffffffffu, src_n, (wl + 1) & 31);
				en = wl + 1 < 64 ? en : 0u;
				if (wl < 64 && (wl << 4) + lane <= last && lane < 16) {
					reds_inc((shr64_lo(ec, en, r0 - 2 * lane) & amask) | hbase);
				}
			}
			cT = nT;
			cC = nCT - nT;
			cG = nGT - nT;
		} else if (nseg == 1) {
			const int s0 = se.x, e0 = se.y;
			eff_len = (u64)(e0 - s0 + 1);
			const int last = e0 - k + 1;
			const bool do_k = last >= s0;
			const int wf = (s0 + 15) >> 4;               // first word whose 16 starts are all >= s0
			const int wl = do_k ? (last + 1) >> 4 : 0;  // words below wl have all 16 starts <= last
			const int wb = s0 >> 4, we = e0 >> 4;
			u32 nCT = 0, nGT = 0, nT = 0;
			int it = 0;
			for (int wi = wb; wi <= we; wi += 32, it++) {
				const int w = wi + lane;
				u32 cur;
				if (wb == 0 && it < 2) {
					cur = it ? rw1 : rw0;
				} else {
					cur = w < (int)nw ? pk[w] : 0u;
				}
				u32 nxt = __shfl_down_sync(0xffffffffu, cur, 1);
				if (lane == 31) {
					nxt = w + 1 < (int)nw ? pk[w + 1] : 0u;
				}
				if (w <= we) {
					const int j0 = w << 4;
					u32 vm = 0x55555555u;
					if (j0 < s0 || j0 + 15 > e0) {
						const int lo_t = max(0, s0 - j0), hi_t = min(15, e0 - j0);
						vm &= 0xFFFFFFFFu >> (2 * lo_t);
						vm &= hi_t >= 15 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> (2 * (hi_t + 1)));
					}
					const u32 lo = cur & vm, hi = (cur >> 1) & vm;
					nT += __popc(hi & lo);
					nCT += __popc(lo);
					nGT += __popc(hi);
					if (do_k && w >= wf && w < wl) {
#pragma unroll
						for (int t = 0; t < 16; t++) {
							reds_inc((shr64_lo(cur, nxt, r0 - 2 * t) & amask) | hbase);
						}
					}
				}
			}
			if (do_k) {
				// starts outside the full words: [s0, wf*16) in front, [max(wl, wf)*16, last] behind; < 16 each
				int pos;
				bool ok;
				if (lane < 16) {
					pos = s0 + lane;
					ok = pos <= min(wf * 16 - 1, last);
				} else {
					pos = max(wl, wf) * 16 + (lane - 16);
					ok = pos <= last;
				}
				if (ok) {
					const int w = pos >> 4, t = pos & 15;
					const u32 cur = pk[w];
					const u32 nxt = w + 1 < (int)nw ? pk[w + 1] : 0u;
					reds_inc((shr64_lo(cur, nxt, r0 - 2 * t) & amask) | hbase);
				}
			}
			cT = nT;
			cC = nCT - nT;
			cG = nGT - nT;
		} else if (nseg > 1) {
			u32 m1[4];
			count_sequence<true, false, false>(a, seq, hist, lane, 32, tmax, m1, eff_len, novf, ovf_from_bins);
			cC = m1[1];
			cG = m1[2];
			cT = m1[3];
		}
		// ---- next sequence's segment and first words, in flight while this one is narrowed
		int2 n_se = make_int2(0, -1);
		u32 n_rw0 = 0, n_rw1 = 0;
		const u32 n_nw = (u32)(n_w1 - n_w0), n_nseg = (u32)(n_sg1 - n_sg0);
		if (more) {
			if (n_nseg) {
				n_se = *reinterpret_cast<const int2 *>(a.segs + 2 * n_sg0);
			}
			if ((u32)lane < n_nw) {
				n_rw0 = a.packed[n_w0 + lane];
			}
			if ((u32)lane + 32u < n_nw) {
				n_rw1 = a.packed[n_w0 + 32 + lane];
			}
		}
		__syncwarp();
		// ---- narrow (saturating) + side-band; leaves the histogram zeroed
		T *dst = reinterpret_cast<T *>(a.bins) + (u64)seq * N;
		u32 s32 = 0, q32 = 0, mx = 0;
		u64 q64 = 0;
		for (u32 b = (u32)lane * 4u; b < N; b += 128u) {
			const uint4 c = lds4(hbase + b * 4u);
			sts_zero4(hbase + b * 4u);
			mx = max(max(mx, c.x), max(max(c.y, c.z), c.w)); // two three-input maxima
			if constexpr (sizeof(T) == 1) {
				const u32 v0 = min(c.x + init, 255u), v1 = min(c.y + init, 255u), v2 = min(c.z + init, 255u),
					  v3 = min(c.w + init, 255u);
				const u32 pv = __byte_perm(__byte_perm(v0, v1, 0x0040), __byte_perm(v2, v3, 0x0040), 0x5410);
				*reinterpret_cast<u32 *>(dst + b) = pv;
				s32 = __dp4a(pv, 0x01010101u, s32);
				q32 = __dp4a(pv, pv, q32);
			} else {
				const u32 v0 = min(c.x + init, 65535u), v1 = min(c.y + init, 65535u), v2 = min(c.z + init, 65535u),
					  v3 = min(c.w + init, 65535u);
				*reinterpret_cast<uint2 *>(dst + b) = make_uint2(v0 | (v1 << 16), v2 | (v3 << 16));
				s32 += v0 + v1 + v2 + v3;
				q64 += (u64)(v0 * v0) + (u64)(v1 * v1) + (u64)(v2 * v2) + (u64)(v3 * v3);
			}
		}
		const u64 sum = __reduce_add_sync(0xffffffffu, s32);
		u64 sumsq;
		if constexpr (sizeof(T) == 1) {
			sumsq = __reduce_add_sync(0xffffffffu, q32);
		} else {
			// per lane < 2^39: reduce in two 20-bit-split halves, each total below 2^32
			const u32 ql = __reduce_add_sync(0xffffffffu, (u32)(q64 & 0xFFFFFu));
			const u32 qh = __reduce_add_sync(0xffffffffu, (u32)(q64 >> 20));
			sumsq = ((u64)qh << 20) + ql;
		}
		mx = __reduce_max_sync(0xffffffffu, mx);
		const u32 tC = __reduce_add_sync(0xffffffffu, cC), tG = __reduce_add_sync(0xffffffffu, cG),
			  tT = __reduce_add_sync(0xffffffffu, cT);
		const u64 tA = eff_len - tC - tG - tT;
		if (ovf_from_bins) { // single segment: it overflowed iff some final count exceeds max(T)
			novf = (u64)init + mx > tmax ? 1 : 0;
		}
		// Loader.cpp:162-171: sqrt(sum((p_i - mag/N)^2)/N) == sqrt(N*sumsq - sum^2)/N; here N*sumsq < 2^57, exact in 64 bits
		const double sd = sqrt((double)((u64)N * sumsq - sum * sum)) * rcpN;
		u64 v64 = sum;
		v64 = lane == 2 ? sumsq : v64;
		v64 = lane == 3 ? eff_len : v64;
		v64 = lane == 4 ? 1 + tA : v64;
		v64 = lane == 5 ? 1 + (u64)tC : v64;
		v64 = lane == 6 ? 1 + (u64)tG : v64;
		v64 = lane == 7 ? 1 + (u64)tT : v64;
		v64 = lane == 8 ? (u64)__double_as_longlong(sd) : v64;
		if (lane < 9) {
			p64[(u64)seq * stride64] = v64;
		} else if (lane < 11) {
			p32[seq] = lane == 9 ? (u32)novf : mx;
		}
		if (!more) {
			break;
		}
		__syncwarp();
		seq = nseq;
		w0 = n_w0;
		sg0 = n_sg0;
		nw = n_nw;
		nseg = n_nseg;
		se = n_se;
		rw0 = n_rw0;
		rw1 = n_rw1;
	}
}

// sums / sums of squares for a set uploaded from the host (mc2_hset_from_host)
template <typename T>
__global__ void __launch_bounds__(256) sideband_kernel(const T *__restrict__ bins, u64 n, u64 N, u64 *sum, u64 *sumsq,
						       u64 *mag, int set_mag)
{
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	for (u64 r = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += warps_total) {
		const T *row = bins + r * N;
		u64 s = 0, q = 0;
		for (u64 i = lane; i < N; i += 32) {
			u64 v = row[i];
			s += v;
			q += v * v;
		}
		s = warp_sum_u64_shfl(s);
		q = warp_sum_u64_shfl(q);
		if (lane == 0) {
			sum[r] = s;
			sumsq[r] = q;
			if (set_mag) {
				mag[r] = s;
			}
		}
	}
}

int launch_sideband(mc2_ctx *ctx, mc2_hset *h, bool set_mag)
{
	if (h->n == 0) {
		return MC2_OK;
	}
	u64 want = (h->n + 7) / 8, cap = (u64)ctx->sm_count * 8;
	int grid = (int)(want < cap ? want : cap);
	prof_begin(ctx, 5);
	switch (h->eb) {
	case 1: sideband_kernel<uint8_t><<<grid, 256, 0, ctx->stream>>>((const uint8_t *)h->bins, h->n, h->N, h->sum, h->sumsq, h->mag, set_mag); break;
	case 2: sideband_kernel<uint16_t><<<grid, 256, 0, ctx->stream>>>((const uint16_t *)h->bins, h->n, h->N, h->sum, h->sumsq, h->mag, set_mag); break;
	case 4: sideband_kernel<uint32_t><<<grid, 256, 0, ctx->stream>>>((const uint32_t *)h->bins, h->n, h->N, h->sum, h->sumsq, h->mag, set_mag); break;
	case 8: sideband_kernel<u64><<<grid, 256, 0, ctx->stream>>>((const u64 *)h->bins, h->n, h->N, h->sum, h->sumsq, h->mag, set_mag); break;
	default: set_error("elem_bytes must be 1, 2, 4 or 8"); return MC2_ERR_ARG;
	}
	prof_end(ctx);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

template <typename T>
static int launch_count_t(mc2_ctx *ctx, const mc2_seqs *s, CountArgs &a)
{
	const u64 N = a.N;
	const u64 hist_bytes = N * 4;
	const u64 avg_len = s->n ? s->total_bases / s->n : 0;
	if (hist_bytes <= 64 * 1024) {
		// shared-memory histograms
		const bool warp_mode = hist_bytes <= 16 * 1024 && avg_len <= 4096;
		if constexpr (sizeof(T) <= 2) {
			const bool legacy = getenv("MC2_K1_LEGACY") != nullptr; // A/B switch for tools/k1_bench.py
			if (warp_mode && a.init <= 255 && s->n < 0xFFFFFFFFull && !legacy) {
				int warps = (int)(32 * 1024 / hist_bytes);
				warps = warps > 8 ? 8 : (warps < 1 ? 1 : warps);
				const size_t smem = (size_t)(warps + 1) * hist_bytes; // one histogram of slack for the alignment
				MC2_CUDA(cudaFuncSetAttribute(count_warp_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
				int per_sm = 0;
				MC2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, count_warp_kernel<T>, warps * 32, smem));
				per_sm = per_sm < 1 ? 1 : per_sm;
				// one resident wave; every warp walks its sequences with the next one's loads in flight
				const u64 want = (s->n + warps - 1) / warps, cap = (u64)ctx->sm_count * per_sm;
				const int grid = (int)(want < cap ? want : cap);
				prof_begin(ctx, 1);
				count_warp_kernel<T><<<grid, warps * 32, smem, ctx->stream>>>(a);
				prof_end(ctx);
				ctx->launches++;
				MC2_CUDA(cudaGetLastError());
				return MC2_OK;
			}
		}
		if (warp_mode) {
			int warps = (int)(48 * 1024 / hist_bytes);
			warps = warps > 8 ? 8 : (warps < 1 ? 1 : warps);
			size_t smem = (size_t)warps * hist_bytes;
			u64 want = (s->n + warps - 1) / warps, cap = (u64)ctx->sm_count * 8;
			int grid = (int)(want < cap ? want : cap);
			MC2_CUDA(cudaFuncSetAttribute(count_kernel<T, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
			prof_begin(ctx, 1);
			count_kernel<T, true, false><<<grid, warps * 32, smem, ctx->stream>>>(a);
			prof_end(ctx);
		} else {
			u64 cap = (u64)ctx->sm_count * 4;
			int grid = (int)(s->n < cap ? s->n : cap);
			MC2_CUDA(cudaFuncSetAttribute(count_kernel<T, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
			prof_begin(ctx, 1);
			count_kernel<T, false, false><<<grid, 256, hist_bytes, ctx->stream>>>(a);
			prof_end(ctx);
		}
		ctx->launches++;
		MC2_CUDA(cudaGetLastError());
		return MC2_OK;
	}
	if (N * 2 <= 200 * 1024 && a.init + s->max_len <= 65535) {
		// 16-bit packed shared histogram, one 1024-thread CTA per sequence (k = 8: 128 KB of the SM's 227 KB): no bin can
		// reach 65 536 occurrences, so halves never carry; counting, narrowing and the side-band stay on chip
		const size_t smem = (size_t)N * 2;
		int grid = (int)(s->n < (u64)ctx->sm_count ? s->n : (u64)ctx->sm_count);
		MC2_CUDA(cudaFuncSetAttribute(count_kernel<T, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		prof_begin(ctx, 1);
		count_kernel<T, false, false, true><<<grid, 1024, smem, ctx->stream>>>(a);
		prof_end(ctx);
		ctx->launches++;
		MC2_CUDA(cudaGetLastError());
		return MC2_OK;
	}
	// global-memory counters, batched so the scratch stays <= 1 GiB
	u64 batch = (1ULL << 30) / hist_bytes;
	batch = batch < 1 ? 1 : batch;
	batch = batch > s->n ? s->n : batch;
	u32 *scratch = nullptr;
	MC2_CUDA(cudaMalloc(&scratch, batch * hist_bytes));
	int rc = MC2_OK;
	for (u64 b0 = 0; b0 < s->n && rc == MC2_OK; b0 += batch) {
		u64 cnt = s->n - b0 < batch ? s->n - b0 : batch;
		cudaError_t e = cudaMemsetAsync(scratch, 0, cnt * hist_bytes, ctx->stream);
		if (e != cudaSuccess) {
			rc = cuda_fail(e, "cudaMemsetAsync", __FILE__, __LINE__);
			break;
		}
		CountArgs b = a;
		b.seq_begin = b0;
		b.n = b0 + cnt;
		b.gscratch = scratch;
		u64 cap = (u64)ctx->sm_count * 4;
		int grid = (int)(cnt < cap ? cnt : cap);
		// sequences b0.. are reached by offsetting the group index through seq_begin
		b.packed = a.packed;
		prof_begin(ctx, 1);
		count_kernel<T, false, true><<<grid, 256, 0, ctx->stream>>>(b);
		prof_end(ctx);
		ctx->launches++;
		e = cudaGetLastError();
		if (e != cudaSuccess) {
			rc = cuda_fail(e, "count_kernel(global)", __FILE__, __LINE__);
		}
	}
	cudaStreamSynchronize(ctx->stream);
	cudaFree(scratch);
	return rc;
}

int launch_count(mc2_ctx *ctx, const mc2_seqs *s, int k, int eb, mc2_hset *h, u64 init_value)
{
	if (s->n == 0) {
		return MC2_OK;
	}
	CountArgs a;
	a.packed = s->packed;
	a.word_off = s->word_off;
	a.segs = s->segs;
	a.seg_off = s->seg_off;
	a.n = s->n;
	a.seq_begin = 0;
	a.k = k;
	a.eb = eb;
	a.N = 1ULL << (2 * k);
	a.init = init_value;
	a.bins = h->bins;
	a.mag = h->mag;
	a.sum = h->sum;
	a.sumsq = h->sumsq;
	a.len = h->len;
	a.mers1 = h->mers1;
	a.stddev = h->stddev;
	a.novf = h->novf;
	a.maxc = h->maxc;
	a.gscratch = nullptr;
	switch (eb) {
	case 1: return launch_count_t<uint8_t>(ctx, s, a);
	case 2: return launch_count_t<uint16_t>(ctx, s, a);
	case 4: return launch_count_t<uint32_t>(ctx, s, a);
	case 8: return launch_count_t<u64>(ctx, s, a);
	}
	set_error("elem_bytes must be 1, 2, 4 or 8");
	return MC2_ERR_ARG;
}

} // namespace mc2
