// topk.cu — per-query selection of the top-K identity search (mc2_identity_topk, orchestrated in mc2_api.cu).
//
// The unchanged identity sweep writes one block of query rows' survivors (q, d, identity), in no order, into a scratch.
// Here they are bucketed by query (a count, an exclusive scan, a scatter) and each bucket is reduced to its first K entries
// in the order (identity descending, database row ascending).  The order is total (a query meets each database row once),
// so the result depends neither on survivor order nor on how the rows were split into blocks.
//
// Selection works on the composite key (identity key, 2^32 - 1 - (d - d_begin)), larger first, where the identity key is
// the IEEE bit pattern of the (non-negative) identity with -0.0 mapped to +0.0: as unsigned integers those bits order like
// the doubles.  A bucket of at most K entries is sorted in shared memory.  A larger one goes through an exact radix select
// of 8-bit digits over the 96-bit key (identity digits first, so the database-row digits only break ties of the K-th
// identity): each pass histograms the digit of the entries that share the prefix chosen so far and picks the digit where
// the K-th entry falls; it stops as soon as every entry with the chosen prefix is needed.  The winners, exactly K, are
// gathered into shared memory and sorted there.  Passes stream the bucket from global memory (L2), so a bucket of any
// size costs shared memory for K entries only.
#include "mc2_internal.cuh"

namespace mc2 {

static constexpr int kTopkThreads = 256;
static constexpr u32 kTopkMaxK = 1024;

// survivors per block query (self pairs dropped when asked)
__global__ void __launch_bounds__(256) topk_count_kernel(const u64 *__restrict__ sq, const u64 *__restrict__ sd, u64 n, u64 qb,
							  int exclude_self, u32 *__restrict__ cnt)
{
	for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
		const u64 q = sq[i];
		if (!(exclude_self && sd[i] == q)) {
			atomicAdd(cnt + (q - qb), 1u);
		}
	}
}

// (identity, d) of each kept survivor into its query's bucket [off[q - qb], off[q - qb + 1]); cur (zeroed) is the fill cursor
__global__ void __launch_bounds__(256) topk_scatter_kernel(const u64 *__restrict__ sq, const u64 *__restrict__ sd,
							    const double *__restrict__ ss, u64 n, u64 qb, int exclude_self,
							    const u64 *__restrict__ off, u32 *__restrict__ cur, double *__restrict__ bid,
							    u64 *__restrict__ bd)
{
	for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
		const u64 q = sq[i], d = sd[i];
		if (exclude_self && d == q) {
			continue;
		}
		const u64 pos = off[q - qb] + atomicAdd(cur + (q - qb), 1u);
		bid[pos] = ss[i];
		bd[pos] = d;
	}
}

__device__ __forceinline__ u64 identity_key(double v)
{
	return v == 0.0 ? 0ull : (u64)__double_as_longlong(v);
}

// entry a = (identity key ka, row da) comes before b in the output order
__device__ __forceinline__ bool topk_before(u64 ka, u64 da, u64 kb, u64 db)
{
	return ka > kb || (ka == kb && da < db);
}

// the 96-bit key: hi = identity key, lo = 2^32 - 1 - (d - d_begin) (>= 1: the database range is below 2^32 rows).  Digit p
// (0..11) is byte 7 - p of hi for p < 8, byte 11 - p of lo after; the masks keep the first p digits.
__device__ __forceinline__ u32 key_digit(int p, u64 hi, u32 lo)
{
	return p < 8 ? (u32)(hi >> (56 - 8 * p)) & 255u : (lo >> (24 - 8 * (p - 8))) & 255u;
}

__device__ __forceinline__ u64 mask_hi(int p)
{
	return p == 0 ? 0ull : (p >= 8 ? ~0ull : ~0ull << (64 - 8 * p));
}

__device__ __forceinline__ u32 mask_lo(int p)
{
	return p <= 8 ? 0u : (p >= 12 ? ~0u : ~0u << (32 - 8 * (p - 8)));
}

// One CTA per block query (grid-stride): out row r = the first min(K, n) entries of bucket r in (identity desc, d asc)
// order, then padding (d = UINT64_MAX, identity -1.0); out_cnt[r] = min(K, n), out_hits[r] = n.
__global__ void __launch_bounds__(kTopkThreads) topk_select_kernel(const u64 *__restrict__ off, const double *__restrict__ bid,
								   const u64 *__restrict__ bd, u64 rows, u32 K, u64 d_begin,
								   u64 *__restrict__ out_d, double *__restrict__ out_id,
								   u32 *__restrict__ out_cnt, u64 *__restrict__ out_hits)
{
	__shared__ double s_id[kTopkMaxK];
	__shared__ u64 s_d[kTopkMaxK];
	__shared__ u32 hist[256];
	__shared__ u32 warp_tot[kTopkThreads / 32];
	__shared__ u32 s_digit, s_above, s_count, s_nwin;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	for (u64 row = blockIdx.x; row < rows; row += gridDim.x) {
		const u64 b = off[row], n = off[row + 1] - b;
		const double *id = bid + b;
		const u64 *dd = bd + b;
		const u32 take = n < K ? (u32)n : K;
		if (n <= K) {
			for (u32 i = tid; i < take; i += kTopkThreads) {
				s_id[i] = id[i];
				s_d[i] = dd[i];
			}
		} else {
			u64 phi = 0;
			u32 plo = 0, need = K;
			int p = 0;
			while (p < 12) {
				hist[tid] = 0;
				__syncthreads();
				const u64 mh = mask_hi(p);
				const u32 ml = mask_lo(p);
				for (u64 i = tid; i < n; i += kTopkThreads) {
					const u64 hi = identity_key(id[i]);
					const u32 lo = 0xffffffffu - (u32)(dd[i] - d_begin);
					if (((hi ^ phi) & mh) == 0 && ((lo ^ plo) & ml) == 0) {
						atomicAdd(&hist[key_digit(p, hi, lo)], 1u);
					}
				}
				__syncthreads();
				// inclusive scan over the digits from 255 down: thread t holds digit 255 - t
				const u32 c = hist[255 - tid];
				u32 incl = c;
#pragma unroll
				for (int s = 1; s < 32; s <<= 1) {
					const u32 v = __shfl_up_sync(0xffffffffu, incl, s);
					if (lane >= s) {
						incl += v;
					}
				}
				if (lane == 31) {
					warp_tot[warp] = incl;
				}
				__syncthreads();
				for (int w = 0; w < warp; w++) {
					incl += warp_tot[w];
				}
				if (incl - c < need && need <= incl) { // the K-th entry of the prefix has this digit
					s_digit = 255 - tid;
					s_above = incl - c;
					s_count = c;
				}
				__syncthreads();
				const u32 dg = s_digit;
				need -= s_above;
				if (p < 8) {
					phi |= (u64)dg << (56 - 8 * p);
				} else {
					plo |= dg << (24 - 8 * (p - 8));
				}
				p++;
				if (s_count == need) { // every entry with this prefix is a winner (always so once the key is complete)
					break;
				}
			}
			// winners: the entries whose first p digits are >= the chosen prefix, exactly K of them
			const u64 mh = mask_hi(p);
			const u32 ml = mask_lo(p);
			if (tid == 0) {
				s_nwin = 0;
			}
			__syncthreads();
			for (u64 i = tid; i < n; i += kTopkThreads) {
				const double v = id[i];
				const u64 d = dd[i];
				const u64 hi = identity_key(v) & mh;
				const u32 lo = (0xffffffffu - (u32)(d - d_begin)) & ml;
				if (hi > phi || (hi == phi && lo >= plo)) {
					const u32 slot = atomicAdd(&s_nwin, 1u);
					s_id[slot] = v;
					s_d[slot] = d;
				}
			}
		}
		// bitonic sort of the `take` entries, padded to a power of two with entries that order last
		u32 P = 1;
		while (P < take) {
			P <<= 1;
		}
		for (u32 i = take + tid; i < P; i += kTopkThreads) {
			s_id[i] = 0.0;
			s_d[i] = ~0ull;
		}
		__syncthreads();
		for (u32 size = 2; size <= P; size <<= 1) {
			for (u32 stride = size >> 1; stride > 0; stride >>= 1) {
				for (u32 i = tid; i < P / 2; i += kTopkThreads) {
					const u32 x = 2 * i - (i & (stride - 1)), y = x + stride;
					const double vx = s_id[x], vy = s_id[y];
					const u64 dx = s_d[x], dy = s_d[y];
					const u64 kx = identity_key(vx), ky = identity_key(vy);
					const bool swap = (x & size) == 0 ? topk_before(ky, dy, kx, dx) : topk_before(kx, dx, ky, dy);
					if (swap) {
						s_id[x] = vy;
						s_id[y] = vx;
						s_d[x] = dy;
						s_d[y] = dx;
					}
				}
				__syncthreads();
			}
		}
		u64 *od = out_d + row * K;
		double *oi = out_id + row * K;
		for (u32 j = tid; j < K; j += kTopkThreads) {
			const bool have = j < take;
			od[j] = have ? s_d[j] : ~0ull;
			oi[j] = have ? s_id[j] : -1.0;
		}
		if (tid == 0) {
			out_cnt[row] = take;
			out_hits[row] = n;
		}
		__syncthreads(); // shared memory is reused by the next query
	}
}

static int grid_for(mc2_ctx *ctx, u64 work, u64 per_cta, u64 ctas_per_sm)
{
	const u64 want = (work + per_cta - 1) / per_cta, cap = (u64)ctx->sm_count * ctas_per_sm;
	return (int)(want < cap ? want : cap);
}

int launch_topk_count(mc2_ctx *ctx, const u64 *sq, const u64 *sd, u64 n, u64 qb, int exclude_self, u32 *cnt)
{
	if (n == 0) {
		return MC2_OK;
	}
	topk_count_kernel<<<grid_for(ctx, n, 256, 8), 256, 0, ctx->stream>>>(sq, sd, n, qb, exclude_self, cnt);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_topk_scatter(mc2_ctx *ctx, const u64 *sq, const u64 *sd, const double *ss, u64 n, u64 qb, int exclude_self,
			const u64 *off, u32 *cur, double *bid, u64 *bd)
{
	if (n == 0) {
		return MC2_OK;
	}
	topk_scatter_kernel<<<grid_for(ctx, n, 256, 8), 256, 0, ctx->stream>>>(sq, sd, ss, n, qb, exclude_self, off, cur, bid, bd);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_topk_select(mc2_ctx *ctx, const u64 *off, const double *bid, const u64 *bd, u64 rows, u32 k_best, u64 d_begin,
		       u64 *out_d, double *out_id, u32 *out_cnt, u64 *out_hits)
{
	if (rows == 0) {
		return MC2_OK;
	}
	topk_select_kernel<<<grid_for(ctx, rows, 1, 8), kTopkThreads, 0, ctx->stream>>>(off, bid, bd, rows, k_best, d_begin, out_d,
											 out_id, out_cnt, out_hits);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

} // namespace mc2
