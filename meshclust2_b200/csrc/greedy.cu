// greedy.cu — greedy representative clustering of the identity graph over rows [begin, end) (mc2_identity_greedy_clusters,
// orchestrated in mc2_api.cu).
//
// Rows are visited in row order: a row is a representative unless an earlier representative has an edge to it, and every
// other row is assigned to the representative r < it whose edge weighs most (identity key descending, then r ascending;
// the key is topk.cu's, -0.0 equal to +0.0).  The identity sweep hands over its survivors one block of query rows Q =
// [qb, qe) at a time, in row order, and an edge (r, c), r < c, arrives with the block of r.  So when Q arrives every row
// below qb is final and every edge leaving such a row has been seen: the state of the rows (GreedyRows) is all that is kept
// between blocks.  Per block, with the block's edges bucketed by c (topk.cu's count and scatter, keyed by d):
//   greedy_resolve_kernel  decides the rows of Q in rounds of one cooperative launch.  A row that an earlier block's
//                          representative reaches (rep[c] set) is a member at once; otherwise it walks its bucket from a
//                          per-row cursor: a representative in-neighbour makes it a member, a member moves the cursor on, an
//                          undecided one ends the walk until the next round (after a look-ahead: a representative further
//                          on makes it a member now), the end of the bucket makes it a representative.
//                          A status only ever moves from undecided to final, so a read that does or does not see this
//                          round's writes gives the sequential result either way; the smallest undecided row always
//                          completes its walk, so at most |Q| rounds run, and the cursor passes each edge once.  Nothing waits
//                          on another thread inside a round.
//   greedy_assign_kernel   one warp per database row of (qb, end) with a bucket: the best in-edge from a representative of Q,
//                          merged into the row's best so far.  One writer per row and a total order: the result does not
//                          depend on block sizes.
// greedy_finish_kernel then writes the outputs and counts the representatives.  Status loads and stores are relaxed
// device-scope atomics, as in components.cu.
#include "mc2_internal.cuh"
#include <cooperative_groups.h>
#include <cuda/atomic>

namespace cg = cooperative_groups;

namespace mc2 {

static constexpr int kGrThreads = 256;
static constexpr u32 kUndecided = 0, kRep = 1, kMember = 2, kNoRep = 0xffffffffu;

__device__ __forceinline__ u32 gr_load(u32 *p)
{
	return cuda::atomic_ref<u32, cuda::thread_scope_device>(*p).load(cuda::memory_order_relaxed);
}

__device__ __forceinline__ void gr_store(u32 *p, u32 v)
{
	cuda::atomic_ref<u32, cuda::thread_scope_device>(*p).store(v, cuda::memory_order_relaxed);
}

// the identity key of topk.cu: the bits of a non-negative double, -0.0 mapped to +0.0, order like the values
__device__ __forceinline__ u64 gr_key(double v)
{
	return v == 0.0 ? 0ull : (u64)__double_as_longlong(v);
}

// (key ka, row ra) is a better in-edge than (kb, rb)
__device__ __forceinline__ bool gr_better(u64 ka, u64 ra, u64 kb, u64 rb)
{
	return ka > kb || (ka == kb && ra < rb);
}

__global__ void __launch_bounds__(kGrThreads) greedy_init_kernel(GreedyRows g, u64 n)
{
	for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
		g.status[i] = kUndecided;
		g.cursor[i] = 0;
		g.rep[i] = kNoRep;
	}
}

// rows [qb, qb + rows) of the block (absolute; state relative to begin); bucket j = the in-edges of row qb + j, query rows
// br[off[j] .. off[j + 1]).  remain: three flags, zero at launch; round k raises flag k mod 3 while a row stays undecided and
// clears flag k + 1 mod 3 for the next round (its last reader passed the barrier of round k - 1).
__global__ void __launch_bounds__(kGrThreads) greedy_resolve_kernel(const u64 *__restrict__ off, const u64 *__restrict__ br, u64 qb,
								     u64 rows, u64 begin, GreedyRows g, u32 *remain)
{
	cg::grid_group grid = cg::this_grid();
	const u64 stride = (u64)gridDim.x * blockDim.x, c0 = qb - begin;
	for (u32 round = 0;; round++) {
		if (grid.thread_rank() == 0) {
			gr_store(remain + (round + 1) % 3, 0);
		}
		bool left = false;
		for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < rows; j += stride) {
			const u64 c = c0 + j;
			if (gr_load(g.status + c) != kUndecided) {
				continue;
			}
			u32 s = kMember;
			if (g.rep[c] == kNoRep) {
				const u64 b = off[j], e1 = off[j + 1];
				u64 e = b + g.cursor[c];
				u32 rs = kMember;
				for (; e < e1; e++) {
					rs = gr_load(g.status + (br[e] - begin));
					if (rs != kMember) {
						break;
					}
				}
				g.cursor[c] = (u32)(e - b);
				s = e == e1 ? kRep : (rs == kRep ? kMember : kUndecided);
				// stopped at an undecided in-neighbour: a representative further on decides the row now (the cursor
				// stays, so a row still undecided waits for the same in-neighbour next round)
				for (u64 f = e + 1; s == kUndecided && f < e1; f++) {
					if (gr_load(g.status + (br[f] - begin)) == kRep) {
						s = kMember;
					}
				}
			}
			if (s == kUndecided) {
				left = true;
			} else {
				gr_store(g.status + c, s);
			}
		}
		if (left) {
			gr_store(remain + round % 3, 1);
		}
		grid.sync();
		if (gr_load(remain + round % 3) == 0) {
			return;
		}
	}
}

// database rows qb + j, j in [1, rows): the best in-edge (bid, br, bstr) of bucket j whose query row is a representative,
// merged into the row's best (an earlier block's representative is smaller, so it wins a tie).  bstr NULL: strand 0.
__global__ void __launch_bounds__(kGrThreads) greedy_assign_kernel(const u64 *__restrict__ off, const double *__restrict__ bid,
								    const u64 *__restrict__ br, const int8_t *__restrict__ bstr, u64 qb,
								    u64 rows, u64 begin, GreedyRows g)
{
	const u32 lane = threadIdx.x & 31u;
	const u64 warps = (u64)gridDim.x * (blockDim.x / 32);
	for (u64 j = 1 + ((u64)blockIdx.x * blockDim.x + threadIdx.x) / 32; j < rows; j += warps) {
		const u64 b = off[j], e1 = off[j + 1];
		if (b == e1) {
			continue;
		}
		u64 key = 0, r = ~0ull, at = ~0ull;
		for (u64 e = b + lane; e < e1; e += 32) {
			const u64 q = br[e];
			if (gr_load(g.status + (q - begin)) == kRep) {
				const u64 k = gr_key(bid[e]);
				if (at == ~0ull || gr_better(k, q, key, r)) {
					key = k;
					r = q;
					at = e;
				}
			}
		}
#pragma unroll
		for (int s = 16; s > 0; s >>= 1) {
			const u64 ok = __shfl_down_sync(0xffffffffu, key, s), orr = __shfl_down_sync(0xffffffffu, r, s),
				  oat = __shfl_down_sync(0xffffffffu, at, s);
			if (oat != ~0ull && (at == ~0ull || gr_better(ok, orr, key, r))) {
				key = ok;
				r = orr;
				at = oat;
			}
		}
		if (lane == 0 && at != ~0ull) {
			const u64 c = qb + j - begin;
			const u32 cur = g.rep[c];
			if (cur == kNoRep || gr_better(key, r, gr_key(g.id[c]), begin + cur)) {
				g.rep[c] = (u32)(r - begin);
				g.id[c] = bid[at];
				g.str[c] = bstr ? bstr[at] : (int8_t)0;
			}
		}
	}
}

// out_rep[i] = begin + the representative of row begin + i (itself for a representative), out_id its edge's identity
// (-1.0), out_str its strand (-1); *n_reps += the representatives (one atomic per warp; whole warps run every iteration so
// the ballot sees all 32 lanes)
__global__ void __launch_bounds__(kGrThreads) greedy_finish_kernel(GreedyRows g, u64 n, u64 begin, u64 *__restrict__ out_rep,
								    double *__restrict__ out_id, int8_t *__restrict__ out_str,
								    unsigned long long *__restrict__ n_reps)
{
	const u64 stride = (u64)gridDim.x * blockDim.x;
	for (u64 base = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += stride) {
		const u64 i = base + (threadIdx.x & 31u);
		bool rep = false;
		if (i < n) {
			rep = g.status[i] == kRep;
			out_rep[i] = begin + (rep ? i : (u64)g.rep[i]);
			out_id[i] = rep ? -1.0 : g.id[i];
			out_str[i] = rep ? (int8_t)-1 : g.str[i];
		}
		const unsigned m = __ballot_sync(0xffffffffu, rep);
		if ((threadIdx.x & 31u) == 0 && m) {
			atomicAdd(n_reps, (unsigned long long)__popc(m));
		}
	}
}

// the part slot records of a staged clustering (mc2_greedy_sweep_part): 16 bytes per edge instead of the sweep's 24
__global__ void __launch_bounds__(kGrThreads) greedy_pack_kernel(const u64 *__restrict__ sq, const u64 *__restrict__ sd,
								  const double *__restrict__ ss, u64 n, u64 begin, GreedyEdge *__restrict__ out)
{
	for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
		out[i] = GreedyEdge{(u32)(sq[i] - begin), (u32)(sd[i] - begin), ss[i]};
	}
}

static int gr_grid(mc2_ctx *ctx, u64 work)
{
	const u64 want = (work + kGrThreads - 1) / kGrThreads, cap = (u64)ctx->sm_count * 8;
	return (int)(want < cap ? (want ? want : 1) : cap);
}

int launch_greedy_init(mc2_ctx *ctx, const GreedyRows &g, u64 n)
{
	if (n == 0) {
		return MC2_OK;
	}
	greedy_init_kernel<<<gr_grid(ctx, n), kGrThreads, 0, ctx->stream>>>(g, n);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_greedy_resolve(mc2_ctx *ctx, const u64 *off, const u64 *br, u64 qb, u64 rows, u64 begin, const GreedyRows &g,
			  u32 *remain)
{
	if (rows == 0) {
		return MC2_OK;
	}
	// every CTA of a cooperative launch must be resident at once
	int per_sm = 0;
	MC2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, greedy_resolve_kernel, kGrThreads, 0));
	const u64 want = (rows + kGrThreads - 1) / kGrThreads, cap = (u64)ctx->sm_count * (u64)(per_sm > 0 ? per_sm : 1);
	const int grid = (int)(want < cap ? want : cap);
	MC2_CUDA(cudaMemsetAsync(remain, 0, 3 * sizeof(u32), ctx->stream));
	GreedyRows gg = g;
	void *args[] = {(void *)&off, (void *)&br, (void *)&qb, (void *)&rows, (void *)&begin, (void *)&gg, (void *)&remain};
	MC2_CUDA(cudaLaunchCooperativeKernel((const void *)greedy_resolve_kernel, dim3(grid), dim3(kGrThreads), args, 0, ctx->stream));
	ctx->launches++;
	return MC2_OK;
}

int launch_greedy_assign(mc2_ctx *ctx, const u64 *off, const double *bid, const u64 *br, const int8_t *bstr, u64 qb, u64 rows,
			 u64 begin, const GreedyRows &g)
{
	if (rows < 2) {
		return MC2_OK;
	}
	greedy_assign_kernel<<<gr_grid(ctx, (rows - 1) * 32), kGrThreads, 0, ctx->stream>>>(off, bid, br, bstr, qb, rows, begin, g);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_greedy_finish(mc2_ctx *ctx, const GreedyRows &g, u64 n, u64 begin, u64 *out_rep, double *out_id, int8_t *out_str,
			 u64 *n_reps)
{
	MC2_CUDA(cudaMemsetAsync(n_reps, 0, 8, ctx->stream));
	if (n == 0) {
		return MC2_OK;
	}
	greedy_finish_kernel<<<gr_grid(ctx, n), kGrThreads, 0, ctx->stream>>>(g, n, begin, out_rep, out_id, out_str,
									     (unsigned long long *)n_reps);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_greedy_pack(mc2_ctx *ctx, const u64 *sq, const u64 *sd, const double *ss, u64 n, u64 begin, GreedyEdge *out)
{
	if (n == 0) {
		return MC2_OK;
	}
	greedy_pack_kernel<<<gr_grid(ctx, n), kGrThreads, 0, ctx->stream>>>(sq, sd, ss, n, begin, out);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

} // namespace mc2
