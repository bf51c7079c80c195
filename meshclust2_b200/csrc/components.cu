// components.cu — connected components of an edge set over rows [begin, end) (mc2_identity_components and
// mc2_components_merge, orchestrated in mc2_api.cu).
//
// A concurrent union-find over a uint32 parent array relative to begin.  Every hook thread finds the roots of its edge's two
// ends (path halving) and links the larger root under the smaller one with one compare-and-swap on the larger root's
// parent slot; a failed swap means that root was linked meanwhile, and the thread retries from the finds.  parent[x] <= x
// always holds: a link writes a smaller root, and halving writes an ancestor, which is smaller still.  So the root of a
// component, once every edge is hooked, is its smallest row, whatever the order in which edges arrived, how they were split
// into launches, or how the races went.  Loads and stores of parent are relaxed device-scope atomics, so a thread never
// reuses a value cached across iterations of its loops.
//
// Edges come from survivor lists of the identity sweep (q, d in absolute rows) or, for a merge, from stacked label arrays
// (row i mod n joined to its label in part i / n).  One kernel template serves both; the source is its parameter.
#include "mc2_internal.cuh"
#include <cuda/atomic>

namespace mc2 {

static constexpr int kCcThreads = 256;

__device__ __forceinline__ u32 cc_load(u32 *parent, u32 x)
{
	return cuda::atomic_ref<u32, cuda::thread_scope_device>(parent[x]).load(cuda::memory_order_relaxed);
}

__device__ __forceinline__ void cc_store(u32 *parent, u32 x, u32 v)
{
	cuda::atomic_ref<u32, cuda::thread_scope_device>(parent[x]).store(v, cuda::memory_order_relaxed);
}

// root of x with path halving: each visited node is pointed at its grandparent
__device__ __forceinline__ u32 cc_find(u32 *parent, u32 x)
{
	u32 p = cc_load(parent, x);
	while (p != x) {
		const u32 g = cc_load(parent, p);
		if (g != p) {
			cc_store(parent, x, g);
		}
		x = g;
		p = cc_load(parent, x);
	}
	return x;
}

// survivors of one sweep block: edge i = {q[i], d[i]}, absolute rows
struct PairEdges {
	const u64 *q, *d;
	u64 begin;
	__device__ __forceinline__ void get(u64 i, u32 &a, u32 &b) const
	{
		a = (u32)(q[i] - begin);
		b = (u32)(d[i] - begin);
	}
};

// n_parts stacked label arrays of n rows each: edge i = {i mod n, labels[i] - begin}
struct LabelEdges {
	const u64 *labels;
	u64 n, begin;
	__device__ __forceinline__ void get(u64 i, u32 &a, u32 &b) const
	{
		a = (u32)(i % n);
		b = (u32)(labels[i] - begin);
	}
};

__global__ void __launch_bounds__(kCcThreads) cc_init_kernel(u32 *__restrict__ parent, u64 n)
{
	for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
		parent[i] = (u32)i;
	}
}

template <typename Src>
__global__ void __launch_bounds__(kCcThreads) cc_hook_kernel(Src src, u64 n_edges, u32 *parent)
{
	for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_edges; i += (u64)gridDim.x * blockDim.x) {
		u32 a, b;
		src.get(i, a, b);
		for (;;) {
			a = cc_find(parent, a);
			b = cc_find(parent, b);
			if (a == b) {
				break;
			}
			const u32 hi = a > b ? a : b, lo = a ^ b ^ hi;
			if (atomicCAS(parent + hi, hi, lo) == hi) {
				break;
			}
		}
	}
}

// out[i] = begin + root of i; *n_roots += the roots (one atomic per warp).  Whole warps run every iteration so the ballot
// sees all 32 lanes.
__global__ void __launch_bounds__(kCcThreads) cc_flatten_kernel(u32 *parent, u64 n, u64 begin, u64 *__restrict__ out,
								 unsigned long long *__restrict__ n_roots)
{
	const u64 stride = (u64)gridDim.x * blockDim.x;
	for (u64 base = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += stride) {
		const u64 i = base + (threadIdx.x & 31u);
		bool root = false;
		if (i < n) {
			const u32 r = cc_find(parent, (u32)i);
			out[i] = begin + r;
			root = r == (u32)i;
		}
		const unsigned m = __ballot_sync(0xffffffffu, root);
		if ((threadIdx.x & 31u) == 0 && m) {
			atomicAdd(n_roots, (unsigned long long)__popc(m));
		}
	}
}

static int cc_grid(mc2_ctx *ctx, u64 work)
{
	const u64 want = (work + kCcThreads - 1) / kCcThreads, cap = (u64)ctx->sm_count * 8;
	return (int)(want < cap ? (want ? want : 1) : cap);
}

int launch_cc_init(mc2_ctx *ctx, u32 *parent, u64 n)
{
	if (n == 0) {
		return MC2_OK;
	}
	cc_init_kernel<<<cc_grid(ctx, n), kCcThreads, 0, ctx->stream>>>(parent, n);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_cc_hook_pairs(mc2_ctx *ctx, const u64 *q, const u64 *d, u64 n, u64 begin, u32 *parent)
{
	if (n == 0) {
		return MC2_OK;
	}
	cc_hook_kernel<PairEdges><<<cc_grid(ctx, n), kCcThreads, 0, ctx->stream>>>(PairEdges{q, d, begin}, n, parent);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_cc_hook_labels(mc2_ctx *ctx, const u64 *labels, u64 n_parts, u64 n, u64 begin, u32 *parent)
{
	if (n == 0 || n_parts == 0) {
		return MC2_OK;
	}
	cc_hook_kernel<LabelEdges><<<cc_grid(ctx, n_parts * n), kCcThreads, 0, ctx->stream>>>(LabelEdges{labels, n, begin}, n_parts * n,
												parent);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_cc_flatten(mc2_ctx *ctx, u32 *parent, u64 n, u64 begin, u64 *out, u64 *n_roots)
{
	MC2_CUDA(cudaMemsetAsync(n_roots, 0, 8, ctx->stream));
	if (n == 0) {
		return MC2_OK;
	}
	cc_flatten_kernel<<<cc_grid(ctx, n), kCcThreads, 0, ctx->stream>>>(parent, n, begin, out, (unsigned long long *)n_roots);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

} // namespace mc2
