// strand.cu — the other DNA strand: reverse-complement histogram sets (mc2_hset_reverse_complement) and the strand merge of
// the both-strand identity search (mc2_identity_pairs_both_strands, orchestrated in mc2_api.cu).
//
// Bin j of a row is the big-endian base-4 k-mer (A=0, C=1, G=2, T=3), so the histogram of the other strand is the
// permutation out[rc(j)] = in[j] with rc(j) = reverse_digits(j) XOR (4^k - 1), an involution.  Read along j (coalesced),
// neighbouring bins land 4^(k-1) apart in the output, and a gather through a staged row hits one shared-memory bank for
// neighbouring lanes.  The kernel splits j into h high, mid middle and l low digits, j = (hi, md, lo), and uses
// rc(hi, md, lo) = (rc_l(lo), rc_mid(md), rc_h(hi)): for a fixed md the 4^h x 4^l tile of (hi, lo) is a transpose with
// digit-reversed row and column indices.  A CTA reads the tile along lo (runs of 4^l contiguous bins), stages it in shared
// memory as 32-bit words (64-bit for uint64 bins) with one word of padding per tile row, and writes the output tile along
// its own low digits (runs of 4^h contiguous bins).  h, l <= 3, so a tile holds at most 4096 bins whatever k: rows of any
// width, wider than shared memory included, go through shared memory one tile at a time.
#include "mc2_internal.cuh"

namespace mc2 {

// reverse the nd base-4 digits of v and complement each (3 - d = d XOR 3)
__device__ __forceinline__ u64 rc_digits(u64 v, int nd)
{
	if (nd == 0) {
		return 0;
	}
	u64 r = __brevll(v) >> (64 - 2 * nd); // digit order reversed, the two bits inside each digit swapped
	r = ((r & 0x5555555555555555ull) << 1) | ((r >> 1) & 0x5555555555555555ull);
	return r ^ ((1ull << (2 * nd)) - 1);
}

template <typename T, typename W>
__global__ void __launch_bounds__(256) revcomp_kernel(const T *__restrict__ src, T *__restrict__ dst, const u64 *__restrict__ mers_in,
						      u64 *__restrict__ mers_out, u64 n, int k, int h, int l)
{
	__shared__ W tile[64 * 65];
	const int mid = k - h - l;
	const u32 sh = 1u << (2 * h), sl = 1u << (2 * l), elems = sh * sl, pitch = sl + 1;
	const u64 N = 1ull << (2 * k), tiles = 1ull << (2 * mid);
	for (u64 item = blockIdx.x; item < n * tiles; item += gridDim.x) {
		const u64 row = item >> (2 * mid), md = item & (tiles - 1);
		const T *s = src + row * N;
		T *d = dst + row * N;
		// in: j = hi 4^(k-h) + md 4^l + lo
		for (u32 e = threadIdx.x; e < elems; e += blockDim.x) {
			const u32 hi = e >> (2 * l), lo = e & (sl - 1);
			tile[hi * pitch + lo] = (W)s[((u64)hi << (2 * (k - h))) + (md << (2 * l)) + lo];
		}
		if (md == 0 && threadIdx.x < 4) { // the k = 1 table: A <-> T, C <-> G
			mers_out[row * 4 + threadIdx.x] = mers_in[row * 4 + 3 - threadIdx.x];
		}
		__syncthreads();
		// out: o = ohi 4^(k-l) + rc_mid(md) 4^h + olo with ohi = rc_l(lo), olo = rc_h(hi)
		const u64 omd = rc_digits(md, mid);
		for (u32 e = threadIdx.x; e < elems; e += blockDim.x) {
			const u32 ohi = e >> (2 * h), olo = e & (sh - 1);
			const u32 hi = (u32)rc_digits(olo, h), lo = (u32)rc_digits(ohi, l);
			d[((u64)ohi << (2 * (k - l))) + (omd << (2 * h)) + olo] = (T)tile[hi * pitch + lo];
		}
		__syncthreads();
	}
}

int launch_revcomp(mc2_ctx *ctx, const mc2_hset *src, mc2_hset *dst)
{
	const int k = src->k, l = (k + 1) / 2 < 3 ? (k + 1) / 2 : 3, h = k / 2 < 3 ? k / 2 : 3;
	const u64 items = src->n << (2 * (k - h - l));
	if (items == 0) {
		return MC2_OK;
	}
	const u64 cap = (u64)ctx->sm_count * 8;
	const int grid = (int)(items < cap ? items : cap);
	cudaStream_t st = ctx->stream;
	switch (src->eb) {
	case 1: revcomp_kernel<uint8_t, u32><<<grid, 256, 0, st>>>((const uint8_t *)src->bins, (uint8_t *)dst->bins, src->mers1, dst->mers1, src->n, k, h, l); break;
	case 2: revcomp_kernel<uint16_t, u32><<<grid, 256, 0, st>>>((const uint16_t *)src->bins, (uint16_t *)dst->bins, src->mers1, dst->mers1, src->n, k, h, l); break;
	case 4: revcomp_kernel<uint32_t, u32><<<grid, 256, 0, st>>>((const uint32_t *)src->bins, (uint32_t *)dst->bins, src->mers1, dst->mers1, src->n, k, h, l); break;
	case 8: revcomp_kernel<u64, u64><<<grid, 256, 0, st>>>((const u64 *)src->bins, (u64 *)dst->bins, src->mers1, dst->mers1, src->n, k, h, l); break;
	default: set_error("elem_bytes must be 1, 2, 4 or 8"); return MC2_ERR_ARG;
	}
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

// Forward survivors: score holds id+ (the forward sweep's output), rev id- of the same pairs.  The larger is kept; equal values
// (a tie) stay on the forward strand.
__global__ void __launch_bounds__(256) strand_pick_kernel(double *score, const double *rev, int8_t *strand, u64 n)
{
	for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
		const double f = score[i], r = rev[i];
		const bool take = r > f;
		if (take) {
			score[i] = r;
		}
		strand[i] = take ? 1 : 0;
	}
}

// Reverse survivors (id- >= t) with fwd = id+ of the same pairs: the pairs the forward sweep rejected (!(id+ >= t), its own
// decision) are appended after the forward survivors; *counter counts all of them, at most max_out are written.
__global__ void __launch_bounds__(256) strand_append_kernel(const u64 *bq, const u64 *bd, const double *bs, const double *fwd, u64 n,
							    double t, unsigned long long *counter, u64 max_out, u64 *oq, u64 *od, double *os,
							    int8_t *ostr)
{
	const int lane = threadIdx.x & 31;
	for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {
		const u64 i = base + threadIdx.x;
		const bool keep = i < n && !(fwd[i] >= t);
		const unsigned m = __ballot_sync(0xffffffffu, keep);
		if (m == 0) {
			continue;
		}
		const int leader = __ffs(m) - 1;
		unsigned long long first = 0;
		if (lane == leader) {
			first = atomicAdd(counter, (unsigned long long)__popc(m));
		}
		first = __shfl_sync(0xffffffffu, first, leader);
		const u64 pos = first + __popc(m & ((1u << lane) - 1));
		if (keep && pos < max_out) {
			oq[pos] = bq[i];
			od[pos] = bd[i];
			os[pos] = bs[i];
			ostr[pos] = 1;
		}
	}
}

int launch_strand_pick(mc2_ctx *ctx, double *score, const double *rev, int8_t *strand, u64 n)
{
	if (n == 0) {
		return MC2_OK;
	}
	const u64 want = (n + 255) / 256, cap = (u64)ctx->sm_count * 8;
	strand_pick_kernel<<<(int)(want < cap ? want : cap), 256, 0, ctx->stream>>>(score, rev, strand, n);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

int launch_strand_append(mc2_ctx *ctx, const u64 *bq, const u64 *bd, const double *bs, const double *fwd, u64 n, double t,
			 u64 *counter, u64 max_out, u64 *oq, u64 *od, double *os, int8_t *ostr)
{
	if (n == 0) {
		return MC2_OK;
	}
	const u64 want = (n + 255) / 256, cap = (u64)ctx->sm_count * 8;
	strand_append_kernel<<<(int)(want < cap ? want : cap), 256, 0, ctx->stream>>>(bq, bd, bs, fwd, n, t, (unsigned long long *)counter,
										       max_out, oq, od, os, ostr);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

} // namespace mc2
