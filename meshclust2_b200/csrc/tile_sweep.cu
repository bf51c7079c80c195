// tile_sweep.cu — K2, all-pairs tile form: query x database sweep over uint8 / uint16 histograms of k = 5 .. 8 (rows of
// 1 .. 64 slabs of 1 KiB) on sm_100a.
//
// fastcar's work() for a whole block (src/fastcar/FC_Runner.cpp:427-470) / the all-pairs sweep of BASELINE configs[2]:
// every (query, database) pair inside the length window gets the model's reductions, the GLM score and the cutoff
// (Feature.cpp:136-171, Trainer.cpp:112-120, Predictor.cpp:323-333), survivors are appended to a list.
//
// One persistent CTA per SM (28 warps, warp specialised, registers re-dealt per warpgroup with setmaxnreg) walks
// 64 (query) x 256 (database) pair tiles in the order of a precomputed schedule (database-tile major inside super-rows
// of query tiles, so concurrently running CTAs share tiles in L2).  Per tile the bins stream through a 4-stage (coarse
// form without SAD sums: 2-stage) shared-memory ring of 40 KB stages filled by TMA (cp.async.bulk.tensor.2d,
// SWIZZLE_128B, one elected producer thread):
// per 1024 bins 16 stages of 64 bins of the u16 cumulative rows and 8 stages of 128 bins of the u8 rows, interleaved 2 : 1.
// Rows of several slabs (k >= 6) and uint16 bins: the cumulative rows are those of (bin - pseudo-count), which keeps them
// in 16 bits without changing any difference cumP - cumQ, and uint16 bins below 256 travel as a byte plane (cum_wide_kernel).
//   S_pq  = sum p*q              tcgen05.mma kind::i8 (u8 x u8 -> s32, exact) issued by one thread straight from the
//                                ring: two 128 x 64 accumulators (database rows = TMEM lanes) per tile, double buffered in
//                                TMEM so the next tile's MMAs overlap the epilogue.
//   S_emd = sum |cumP - cumQ|    16 compute warps on precomputed u16 cumulative rows (mc2_hset::cum16, cum16_kernel)
//                                through sum|a-b| = sum a + sum b - 2 sum min(a,b): VIMNMX.U16x2 (2 bins / instruction,
//                                ALU pipe) feeding IDP.2A with weights 0x0101 (FMA pipe) into a 32-bit accumulator: two
//                                instructions per two bins.  A thread owns database rows L and 128 + L (L = its TMEM lane)
//                                against 16 query rows: its rows are conflict-free 128-bit loads from the swizzled
//                                tile, the query rows warp-uniform shared-memory broadcasts, 32 accumulators in registers.
//                                The sums go to TMEM (tcgen05.st) for the epilogue warps, double buffered.
//   S_sad = sum |p - q|          VABSDIFF4.U8.ACC on the u8 stages (4 bins / instruction) -> S_min = (sumP+sumQ-S_sad)/2
// Epilogue (8 warps, thread = TMEM lane, two warps per lane quarter splitting the query columns; one warp per scheduler
// is latency bound and stalls the compute warps at the tile hand-over; 16 epilogue and 8 compute warps in the coarse
// form without SAD sums, see Layout): tcgen05.ld of 4 (or 2) query columns at a time; length window
// (FC_Runner.cpp:435-444) in 32 bits with an exact 64-bit path for lengths >= 2^32; an fp32 evaluation of the GLM sum
// with a rigorous host-derived error bound that can only REJECT (sum + bound < logit(0.5 - bias) - 1e-6 => not close
// whatever the rounding); the rest is ballot-compacted into a per-warp list and goes, one pair per lane, through the exact fp64
// epilogue shared with the other pair kernels (eval_pair_fast), so scores and decisions are the same bits as theirs.
// The screen is for 1024-bin rows; wider rows send every in-window pair through the exact epilogue.
// Coarse form (COARSE, one-slab rows with a screen, the bench shape): the screen needs an upper bound on the GLM sum, not
// the exact EMD.  Cumulative rows are non-decreasing (every bin >= base), so m_i = min(cumP_i, cumQ_i) is too, and its
// values at the 64 block ends s_j = 16 j + 15 (mc2_hset::cum16s, one ring stage) bound the whole sum:
// 16 (M - T) <= sum_i m_i <= 16 M with M = sum_j m(s_j), T = m(s_63) = min(totP, totQ).  A tile streams the 8 u8 stages
// and that single stage; the screen takes the EMD as the interval [cs - 32 M, cs - 32 (M - T)] and the candidates it
// keeps get the exact sum min(cumP, cumQ) over the full rows from global memory (one warp per candidate; the rows are
// prefetched into L2 when the screen keeps the pair) before the same exact epilogue, so scores and decisions are the bits
// of the full form.
// Identity search (Params::identity, mc2_identity_pairs): a regression model, clamp(sum) >= t <=> sum >= t for 0 < t <= 1,
// so the same screen rejects on sum + bound < t - margin (DevModel::scr_thr, set per call) and the exact epilogue keeps
// the pairs whose clamped sum is >= t.  The mode is a uniform runtime field read by the epilogue warps only.
#include "mc2_internal.cuh"
#include "pair_eval.cuh"
#include <cuda.h>
#include <cstring>
#include <cstdlib>

namespace mc2 {

namespace ts {

constexpr int TQ = 64;          // query rows per tile (UMMA N, TMEM columns per region)
constexpr int TD = 256;         // database rows per tile: two regions of 128 (UMMA M = 128 = the TMEM lanes)
constexpr int NBINS = 1024;      // bins per slab; rows are Params::n_slabs slabs long
constexpr int KC_CUM = 64;      // bins per ring stage while the u16 cumulative rows stream (128-byte rows)
constexpr int KC_U8 = 128;      // bins per ring stage while the u8 rows stream (128-byte rows)
constexpr int D_BYTES = TD * 128;        // 32 KB, SWIZZLE_128B
constexpr int Q_BYTES = TQ * 128;        //  8 KB
constexpr int STAGE_BYTES = D_BYTES + Q_BYTES; // 40 KB
constexpr int MAX_SUPER = 1024;          // entries of the tile schedule's prefix array

// Warp layout of an instantiation, in whole warpgroups (setmaxnreg is per warpgroup, and a warp reaches only the TMEM lane
// quarter warp % 4).  Warpgroup 0: TMA producer, MMA issuer, two idle warps; then NCW compute warps; then NEW epilogue
// warps, NEW / 4 per TMEM lane quarter, each taking QE query columns of both regions.
//  - full form, and the coarse form with SAD sums (its compute warps still stream the eight u8 stages): 16 compute +
//    8 epilogue warps, a 4-stage ring.  Measured on 100 k x 1 kb (bench model, full form), ms per 1.8e9 pairs: 4 epilogue
//    warps x 4 pairs per thread 95.6, 8 x 2: 91.5, 4 x 2: 105.7.
//  - coarse form without SAD sums: the compute warps work on one ring stage of nine (the 64 samples) and the epilogue's
//    per-pair work paces the tile, so the warps go the other way: 8 compute + 16 epilogue warps.  A compute thread then
//    covers 32 query rows, in two passes of 16 stored to TMEM one after the other (80 registers).  The screen's scratch
//    grows with the epilogue threads (NEED 6: 7 slots x 4 pairs x 512 threads x 4 B = 56 KiB), which leaves room for a
//    2-stage ring: a tile streams 9 stages, and the MMAs and sample sums of the next tile overlap this tile's epilogue
//    through the double-buffered TMEM.
// Registers (setmaxnreg per warpgroup; the pool is threads x launch registers, at most 64 K) are the same for both:
// launch 72, control 24, compute 80, epilogue 80 = 128 x 24 + 512 x 80 + 256 x 80 = 28 x 32 x 72.
template <int NEED, bool COARSE> struct Layout {
	static constexpr bool EPI_HEAVY = COARSE && (NEED & NEED_MIN) == 0;
	static constexpr int NCW = EPI_HEAVY ? 8 : 16;
	static constexpr int NEW = EPI_HEAVY ? 16 : 8;
	static constexpr int THREADS = (4 + NCW + NEW) * 32;
	static constexpr int QN = 16;                      // query rows per compute pass (x 2 database rows): 32 accumulators
	static constexpr int QPASS = TQ / (NCW / 4) / QN;  // passes per stage over a compute warpgroup's TQ / (NCW / 4) rows
	static constexpr int QE = TQ / (NEW / 4);          // query columns per epilogue warp
	// pairs a thread of the epilogue screens at a time (query columns per tcgen05.ld): 4 where the screen's scratch
	// (slots x pairs x NEW * 32 threads x 4 bytes) leaves room for a candidate list that is flushed once per tile, else 2
	static constexpr int NP = scr_slots(NEED & 7) <= 7 ? 4 : 2;
	static constexpr int LIST_CAP = NP == 4 ? 192 : 128; // candidate records per epilogue warp
	static constexpr int STAGES = EPI_HEAVY ? 2 : 4;
	static constexpr int REGS_LAUNCH = 72, REGS_CTRL = 24, REGS_COMPUTE = 80, REGS_EPI = 80;
	static_assert(NCW % 4 == 0 && NEW % 4 == 0, "roles are whole warpgroups");
	static_assert(QPASS >= 1 && QPASS * QN * (NCW / 4) == TQ && QE * (NEW / 4) == TQ && QE % NP == 0, "query rows and columns");
	static_assert(QPASS == 1 || (COARSE && (NEED & NEED_MIN) == 0), "several passes only over the one sample stage");
	static_assert(128 * REGS_CTRL + NCW * 32 * REGS_COMPUTE + NEW * 32 * REGS_EPI <= THREADS * REGS_LAUNCH, "register pool");
	static_assert(THREADS * REGS_LAUNCH <= 65536 && 65536 / THREADS >= REGS_LAUNCH, "register file");
	static_assert(LIST_CAP >= 32 * NP, "a batch of candidates fits the list");
};
// TMEM columns (512 allocated): Gram accumulators double buffered, EMD / SAD sums single buffered
constexpr u32 TM_DOT = 0;                // + buf * 128 + region * 64
constexpr u32 TM_EMD = 256;              // + ebuf * 128 + region * 64 (double buffered when no SAD sums are needed)
constexpr u32 TM_SAD = 384;              // + region * 64

struct Params {
	u64 q0, q1, d0, d1;     // row ranges (query set / database set)
	int upper_only;
	double cutoff;
	u64 max_out;
	u64 *out_q, *out_d;
	double *out_score;
	u64 *counters;          // [0] survivors, [1] scored pairs, [2] pairs through the exact epilogue, [3] 1: coarse form
	int *err;
	int identity;           // 0: survivors are the classifier's close pairs; 1: pairs whose score >= min_identity
	double min_identity;
	Sideband sbQ, sbD;
	const u32 *csQ, *csD;   // per-row sum of the cumulative row (EMD identity)
	// coarse form: the full cumulative rows (exact refinement of the candidates) and the 64 samples per row (the last one
	// is the row's total)
	const unsigned short *cumQ, *cumD, *smpQ, *smpD;
	u32 nqt, ndt;           // tiles along each side
	u32 group;              // query tiles per super-row of the schedule
	u32 n_super;
	u32 n_slabs;            // bins per row / 1024 (1 for k = 5, 64 for k = 8)
	const u32 *sched;       // [n_super + 1] exclusive prefix of items per super-row (device)
	// raw mode (tests): dense (q1-q0) x (d1-d0) matrices of the reductions instead of scoring
	u32 *raw_dot, *raw_emd, *raw_sad;
};

// ---------------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u32 bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(u32 bar, u32 bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(u32 bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ bool mbar_try(u32 bar, u32 parity)
{
	// the suspend-time hint (ns) lets the hardware park the warp instead of returning at once: a polling warp would
	// take issue slots from the compute warps that share its scheduler
	u32 ok;
	asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
		     : "=r"(ok)
		     : "r"(bar), "r"(parity), "r"(10000u)
		     : "memory");
	return ok != 0;
}
// bounded wait: a pipeline bug must end in an error, never in a hung GPU
__device__ __forceinline__ void mbar_wait(u32 bar, u32 parity, int *err)
{
	u32 spins = 0;
	while (!mbar_try(bar, parity)) {
		if (++spins > (1u << 20)) {
			atomicOr(err, 16);
			__trap();
		}
	}
}
__device__ __forceinline__ void tma_load_2d(u32 dst, const CUtensorMap *map, int x, int y, u32 bar)
{
	asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
		     "l"(map), "r"(x), "r"(y), "r"(bar)
		     : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(u32 bar)
{
	asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_i8(u32 tmem_d, u64 desc_a, u64 desc_b, u32 idesc, u32 accumulate)
{
	asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
		     "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
		     : "memory");
}
__device__ __forceinline__ void tc_ld4(u32 taddr, u32 (&v)[4])
{
	asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld2(u32 taddr, u32 (&v)[2])
{
	asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(v[0]), "=r"(v[1]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ldn(u32 taddr, u32 (&v)[4]) { tc_ld4(taddr, v); }
__device__ __forceinline__ void tc_ldn(u32 taddr, u32 (&v)[2]) { tc_ld2(taddr, v); }
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_st32(u32 taddr, const u32 (&v)[32])
{
	asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
		     "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
		     "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]),
		     "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]),
		     "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
		     : "memory");
}
__device__ __forceinline__ void tc_st16(u32 taddr, const u32 (&v)[16])
{
	asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr), "r"(v[0]),
		     "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]),
		     "r"(v[13]), "r"(v[14]), "r"(v[15])
		     : "memory");
}
__device__ __forceinline__ void tc_st(u32 taddr, const u32 (&v)[32]) { tc_st32(taddr, v); }
__device__ __forceinline__ void tc_st(u32 taddr, const u32 (&v)[16]) { tc_st16(taddr, v); }
__device__ __forceinline__ void tc_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// bulk prefetch of global memory into L2 (no registers, no completion to wait for)
__device__ __forceinline__ void l2_prefetch(const void *ptr, u32 bytes)
{
	asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ptr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void named_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ uint4 lds128(u32 addr)
{
	uint4 v;
	asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
	return v;
}
__device__ __forceinline__ u32 vmin2(u32 a, u32 b)
{
	u32 d;
	asm("min.u16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
	return d;
}
__device__ __forceinline__ u32 dp2a_sum(u32 packed, u32 acc)
{
	u32 d;
	asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(packed), "r"(0x0101u), "r"(acc));
	return d;
}
__device__ __forceinline__ u32 sad4(u32 a, u32 b, u32 c)
{
	u32 d;
	asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
	return d;
}

// K-major shared-memory operand descriptor for 128-byte rows under SWIZZLE_128B (cute::UMMA::SmemDescriptor: start >> 4 at
// [0,14), leading byte offset >> 4 at [16,30) (1 for swizzled K-major), stride byte offset >> 4 at [32,46) = 8 rows x 128 B,
// version 1 at [46,48), layout type at [61,64): 2 = SWIZZLE_128B)
__device__ __forceinline__ u64 umma_desc_sw128(u32 saddr)
{
	return (u64)((saddr & 0x3FFFFu) >> 4) | ((u64)1 << 16) | ((u64)(1024 >> 4) << 32) | ((u64)1 << 46) | ((u64)2 << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format S32 = 2 at [4,6), a/b format U8 = 0, K-major both,
// N >> 3 at [17,23), M >> 4 at [24,29)
constexpr u32 IDESC_U8 = (2u << 4) | ((u32)(TQ >> 3) << 17) | ((u32)(128 >> 4) << 24);

// ---------------------------------------------------------------------------------------------------------------
// tile schedule: super-rows of `group` query tiles; inside a super-row the items run database-tile major, query-tile
// minor, so the CTAs working at the same time share one database tile and a handful of query tiles (L2 reuse).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 first_dt(const Params &p, u32 qt)
{
	if (!p.upper_only) {
		return 0;
	}
	// smallest database offset that can pair with the tile's first query row: d > q
	const s64 x = (s64)(p.q0 + (u64)qt * TQ) + 1 - (s64)p.d0;
	return x <= 0 ? 0u : (u32)(x / TD);
}

__global__ void __launch_bounds__(1024) sched_kernel(Params p, u32 *sched)
{
	__shared__ u32 cnt[MAX_SUPER];
	const u32 s = threadIdx.x;
	u32 c = 0;
	if (s < p.n_super) {
		const u32 f = first_dt(p, s * p.group);
		c = f < p.ndt ? (p.ndt - f) * p.group : 0;
	}
	if (s < (u32)MAX_SUPER) {
		cnt[s] = c;
	}
	__syncthreads();
	if (s == 0) {
		u32 run = 0;
		for (u32 i = 0; i < p.n_super; i++) {
			sched[i] = run;
			run += cnt[i];
		}
		sched[p.n_super] = run;
	}
}

struct Tile {
	u32 qt, dt;
	bool valid;
};
__device__ __forceinline__ Tile decode_item(const Params &p, const u32 *s_sched, u32 item)
{
	// largest s with sched[s] <= item
	u32 lo = 0, hi = p.n_super;
	while (hi - lo > 1) {
		const u32 mid = (lo + hi) >> 1;
		if (s_sched[mid] <= item) {
			lo = mid;
		} else {
			hi = mid;
		}
	}
	const u32 r = item - s_sched[lo];
	Tile t;
	t.qt = lo * p.group + r % p.group;
	t.dt = first_dt(p, lo * p.group) + r / p.group;
	t.valid = t.qt < p.nqt && t.dt < p.ndt && t.dt >= first_dt(p, t.qt);
	return t;
}

// ---------------------------------------------------------------------------------------------------------------
// CUDA-core work of one compute warp on one ring stage.  The thread owns database rows L and 128 + L of the tile
// (L = 32 * (warp % 4) + lane, its TMEM lane) against QN query rows of its share: 2 * QN accumulators (QN = 16).  Per
// 16-byte step: 2 conflict-free row loads, QN warp-uniform (broadcast) query loads, 16 * QN (EMD: VIMNMX.U16x2 + IDP.2A
// per word) or 8 * QN (SAD: VABSDIFF4 per word) arithmetic instructions.
// 128-byte rows under SWIZZLE_128B: 16-byte chunk c of row r sits at r * 128 + ((c ^ (r & 7)) << 4).
// ---------------------------------------------------------------------------------------------------------------
template <bool IS_EMD, int QN>
__device__ __forceinline__ void stage_compute(const unsigned char *stage, u32 lane_row, int qsel, u32 (&acc)[2][QN])
{
	// plain loads (not asm): the compiler may order and pipeline them freely inside the stage.  Query rows QN * qsel ..
	// QN * qsel + QN - 1
	const uint4 *dptr = reinterpret_cast<const uint4 *>(stage) + lane_row * 8;
	const uint4 *qptr = reinterpret_cast<const uint4 *>(stage + D_BYTES) + qsel * (QN * 8);
	const u32 dsw = lane_row & 7;
	// fully unrolled over the eight 16-byte steps: every query-row address is an immediate offset (the swizzle XOR folds at
	// compile time), ~2.3 k instructions per stage
	uint4 D0 = dptr[dsw], D1 = dptr[1024 + dsw];
#pragma unroll
	for (int c = 0; c < 8; c++) {
		const uint4 E0 = D0, E1 = D1;
		if (c < 7) { // next step's rows are requested before this step's arithmetic
			D0 = dptr[(u32)(c + 1) ^ dsw];
			D1 = dptr[1024 + ((u32)(c + 1) ^ dsw)];
		}
#pragma unroll
		for (int g = 0; g < QN / 4; g++) {
			uint4 Q[4];
#pragma unroll
			for (int j = 0; j < 4; j++) {
				const int q = g * 4 + j;
				Q[j] = qptr[q * 8 + (c ^ (q & 7))];
			}
			// word by word over the four query rows x two database rows: eight independent accumulator chains
#define MC2_STEP(W)                                                                       \
	_Pragma("unroll") for (int j = 0; j < 4; j++)                                     \
	{                                                                                 \
		const int q = g * 4 + j;                                                  \
		if constexpr (IS_EMD) {                                                   \
			acc[0][q] = dp2a_sum(vmin2(Q[j].W, E0.W), acc[0][q]);             \
			acc[1][q] = dp2a_sum(vmin2(Q[j].W, E1.W), acc[1][q]);             \
		} else {                                                                  \
			acc[0][q] = sad4(Q[j].W, E0.W, acc[0][q]);                        \
			acc[1][q] = sad4(Q[j].W, E1.W, acc[1][q]);                        \
		}                                                                         \
	}
			MC2_STEP(x)
			MC2_STEP(y)
			MC2_STEP(z)
			MC2_STEP(w)
#undef MC2_STEP
		}
	}
}

// ---------------------------------------------------------------------------------------------------------------
// fp32 screen: the GLM sum of NP pairs in single precision with a rigorous bound on |fp32 sum - exact sum| (constants and
// derivation: build_screen in mc2_api.cu).  A pair whose bit is clear in the result is certainly not close; everything
// else goes to the exact fp64 epilogue.  Every raw single is a cancellation-free expression of exact integers (at most 8
// operations of <= 2 ulp); the NP pairs share the control flow, so the model's uniform branches are paid once per NP
// pairs and the dependency chains interleave.  No local memory: combo products are built single by single.
// ---------------------------------------------------------------------------------------------------------------
struct RowF {          // per-row values of the screen
	u32 mag, sum, sumsq; // low words (valid when !big)
	u32 cs;        // sum of the row's cumulative sums (EMD identity)
	float magf, lenf;
	float rss;     // 1 / sqrt(sumsq)
	float rnn;     // 1 / sqrt(N*sumsq - 2*mag*sum + mag^2)  (pearson's centred norm, exact integer -> float)
	u32 big;       // mag or len outside the screen's comfortable range -> exact path
	u32 tot;       // coarse form: the row's last cumulative value
};

// smp: the coarse form's samples (64 per row) or nullptr
__device__ __forceinline__ RowF make_rowf(const Sideband &sb, const u32 *cs, const unsigned short *smp, u64 row, bool ok, u64 &len)
{
	RowF r;
	memset(&r, 0, sizeof r);
	r.big = 1;
	len = 0;
	if (ok) {
		const u64 mag = sb.mag[row], sum = sb.sum[row], sumsq = sb.sumsq[row];
		len = sb.len[row];
		r.mag = (u32)mag;
		r.sum = (u32)sum;
		r.sumsq = (u32)sumsq;
		r.magf = (float)mag;
		r.lenf = (float)len;
		r.rss = rsqrtf((float)sumsq);
		// the screen wants exact float lengths (their difference cancels) and 64-bit pearson terms
		r.big = (mag >= (1ull << 26) || len >= (1ull << 24) || len == 0 || mag == 0) ? 1u : 0u;
		const long long m = (long long)(mag & 0x3FFFFFFull);
		r.rnn = rsqrtf((float)(1024ll * (long long)sumsq - 2ll * m * (long long)sum + m * m));
		r.cs = cs ? cs[row] : 0u;
		r.tot = smp ? smp[row * 64 + 63] : 0u;
	}
	return r;
}

__device__ __forceinline__ float sqrt_approx(float x)
{
	float r;
	asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
	return r;
}

// sx: this thread's column of the epilogue's scratch, element (slot, t) at sx[(slot * NP + t) * ET] (ET: epilogue
// threads); slot = single slot (scr_slot), the last slot holds the constant 1 (written once per kernel)
// COARSE: the EMD is only known to lie in [emd[t], emd_hi[t]] (exact integers).  x is evaluated at both ends, u covers
// both, and a combo with the EMD factor adds the larger of its values at the two ends: the other factor is fixed, so the
// combo is linear in x or in x^2, and x^2 over an interval that spans 0 also takes the value 0 (the fused sums are
// monotone in the exact value, so max(fma(w, f1, s), fma(w, f2, s)) = fl(max(w f1, w f2) + s) keeps the error model).
template <int NEED, int NP, bool COARSE, int ET>
__device__ __forceinline__ u32 screen_pairs(const DevModel &dm, float *sx, const u32 (&dot)[NP], const u32 (&emd)[NP], const u32 (&emd_hi)[NP],
					    const u32 (&sad)[NP], const RowF &P, const RowF *Q)
{
	float m[NP];
#pragma unroll
	for (int t = 0; t < NP; t++) {
		m[t] = 0.0f;
	}
	// one single: x = a * raw + b -> scratch; max |x| over the singles the model uses.  The model is the same for the
	// whole grid, so skipping a single it does not use is a uniform branch.
#define MC2_SCR(CODE, RAW)                                                                       \
	if (dm.slot[CODE] >= 0) {                                                                \
		const float a_ = dm.scr_a[CODE], b_ = dm.scr_b[CODE];                            \
		_Pragma("unroll") for (int t = 0; t < NP; t++)                                   \
		{                                                                                \
			const float x_ = __fmaf_rn(a_, (RAW), b_);                               \
			sx[(scr_slot(NEED & 7, CODE) * NP + t) * ET] = x_;                       \
			m[t] = fmaxf(m[t], fabsf(x_));                                           \
		}                                                                                \
	}
	if constexpr ((NEED & NEED_DOT) != 0) {
		float n2f[NP], dotf[NP], rt[NP];
#pragma unroll
		for (int t = 0; t < NP; t++) {
			n2f[t] = (float)(P.sumsq + Q[t].sumsq - 2u * dot[t]); // exact integer: sum (p-q)^2 < 2^27 for 1024 uint8 bins
			dotf[t] = (float)dot[t];
			rt[t] = sqrt_approx(n2f[t]);
		}
		MC2_SCR(SC_EUCLIDEAN, rt[t])
		MC2_SCR(SC_SIMRATIO, __fdividef(dotf[t], dotf[t] + rt[t]))
		MC2_SCR(SC_NORMALIZED_VECTORS, dotf[t] * (P.rss * Q[t].rss))
		MC2_SCR(SC_PEARSON, (float)(1024ll * (long long)dot[t] - (long long)P.mag * (long long)Q[t].sum - (long long)Q[t].mag * (long long)P.sum +
					    (long long)P.mag * (long long)Q[t].mag) *
					    (P.rnn * Q[t].rnn))
	}
	if constexpr ((NEED & NEED_MIN) != 0) {
		float two_smin[NP];
#pragma unroll
		for (int t = 0; t < NP; t++) {
			two_smin[t] = (float)(P.sum + Q[t].sum - sad[t]);
		}
		MC2_SCR(SC_MANHATTAN, (float)sad[t])
		MC2_SCR(SC_INTERSECTION, __fdividef(two_smin[t], P.magf + Q[t].magf))
		MC2_SCR(SC_KULCZYNSKI2, __fdividef(P.magf + Q[t].magf, 2.0f * (P.magf * (1.0f / 1024.0f)) * (Q[t].magf * (1.0f / 1024.0f))) * (0.5f * two_smin[t]))
	}
	float xe_hi[NP]; // COARSE: the EMD single at the upper end of its interval (the lower end is in its slot)
	if constexpr ((NEED & NEED_EMD) != 0) {
		if constexpr (COARSE) {
			if (dm.slot[SC_EMD] >= 0) {
				const float a_ = dm.scr_a[SC_EMD], b_ = dm.scr_b[SC_EMD];
#pragma unroll
				for (int t = 0; t < NP; t++) {
					const float x1 = __fmaf_rn(a_, (float)emd[t], b_);
					sx[(scr_slot(NEED & 7, SC_EMD) * NP + t) * ET] = x1;
					xe_hi[t] = __fmaf_rn(a_, (float)emd_hi[t], b_);
					m[t] = fmaxf(m[t], fmaxf(fabsf(x1), fabsf(xe_hi[t])));
				}
			}
		} else {
			MC2_SCR(SC_EMD, (float)emd[t])
		}
	}
	MC2_SCR(SC_LENGTHD, fabsf(P.lenf - Q[t].lenf))
#undef MC2_SCR
	float s[NP];
#pragma unroll
	for (int t = 0; t < NP; t++) {
		s[t] = dm.scr_w[0];
	}
	constexpr int KE = scr_slot(NEED & 7, SC_EMD);
#pragma unroll 1
	for (int c = 0; c < dm.n_combos; c++) {
		const int sa = dm.scr_ka[c], sb = dm.scr_kb[c];
		const int ka = sa * NP * ET, kb = sb * NP * ET;
		const bool pa2 = dm.scr_pa2[c] != 0, pb2 = dm.scr_pb2[c] != 0;
		const float w = dm.scr_w[c + 1];
		if (COARSE && (NEED & NEED_EMD) != 0 && (sa == KE || sb == KE)) {
			// the EMD factor (a combo holds it once: EMD x EMD is one factor squared) against the other, fixed one
			const bool ea = sa == KE, e2 = ea ? pa2 : pb2, o2 = ea ? pb2 : pa2;
			const int ko = ea ? kb : ka;
#pragma unroll
			for (int t = 0; t < NP; t++) {
				const float xo = sx[ko + t * ET], fo = o2 ? xo * xo : xo;
				const float x1 = sx[KE * NP * ET + t * ET], x2 = xe_hi[t];
				const float f1 = e2 ? x1 * x1 : x1, f2 = e2 ? x2 * x2 : x2;
				float sn = fmaxf(__fmaf_rn(w, f1 * fo, s[t]), __fmaf_rn(w, f2 * fo, s[t]));
				// x^2 reaches 0 inside the interval: tested on the interval widened by the bound on |fl(x) - x|, so a
				// sign change the rounding hides is still taken
				const float tol = dm.scr_dx * ((1.0f + m[t]) * 1.001f);
				if (e2 && fminf(x1, x2) <= tol && fmaxf(x1, x2) >= -tol) {
					sn = fmaxf(sn, s[t]);
				}
				s[t] = sn;
			}
		} else {
#pragma unroll
			for (int t = 0; t < NP; t++) {
				const float xa = sx[ka + t * ET], xb = sx[kb + t * ET];
				const float fa = pa2 ? xa * xa : xa, fb = pb2 ? xb * xb : xb;
				s[t] = __fmaf_rn(w, fa * fb, s[t]);
			}
		}
	}
	u32 maybe = 0;
#pragma unroll
	for (int t = 0; t < NP; t++) {
		const float u = (1.0f + m[t]) * 1.001f, u2 = u * u;
		const float e = __fmaf_rn(dm.scr_k1, u2 * u2, dm.scr_k0);
		const bool reject = (e < 1.0f) && (s[t] + e < dm.scr_thr);
		maybe |= reject ? 0u : (1u << t);
	}
	return maybe;
}

// ---------------------------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------------------------
struct Cand {
	u32 pair; // region << 6 | query row in the tile
	u32 dot, emd, sad;
};

template <int NEED, bool COARSE> struct Smem {
	using LY = Layout<NEED, COARSE>;
	static constexpr int RING = 0;
	static constexpr int LIST = LY::STAGES * STAGE_BYTES;                             // Cand[NEW][LIST_CAP]
	static constexpr int SCRX = LIST + LY::NEW * LY::LIST_CAP * (int)sizeof(Cand);     // float [slots][NP][NEW * 32]: the screen's scratch
	static constexpr int ROWQ = SCRX + scr_slots(NEED & 7) * LY::NP * LY::NEW * 32 * 4; // RowF[2][TQ]
	static constexpr int WINQ = ROWQ + 2 * TQ * (int)sizeof(RowF);                    // u64 window [2][TQ][2]
	static constexpr int WIN32 = WINQ + 2 * TQ * 16;                                  // uint2 window [2][TQ], saturated to 32 bits
	static constexpr int SCHED = WIN32 + 2 * TQ * 8;                                  // u32 [MAX_SUPER + 1]
	static constexpr int BARS = SCHED + (MAX_SUPER + 1) * 4 + 4;                      // mbarriers
	static constexpr int MISC = BARS + 32 * 8;                                        // tmem base
	static constexpr int TOTAL = MISC + 64 + 1024;                                    // + alignment slack
	static_assert(2 * LY::STAGES + 8 <= 32, "mbarriers");
	static_assert(TOTAL <= 232448, "shared memory per CTA");
};

// ONE: rows of one 1 KiB slab (k = 5), stage counts known at compile time; otherwise Params::n_slabs slabs per row.
// COARSE: the coarse form (header comment); the cumulative tensor maps are those of the samples (64 per row)
template <int NEED, bool RAW, bool ONE, bool COARSE>
__global__ void __launch_bounds__(Layout<NEED, COARSE>::THREADS, 1)
tile_sweep_kernel(const __grid_constant__ DevModel dm, const __grid_constant__ Params p, const __grid_constant__ CUtensorMap mapCumD,
		  const __grid_constant__ CUtensorMap mapCumQ, const __grid_constant__ CUtensorMap mapU8D,
		  const __grid_constant__ CUtensorMap mapU8Q)
{
	using L = Smem<NEED, COARSE>;
	using LY = Layout<NEED, COARSE>;
	constexpr int NCW = LY::NCW, NEW = LY::NEW, STAGES = LY::STAGES, QN = LY::QN, QE = LY::QE, NP = LY::NP, LIST_CAP = LY::LIST_CAP;
	constexpr int REGS_LAUNCH = LY::REGS_LAUNCH, REGS_CTRL = LY::REGS_CTRL, REGS_COMPUTE = LY::REGS_COMPUTE, REGS_EPI = LY::REGS_EPI;
	constexpr bool DOT = (NEED & NEED_DOT) != 0, EMD = (NEED & NEED_EMD) != 0, MIN = (NEED & NEED_MIN) != 0;
	static_assert(!COARSE || (ONE && EMD && !RAW), "the coarse form is for one-slab rows, a model with EMD, scoring");
	constexpr bool U8_PHASE = DOT || MIN;
	constexpr bool CUDA_RED = EMD || MIN;             // compute warps produce sums for the epilogue
	const int n_slabs = ONE ? 1 : (int)p.n_slabs;
	const int N_U8 = U8_PHASE ? n_slabs * (NBINS / KC_U8) : 0;   // ring stages per tile while the u8 rows stream
	const int N_CUM = EMD ? (COARSE ? 1 : n_slabs * (NBINS / KC_CUM)) : 0; // ... while the cumulative rows (samples) stream
	// Gram + EMD models: every third stage carries u8 rows (for the MMA issuer only), so the compute warps never sit
	// through a whole u8 phase; otherwise (and in the coarse form, 8 + 1 stages) the u8 stages come first, then the
	// cumulative ones
	constexpr bool INTERLEAVE = DOT && EMD && !MIN && !COARSE;
	auto stage_is_u8 = [N_U8](int c) { return INTERLEAVE ? (c % 3 == 2) : (c < N_U8); };
	auto stage_index = [N_U8](int c) { return INTERLEAVE ? (c % 3 == 2 ? c / 3 : c - c / 3) : (c < N_U8 ? c : c - N_U8); };
	extern __shared__ unsigned char smem_raw[];
	// SWIZZLE_128B tiles and the UMMA descriptors want 1024-byte alignment: align by hand (the launch adds the slack)
	unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
	const u32 sbase = smem_u32(smem);
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	u32 *s_sched = reinterpret_cast<u32 *>(smem + L::SCHED);
	const u32 bar_full = sbase + L::BARS, bar_empty = bar_full + STAGES * 8, bar_tfull = bar_empty + STAGES * 8, bar_tempty = bar_tfull + 2 * 8;
	const u32 bar_efull = bar_tempty + 2 * 8, bar_eempty = bar_efull + 2 * 8; // [2] each
	constexpr int EBUFS = MIN ? 1 : 2; // EMD sums in TMEM: two buffers unless the SAD sums need the columns
	u32 *s_tmem = reinterpret_cast<u32 *>(smem + L::MISC);

	for (u32 i = threadIdx.x; i <= p.n_super; i += blockDim.x) {
		s_sched[i] = p.sched[i];
	}
	if (threadIdx.x == 0) {
		for (int s = 0; s < STAGES; s++) {
			mbar_init(bar_full + s * 8, 1);
			mbar_init(bar_empty + s * 8, NCW + 1); // every compute warp and the MMA thread release every stage
		}
		for (int b = 0; b < 2; b++) {
			mbar_init(bar_tfull + b * 8, 1);
			mbar_init(bar_tempty + b * 8, NEW);
		}
		for (int b = 0; b < 2; b++) {
			mbar_init(bar_efull + b * 8, NCW);
			mbar_init(bar_eempty + b * 8, NEW);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	if (warp == 1) { // the whole tensor memory: one CTA per SM
		asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(s_tmem)) : "memory");
		asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
	}
	tc_fence_before();
	__syncthreads();
	tc_fence_after();
	const u32 tmem_base = *s_tmem;
	const u32 n_items = s_sched[p.n_super];

	if (warp == 0) {
		// ===== TMA producer =====
		asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
		if (lane == 0) {
			u32 s = 0, ph = 0;
			for (u32 item = blockIdx.x; item < n_items; item += gridDim.x) {
				const Tile t = decode_item(p, s_sched, item);
				if (!t.valid) {
					continue;
				}
				const int qrow = (int)(p.q0 + (u64)t.qt * TQ), drow = (int)(p.d0 + (u64)t.dt * TD);
				for (int c = 0; c < N_U8 + N_CUM; c++) {
					mbar_wait(bar_empty + s * 8, ph ^ 1, p.err);
					const u32 st = sbase + s * STAGE_BYTES, fb = bar_full + s * 8;
					mbar_expect_tx(fb, STAGE_BYTES);
					if (stage_is_u8(c)) {
						tma_load_2d(st, &mapU8D, stage_index(c) * KC_U8, drow, fb);
						tma_load_2d(st + D_BYTES, &mapU8Q, stage_index(c) * KC_U8, qrow, fb);
					} else {
						tma_load_2d(st, &mapCumD, stage_index(c) * KC_CUM, drow, fb);
						tma_load_2d(st + D_BYTES, &mapCumQ, stage_index(c) * KC_CUM, qrow, fb);
					}
					if (++s == (u32)STAGES) {
						s = 0;
						ph ^= 1;
					}
				}
			}
		}
	} else if (warp == 1) {
		// ===== MMA issuer =====
		asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
		if (lane == 0) {
			u32 s = 0, ph = 0, it = 0;
			for (u32 item = blockIdx.x; item < n_items; item += gridDim.x) {
				const Tile t = decode_item(p, s_sched, item);
				if (!t.valid) {
					continue;
				}
				const u32 buf = it & 1;
				if (DOT) {
					mbar_wait(bar_tempty + buf * 8, ((it >> 1) & 1) ^ 1, p.err);
					tc_fence_after();
				}
				for (int c = 0; c < N_U8 + N_CUM; c++) {
					mbar_wait(bar_full + s * 8, ph, p.err);
					if (DOT && stage_is_u8(c)) {
						const int ku = stage_index(c);
						tc_fence_after();
						const u32 a = sbase + s * STAGE_BYTES, b = a + D_BYTES;
#pragma unroll
						for (int r = 0; r < 2; r++) {
#pragma unroll
							for (int k = 0; k < KC_U8 / 32; k++) {
								tc_mma_i8(tmem_base + TM_DOT + buf * 128 + r * 64, umma_desc_sw128(a + r * 16384 + k * 32),
									  umma_desc_sw128(b + k * 32), IDESC_U8, (ku | k) != 0);
							}
						}
						tc_commit(bar_empty + s * 8);
						if (ku == N_U8 - 1) {
							tc_commit(bar_tfull + buf * 8);
						}
					} else {
						mbar_arrive(bar_empty + s * 8);
					}
					if (++s == (u32)STAGES) {
						s = 0;
						ph ^= 1;
					}
				}
				it++;
			}
		}
	} else if (warp < 4) {
		// idle: their registers go to the other warpgroups
		asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
	} else if (warp < 4 + NCW) {
		// ===== compute warps =====
		if (REGS_COMPUTE > REGS_LAUNCH) {
			asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_COMPUTE));
		}
		const int cw = warp - 4;
		const u32 quarter = (u32)warp & 3;          // the TMEM lanes this warp may touch: 32 * quarter ..
		const int qsel = cw >> 2;                   // query rows QN * QPASS * qsel .. of the tile
		const u32 lane_row = quarter * 32 + (u32)lane;
		const u32 tlane = (quarter * 32) << 16;
		u32 s = 0, ph = 0, it = 0;
		for (u32 item = blockIdx.x; item < n_items; item += gridDim.x) {
			const Tile t = decode_item(p, s_sched, item);
			if (!t.valid) {
				continue;
			}
			bool tmem_free = false;
			const u32 eb = EBUFS == 2 ? (it & 1) : 0, eit = EBUFS == 2 ? (it >> 1) : it; // buffer and its use count
			if (INTERLEAVE) {
				u32 acc[2][QN];
#pragma unroll
				for (int q = 0; q < QN; q++) {
					acc[0][q] = acc[1][q] = 0;
				}
#pragma unroll 1
				for (int c = 0; c < N_U8 + N_CUM; c++) {
					mbar_wait(bar_full + s * 8, ph, p.err);
					if (c % 3 != 2) {
						stage_compute<true>(smem + s * STAGE_BYTES, lane_row, qsel, acc);
					}
					__syncwarp();
					if (lane == 0) {
						mbar_arrive(bar_empty + s * 8);
					}
					if (++s == (u32)STAGES) {
						s = 0;
						ph ^= 1;
					}
				}
				mbar_wait(bar_eempty + eb * 8, (eit & 1) ^ 1, p.err); // the epilogue is done with this buffer's previous sums
				tc_fence_after();
				tc_st(tmem_base + tlane + TM_EMD + eb * 128 + qsel * QN, acc[0]);
				tc_st(tmem_base + tlane + TM_EMD + eb * 128 + 64 + qsel * QN, acc[1]);
			}
			if (!INTERLEAVE && U8_PHASE) {
				u32 acc[2][QN];
				if (MIN) {
#pragma unroll
					for (int q = 0; q < QN; q++) {
						acc[0][q] = acc[1][q] = 0;
					}
				}
#pragma unroll 1
				for (int c = 0; c < N_U8; c++) {
					mbar_wait(bar_full + s * 8, ph, p.err);
					if (MIN) {
						stage_compute<false>(smem + s * STAGE_BYTES, lane_row, qsel, acc);
					}
					__syncwarp();
					if (lane == 0) {
						mbar_arrive(bar_empty + s * 8);
					}
					if (++s == (u32)STAGES) {
						s = 0;
						ph ^= 1;
					}
				}
				if (MIN) {
					mbar_wait(bar_eempty + eb * 8, (eit & 1) ^ 1, p.err); // the epilogue is done with this buffer's previous sums
					tc_fence_after();
					tmem_free = true;
					tc_st(tmem_base + tlane + TM_SAD + qsel * QN, acc[0]);
					tc_st(tmem_base + tlane + TM_SAD + 64 + qsel * QN, acc[1]);
				}
			}
			if (!INTERLEAVE && EMD && LY::QPASS > 1) {
				// the one sample stage, the warpgroup's query rows in passes of QN: each pass goes to TMEM before the next
				// one reuses the accumulators
				mbar_wait(bar_full + s * 8, ph, p.err);
#pragma unroll 1
				for (int h = 0; h < LY::QPASS; h++) {
					u32 acc[2][QN];
#pragma unroll
					for (int q = 0; q < QN; q++) {
						acc[0][q] = acc[1][q] = 0;
					}
					stage_compute<true>(smem + s * STAGE_BYTES, lane_row, qsel * LY::QPASS + h, acc);
					if (h == 0) {
						mbar_wait(bar_eempty + eb * 8, (eit & 1) ^ 1, p.err);
						tc_fence_after();
					}
					tc_st(tmem_base + tlane + TM_EMD + eb * 128 + (qsel * LY::QPASS + h) * QN, acc[0]);
					tc_st(tmem_base + tlane + TM_EMD + eb * 128 + 64 + (qsel * LY::QPASS + h) * QN, acc[1]);
				}
				__syncwarp();
				if (lane == 0) {
					mbar_arrive(bar_empty + s * 8);
				}
				if (++s == (u32)STAGES) {
					s = 0;
					ph ^= 1;
				}
			}
			if (!INTERLEAVE && EMD && LY::QPASS == 1) {
				u32 acc[2][QN];
#pragma unroll
				for (int q = 0; q < QN; q++) {
					acc[0][q] = acc[1][q] = 0;
				}
#pragma unroll 1
				for (int c = 0; c < N_CUM; c++) {
					mbar_wait(bar_full + s * 8, ph, p.err);
					stage_compute<true>(smem + s * STAGE_BYTES, lane_row, qsel, acc);
					__syncwarp();
					if (lane == 0) {
						mbar_arrive(bar_empty + s * 8);
					}
					if (++s == (u32)STAGES) {
						s = 0;
						ph ^= 1;
					}
				}
				if (!tmem_free) {
					mbar_wait(bar_eempty + eb * 8, (eit & 1) ^ 1, p.err);
					tc_fence_after();
				}
				tc_st(tmem_base + tlane + TM_EMD + eb * 128 + qsel * QN, acc[0]);
				tc_st(tmem_base + tlane + TM_EMD + eb * 128 + 64 + qsel * QN, acc[1]);
			}
			if (CUDA_RED) {
				tc_st_wait();
				tc_fence_before();
				__syncwarp();
				if (lane == 0) {
					mbar_arrive(bar_efull + eb * 8);
				}
			}
			it++;
		}
	} else {
		// ===== epilogue warps: thread = TMEM lane (database rows L and 128 + L), all 64 query columns of each region =====
		if (REGS_EPI > REGS_LAUNCH) {
			asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
		}
		const int ew = warp - 4 - NCW;
		const int etid = threadIdx.x - (4 + NCW) * 32; // 0 .. NEW * 32 - 1
		const u32 quarter = (u32)warp & 3;
		const u32 lane_row = quarter * 32 + (u32)lane;
		const u32 tlane = (quarter * 32) << 16;
		RowF *s_rowQ = reinterpret_cast<RowF *>(smem + L::ROWQ);
		u64 *s_winQ = reinterpret_cast<u64 *>(smem + L::WINQ);
		uint2 *s_win32 = reinterpret_cast<uint2 *>(smem + L::WIN32);
		Cand *s_list = reinterpret_cast<Cand *>(smem + L::LIST) + ew * LIST_CAP;
		float *sx = reinterpret_cast<float *>(smem + L::SCRX) + etid;
#pragma unroll
		for (int t = 0; t < NP; t++) {
			sx[(scr_slot(NEED & 7, SC_COUNT) * NP + t) * (NEW * 32)] = 1.0f;
		}
		const int qc0 = (ew >> 2) * QE; // this warp's query columns: qc0 .. qc0 + QE - 1
		u32 it = 0;
		u64 scored_total = 0, exact_total = 0;
		if (COARSE && blockIdx.x == 0 && etid == 0) {
			p.counters[3] = 1;
		}
		for (u32 item = blockIdx.x; item < n_items; item += gridDim.x) {
			const Tile t = decode_item(p, s_sched, item);
			if (!t.valid) {
				continue;
			}
			const u64 qrow0 = p.q0 + (u64)t.qt * TQ, drow0 = p.d0 + (u64)t.dt * TD;
			const int par = it & 1; // query-row info is double buffered: one barrier per tile is enough
			RowF PD[2];
			u64 lenD[2];
			if (!RAW) {
				if (etid < TQ) {
					const u64 row = qrow0 + etid;
					const bool ok = row < p.q1;
					u64 len;
					s_rowQ[par * TQ + etid] = make_rowf(p.sbQ, p.csQ, COARSE ? p.smpQ : nullptr, row, ok, len);
					// FC_Runner.cpp:435-444: size_t truncation of len * id and len / id; an empty window marks an unused row
					const u64 wlo = ok ? (u64)((double)len * p.cutoff) : 1, whi = ok ? (u64)((double)len / p.cutoff) : 0;
					s_winQ[(par * TQ + etid) * 2] = wlo;
					s_winQ[(par * TQ + etid) * 2 + 1] = whi;
					// 32-bit copy for lengths below 2^32 (everything real); a saturated bound sends the pair to the 64-bit compare
					s_win32[par * TQ + etid] = make_uint2(wlo > 0xFFFFFFFFull ? 0xFFFFFFFFu : (u32)wlo, whi >= 0xFFFFFFFFull ? 0xFFFFFFFFu : (u32)whi);
				}
#pragma unroll
				for (int r = 0; r < 2; r++) {
					const u64 row = drow0 + r * 128 + lane_row;
					const bool ok = row < p.d1;
					PD[r] = make_rowf(p.sbD, p.csD, COARSE ? p.smpD : nullptr, row, ok, lenD[r]);
					if (!ok) {
						lenD[r] = ~0ull;
					}
				}
				named_sync(2, NEW * 32);
			}
			const u32 buf = it & 1;
			const u32 eb = EBUFS == 2 ? (it & 1) : 0, eit = EBUFS == 2 ? (it >> 1) : it;
			if (CUDA_RED) {
				mbar_wait(bar_efull + eb * 8, eit & 1, p.err);
			}
			if (DOT) {
				mbar_wait(bar_tfull + buf * 8, (it >> 1) & 1, p.err);
			}
			tc_fence_after();
			u32 n_list = 0, scored = 0;
#pragma unroll 1
			for (int r = 0; r < 2; r++) {
#pragma unroll 1
				for (int qc = qc0; qc < qc0 + QE; qc += NP) {
					u32 vd[NP] = {}, ve[NP] = {}, vs[NP] = {}, ve_hi[NP] = {};
					if (DOT) tc_ldn(tmem_base + tlane + TM_DOT + buf * 128 + r * 64 + qc, vd);
					if (EMD) tc_ldn(tmem_base + tlane + TM_EMD + eb * 128 + r * 64 + qc, ve);
					if (MIN) tc_ldn(tmem_base + tlane + TM_SAD + r * 64 + qc, vs);
					tc_ld_wait();
					const u64 d = drow0 + r * 128 + lane_row;
					const u32 len32 = RAW ? 0u : (lenD[r] >= 0xFFFFFFFFull ? 0xFFFFFFFFu : (u32)lenD[r]);
					if constexpr (RAW) {
#pragma unroll
						for (int k = 0; k < NP; k++) {
							const u64 q = qrow0 + qc + k;
							if (q < p.q1 && d < p.d1) {
								const u64 o = (q - p.q0) * (p.d1 - p.d0) + (d - p.d0);
								if (DOT) p.raw_dot[o] = vd[k];
								if (EMD) p.raw_emd[o] = p.csQ[q] + p.csD[d] - 2u * ve[k];
								if (MIN) p.raw_sad[o] = vs[k];
							}
						}
					} else {
						const RowF *Q = s_rowQ + par * TQ + qc;
						u32 go = 0;
#pragma unroll
						for (int k = 0; k < NP; k++) {
							const uint2 w = s_win32[par * TQ + qc + k];
							bool inwin = len32 >= w.x && len32 <= w.y;
							if (len32 == 0xFFFFFFFFu || w.y == 0xFFFFFFFFu) { // beyond 32 bits: the exact 64-bit window
								inwin = lenD[r] >= s_winQ[(par * TQ + qc + k) * 2] && lenD[r] <= s_winQ[(par * TQ + qc + k) * 2 + 1];
							}
							const bool g = inwin && (!p.upper_only || d > qrow0 + qc + k);
							go |= g ? (1u << k) : 0u;
							if constexpr (COARSE) {
								// ve = M: sum_i m_i lies in [16 (M - T), 16 M], so the EMD in [cs - 32 M, cs - 32 (M - T)]
								// (the exact EMD is >= 0, which also bounds it from below)
								const u32 cs = Q[k].cs + PD[r].cs, M32 = 32u * ve[k];
								const u32 T = min(Q[k].tot, PD[r].tot);
								ve_hi[k] = g ? cs - M32 + 32u * T : 0u;
								ve[k] = g && cs > M32 ? cs - M32 : 0u;
							} else if (EMD) {
								ve[k] = g ? Q[k].cs + PD[r].cs - 2u * ve[k] : 0u;
							}
						}
						scored += __popc(go);
						u32 cand = go;
						const bool can_screen = dm.scr_ok != 0 && n_slabs == 1; // the screen's constants and bound are for 1024 bins
						u32 anybig = PD[r].big;
#pragma unroll
						for (int k = 0; k < NP; k++) {
							anybig |= Q[k].big;
						}
						if (can_screen && __any_sync(0xffffffffu, cand != 0 && !anybig)) {
							const u32 maybe = screen_pairs<NEED, NP, COARSE, NEW * 32>(dm, sx, vd, ve, ve_hi, vs, PD[r], Q);
							if (!anybig) {
								cand &= maybe;
							}
						}
						// candidate records -> the warp's list (ballot-compacted), flushed through the exact epilogue when full
						if (__any_sync(0xffffffffu, cand != 0)) {
#pragma unroll
						for (int k = 0; k < NP; k++) {
							const bool c = (cand >> k) & 1;
							const unsigned m = __ballot_sync(0xffffffffu, c);
							if (c) {
								Cand rec;
								rec.pair = ((u32)r << 6) | (u32)(qc + k) | ((u32)lane << 8);
								rec.dot = vd[k];
								rec.emd = ve[k];
								rec.sad = vs[k];
								s_list[n_list + __popc(m & ((1u << lane) - 1))] = rec;
								if constexpr (COARSE) {
									// the flush refines one candidate at a time, and each reads both full cumulative
									// rows (cum16 is larger than L2): start bringing them into L2 now, so that the
									// flush's loads wait for L2 and not for a DRAM round trip each
									l2_prefetch(p.cumQ + (qrow0 + qc + k) * NBINS, NBINS * 2);
									l2_prefetch(p.cumD + d * NBINS, NBINS * 2);
								}
							}
							n_list += __popc(m);
						}
						}
						if (n_list > LIST_CAP - 32 * NP || (r == 1 && qc == qc0 + QE - NP)) {
							__syncwarp();
							exact_total += n_list;
							for (u32 base = 0; base < n_list; base += 32) {
								const u32 e = base + (u32)lane;
								// coarse form: the exact sum min(cumP, cumQ) of the batch's candidates, one warp per
								// candidate (lane l: bins 32 l .. 32 l + 31 of both rows), kept by the candidate's lane
								u32 smin = 0;
								if constexpr (COARSE) {
									const u32 nb = min(n_list - base, 32u);
#pragma unroll 1
									for (u32 j = 0; j < nb; j++) {
										const u32 pr = s_list[base + j].pair;
										const u64 jq = qrow0 + (pr & 63), jd = drow0 + ((pr >> 6) & 1) * 128 + quarter * 32 + ((pr >> 8) & 31);
										const uint4 *a = reinterpret_cast<const uint4 *>(p.cumQ + jq * NBINS) + lane * 4;
										const uint4 *b = reinterpret_cast<const uint4 *>(p.cumD + jd * NBINS) + lane * 4;
										uint4 A[4], B[4];
#pragma unroll
										for (int i = 0; i < 4; i++) {
											A[i] = __ldg(a + i);
											B[i] = __ldg(b + i);
										}
										u32 acc = 0;
#pragma unroll
										for (int i = 0; i < 4; i++) {
											acc = dp2a_sum(vmin2(A[i].x, B[i].x), acc);
											acc = dp2a_sum(vmin2(A[i].y, B[i].y), acc);
											acc = dp2a_sum(vmin2(A[i].z, B[i].z), acc);
											acc = dp2a_sum(vmin2(A[i].w, B[i].w), acc);
										}
										acc = __reduce_add_sync(0xffffffffu, acc);
										if ((u32)lane == j) {
											smin = acc;
										}
									}
								}
								int close = 0;
								double score = 0, d0v;
								u64 cq = 0, cd = 0;
								if (e < n_list) {
									const Cand c = s_list[e];
									cq = qrow0 + (c.pair & 63);
									cd = drow0 + ((c.pair >> 6) & 1) * 128 + quarter * 32 + ((c.pair >> 8) & 31);
									const Side sd = load_side(p.sbD, cd), sq = load_side(p.sbQ, cq);
									RedN rd;
									rd.jeff = rd.js = 0;
									rd.dot = c.dot;
									rd.emd = COARSE ? p.csQ[cq] + p.csD[cd] - 2u * smin : c.emd; // u32, as the full form's
									rd.smin = MIN ? (sd.sum + sq.sum - (u64)c.sad) >> 1 : 0;
									const int bad = eval_pair_fast(dm, (u64)n_slabs * NBINS, rd, sd, sq, true, score, d0v, close);
									if (bad) {
										atomicOr(p.err, bad & 1 ? 1 : 2);
									}
									if (p.identity) {
										close = score >= p.min_identity;
									}
								}
								const unsigned cm = __ballot_sync(0xffffffffu, close);
								u64 obase = 0;
								if (lane == 0 && cm) {
									obase = atomicAdd(p.counters, (u64)__popc(cm));
								}
								obase = __shfl_sync(0xffffffffu, obase, 0);
								if (close) {
									const u64 idx = obase + __popc(cm & ((1u << lane) - 1));
									if (idx < p.max_out) {
										p.out_q[idx] = cq;
										p.out_d[idx] = cd;
										p.out_score[idx] = score;
									}
								}
							}
							__syncwarp();
							n_list = 0;
						}
					}
				}
			}
			// TMEM reads of this tile are complete: hand the buffers back
			tc_fence_before();
			__syncwarp();
			if (lane == 0) {
				if (CUDA_RED) mbar_arrive(bar_eempty + eb * 8);
				if (DOT) mbar_arrive(bar_tempty + buf * 8);
			}
			scored_total += scored;
			it++;
		}
		if (!RAW) {
			// u64 warp sum through two 32-bit halves
			const u32 lo = __reduce_add_sync(0xffffffffu, (u32)(scored_total & 0xFFFFu));
			const u32 hi = __reduce_add_sync(0xffffffffu, (u32)(scored_total >> 16));
			if (lane == 0 && (lo | hi)) {
				atomicAdd(p.counters + 1, ((u64)hi << 16) + lo);
			}
			if (lane == 0 && exact_total) { // warp-uniform
				atomicAdd(p.counters + 2, exact_total);
			}
		}
	}
	tc_fence_before();
	__syncthreads();
	if (warp == 1) {
		asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
	}
}

// cumulative rows: warp per row, lane l owns bins [32 l, 32 l + 32); inclusive prefix, u16 (row sums < 65536), plus the
// row's sum of prefixes for the EMD identity and the samples at bins 16 j + 15 (j = 2 l, 2 l + 1) of the coarse form
__global__ void __launch_bounds__(256) cum16_kernel(const unsigned char *__restrict__ bins, u64 n, unsigned short *__restrict__ cum,
						    u32 *__restrict__ cumsum, unsigned short *__restrict__ samples)
{
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	for (u64 r = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += warps_total) {
		const uint4 *src = reinterpret_cast<const uint4 *>(bins + r * 1024 + lane * 32);
		const uint4 a = __ldg(src), b = __ldg(src + 1);
		const u32 w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
		u32 tot = 0;
#pragma unroll
		for (int i = 0; i < 8; i++) {
			tot = __dp4a(w[i], 0x01010101u, tot);
		}
		u32 x = tot;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			const u32 y = __shfl_up_sync(0xffffffffu, x, d);
			if (lane >= d) {
				x += y;
			}
		}
		u32 run = x - tot, cs = 0;
		u32 out[16];
#pragma unroll
		for (int i = 0; i < 8; i++) {
			u32 c0 = run + (w[i] & 0xFF);
			u32 c1 = c0 + ((w[i] >> 8) & 0xFF);
			u32 c2 = c1 + ((w[i] >> 16) & 0xFF);
			u32 c3 = c2 + (w[i] >> 24);
			run = c3;
			cs += c0 + c1 + c2 + c3;
			out[2 * i] = c0 | (c1 << 16);
			out[2 * i + 1] = c2 | (c3 << 16);
		}
		uint4 *dst = reinterpret_cast<uint4 *>(cum + r * 1024 + lane * 32);
		dst[0] = make_uint4(out[0], out[1], out[2], out[3]);
		dst[1] = make_uint4(out[4], out[5], out[6], out[7]);
		dst[2] = make_uint4(out[8], out[9], out[10], out[11]);
		dst[3] = make_uint4(out[12], out[13], out[14], out[15]);
		reinterpret_cast<u32 *>(samples + r * 64)[lane] = (out[7] >> 16) | (out[15] & 0xFFFF0000u); // bins 32 l + 15, 32 l + 31
		cs = __reduce_add_sync(0xffffffffu, cs);
		if (lane == 0) {
			cumsum[r] = cs;
		}
	}
}

// The general form: rows of n_slabs x 1024 bins of T (uint8 / uint16), cumulative values of (bin - base).  Both operands of
// sum |cumP - cumQ| carry the same pseudo-count per bin, so subtracting it from every bin of both rows leaves every
// difference of cumulative values unchanged -- and brings rows whose sums reach 65536 only through the 4^k pseudo-counts
// (k >= 6) back into 16 bits.  For uint16 bins the kernel also writes the row as bytes (the tensor-core and VABSDIFF4
// operands).  flags: 1 a bin below base, 2 a uint16 bin above 255, 4 a cumulative value beyond 16 bits -- any of them
// means the set cannot take the tile sweep with this base.  Rows of one slab also get the coarse form's samples (as
// cum16_kernel).
template <typename T>
__global__ void __launch_bounds__(256) cum_wide_kernel(const T *__restrict__ bins, u64 n, u32 n_slabs, u32 base, unsigned short *__restrict__ cum,
						       u32 *__restrict__ cumsum, unsigned char *__restrict__ plane, unsigned short *__restrict__ samples,
						       int *flags)
{
	const int lane = threadIdx.x & 31;
	const u64 warps_total = (u64)gridDim.x * (blockDim.x >> 5);
	const u64 N = (u64)n_slabs * 1024;
	int bad = 0;
	for (u64 r = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += warps_total) {
		u32 carry = 0, cs = 0;
		for (u32 s = 0; s < n_slabs; s++) {
			const u64 at = r * N + (u64)s * 1024 + (u64)lane * 32;
			u32 v[32];
			if (sizeof(T) == 1) {
				const uint4 *src = reinterpret_cast<const uint4 *>(bins + at);
				const uint4 a = __ldg(src), b = __ldg(src + 1);
				const u32 w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
				for (int i = 0; i < 32; i++) {
					v[i] = (w[i >> 2] >> (8 * (i & 3))) & 0xFFu;
				}
			} else {
				const uint4 *src = reinterpret_cast<const uint4 *>(bins + at);
				u32 w[16];
#pragma unroll
				for (int i = 0; i < 4; i++) {
					const uint4 a = __ldg(src + i);
					w[4 * i] = a.x; w[4 * i + 1] = a.y; w[4 * i + 2] = a.z; w[4 * i + 3] = a.w;
				}
				u32 pk[8];
#pragma unroll
				for (int i = 0; i < 32; i++) {
					v[i] = (w[i >> 1] >> (16 * (i & 1))) & 0xFFFFu;
					bad |= v[i] > 255u ? 2 : 0;
				}
#pragma unroll
				for (int i = 0; i < 8; i++) {
					pk[i] = (v[4 * i] & 0xFFu) | ((v[4 * i + 1] & 0xFFu) << 8) | ((v[4 * i + 2] & 0xFFu) << 16) | ((v[4 * i + 3] & 0xFFu) << 24);
				}
				uint4 *dp = reinterpret_cast<uint4 *>(plane + at);
				dp[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
				dp[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
			}
			u32 tot = 0;
#pragma unroll
			for (int i = 0; i < 32; i++) {
				bad |= v[i] < base ? 1 : 0;
				v[i] -= base;
				tot += v[i];
			}
			u32 x = tot;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				const u32 y = __shfl_up_sync(0xffffffffu, x, d);
				if (lane >= d) {
					x += y;
				}
			}
			u32 run = carry + x - tot;
			u32 out[16];
#pragma unroll
			for (int i = 0; i < 16; i++) {
				const u32 c0 = run + v[2 * i], c1 = c0 + v[2 * i + 1];
				run = c1;
				cs += c0 + c1;
				out[i] = (c0 & 0xFFFFu) | (c1 << 16);
			}
			bad |= run > 0xFFFFu ? 4 : 0; // cumulative values are non-decreasing: the lane's last one bounds the others
			uint4 *dst = reinterpret_cast<uint4 *>(cum + at);
			dst[0] = make_uint4(out[0], out[1], out[2], out[3]);
			dst[1] = make_uint4(out[4], out[5], out[6], out[7]);
			dst[2] = make_uint4(out[8], out[9], out[10], out[11]);
			dst[3] = make_uint4(out[12], out[13], out[14], out[15]);
			if (samples && n_slabs == 1) { // bins 32 l + 15, 32 l + 31
				reinterpret_cast<u32 *>(samples + r * 64)[lane] = (out[7] >> 16) | (out[15] & 0xFFFF0000u);
			}
			carry += __shfl_sync(0xffffffffu, x, 31);
		}
		cs = __reduce_add_sync(0xffffffffu, cs);
		if (lane == 0) {
			cumsum[r] = cs;
		}
	}
	if (bad) {
		atomicOr(flags, bad);
	}
}

// issue-rate probe: the tile sweep's inner pair of instructions (VIMNMX.U16x2 on the ALU pipe feeding IDP.2A on the FMA
// pipe), 16 independent chains per thread, 32 resident warps per SM, no memory traffic: the measured denominator of
// bench.py's roofline for the CUDA-core EMD term
__global__ void __launch_bounds__(256) issue_probe_kernel(u32 *out, u32 seed, int iters)
{
	u32 a = threadIdx.x * 2654435761u + seed, b = a ^ 0x5bd1e995u;
	u32 c[16];
#pragma unroll
	for (int i = 0; i < 16; i++) {
		c[i] = a + i;
	}
	for (int it = 0; it < iters; it++) {
#pragma unroll
		for (int i = 0; i < 16; i++) {
			u32 m;
			asm volatile("min.u16x2 %0, %1, %2;" : "=r"(m) : "r"(a), "r"(c[i]));
			asm volatile("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(c[i]) : "r"(m), "r"(0x0101u), "r"(c[i]));
		}
		a += b;
	}
	u32 s = 0;
#pragma unroll
	for (int i = 0; i < 16; i++) {
		s += c[i];
	}
	out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

} // namespace ts

// Operands of the tile sweep for one set: u16 cumulative rows of (bin - base) + their sums, and for uint16 bins the
// byte plane.  cum16_valid: 0 not built, 1 built for cum_base, -1 this set cannot be served with cum_base (cached until
// the bins change).  1 KiB uint8 rows with base 0 (the bench shape) need no check on the device and no synchronisation.
int ensure_tile_operands(mc2_ctx *ctx, const mc2_hset *hc, int base)
{
	mc2_hset *h = const_cast<mc2_hset *>(hc);
	if (h->n == 0) {
		return MC2_ERR_UNSUPPORTED;
	}
	if (h->cum16_valid != 0 && h->cum_base == base) {
		return h->cum16_valid > 0 ? MC2_OK : MC2_ERR_UNSUPPORTED;
	}
	const u64 N = h->N;
	if ((h->eb != 1 && h->eb != 2) || N % 1024 != 0 || N > 65536 || h->max_sum >= 65536 + (u64)base * N) {
		h->cum16_valid = -1;
		h->cum_base = base;
		return MC2_ERR_UNSUPPORTED;
	}
	if (!h->cum16) {
		MC2_CUDA(cudaMalloc((void **)&h->cum16, h->n * N * 2));
		MC2_CUDA(cudaMalloc((void **)&h->cumsum, h->n * 4));
	}
	if (h->eb == 2 && !h->plane8) {
		MC2_CUDA(cudaMalloc((void **)&h->plane8, h->n * N));
	}
	if (N == 1024 && !h->cum16s) {
		MC2_CUDA(cudaMalloc((void **)&h->cum16s, h->n * 64 * 2));
	}
	h->cum_base = base;
	u64 want = (h->n + 7) / 8, cap = (u64)ctx->sm_count * 8;
	int grid = (int)(want < cap ? want : cap);
	if (h->eb == 1 && N == 1024 && base == 0) {
		prof_begin(ctx, 5);
		ts::cum16_kernel<<<grid, 256, 0, ctx->stream>>>((const unsigned char *)h->bins, h->n, h->cum16, h->cumsum, h->cum16s);
		prof_end(ctx);
		ctx->launches++;
		MC2_CUDA(cudaGetLastError());
		h->cum16_valid = 1;
		return MC2_OK;
	}
	// the general form reports what it met in a word of the context's result slot (bytes 3072..3075, unused otherwise)
	int *d_flags = reinterpret_cast<int *>(reinterpret_cast<char *>(ctx->d_slot) + 3072);
	MC2_CUDA(cudaMemsetAsync(d_flags, 0, sizeof(int), ctx->stream));
	prof_begin(ctx, 5);
	if (h->eb == 1) {
		ts::cum_wide_kernel<unsigned char><<<grid, 256, 0, ctx->stream>>>((const unsigned char *)h->bins, h->n, (u32)(N / 1024), (u32)base,
										      h->cum16, h->cumsum, nullptr, h->cum16s, d_flags);
	} else {
		ts::cum_wide_kernel<unsigned short><<<grid, 256, 0, ctx->stream>>>((const unsigned short *)h->bins, h->n, (u32)(N / 1024), (u32)base,
										       h->cum16, h->cumsum, h->plane8, h->cum16s, d_flags);
	}
	prof_end(ctx);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	int flags = 0;
	MC2_CUDA(cudaMemcpyAsync(&flags, d_flags, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
	MC2_CUDA(cudaStreamSynchronize(ctx->stream));
	h->cum16_valid = flags ? -1 : 1;
	return flags ? MC2_ERR_UNSUPPORTED : MC2_OK;
}

int launch_issue_probe(mc2_ctx *ctx, int iters, u32 *d_out, u64 *warp_instr)
{
	const int grid = ctx->sm_count * 4;
	ts::issue_probe_kernel<<<grid, 256, 0, ctx->stream>>>(d_out, 1u, iters);
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	*warp_instr = (u64)grid * 8 * (u64)iters * 32; // 16 x (VIMNMX + IDP.2A) per iteration and warp
	return MC2_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
				  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
				  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn()
{
	static EncodeTiledFn fn = nullptr;
	static bool tried = false;
	if (!tried) {
		tried = true;
		void *p = nullptr;
		cudaDriverEntryPointQueryResult qr;
		if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess) {
			fn = reinterpret_cast<EncodeTiledFn>(p);
		}
	}
	return fn;
}

// rows of `row_elems` elements (u8 or u16), box = 128 bytes x `box_rows` rows, SWIZZLE_128B
static int make_map(CUtensorMap *m, const void *base, u64 n_rows, u64 row_elems, int elem_bytes, int box_rows)
{
	EncodeTiledFn fn = encode_fn();
	if (!fn) {
		set_error("tile sweep: cuTensorMapEncodeTiled is not available from this driver");
		return MC2_ERR_CUDA;
	}
	const cuuint64_t dims[2] = {row_elems, n_rows};
	const cuuint64_t strides[1] = {(cuuint64_t)row_elems * elem_bytes};
	const cuuint32_t box[2] = {(cuuint32_t)(128 / elem_bytes), (cuuint32_t)box_rows};
	const cuuint32_t es[2] = {1, 1};
	const CUresult r = fn(m, elem_bytes == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<void *>(base), dims,
			      strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
			      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
	if (r != CUDA_SUCCESS) {
		set_error("tile sweep: cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
		return MC2_ERR_CUDA;
	}
	return MC2_OK;
}

// the base both sets' cumulative rows are built with: 0 when the row sums themselves fit 16 bits, else the pseudo-count
static int tile_base(const mc2_hset *q, const mc2_hset *d)
{
	return (q->max_sum < 65536 && d->max_sum < 65536) ? 0 : 1;
}

// what the host can tell without touching the data: rows of whole 1 KiB slabs of uint8 / uint16 bins, at most 65536 bins
// (32-bit sums of 16-bit cumulative values), row sums that fit 16 bits once the pseudo-counts are taken out
bool tile_sweep_shape_ok(const mc2_hset *q, const mc2_hset *d)
{
	const int base = tile_base(q, d);
	const u64 N = q->N;
	const bool shape = q->eb == d->eb && (q->eb == 1 || q->eb == 2) && N == d->N && N % 1024 == 0 && N <= 65536 && q->n > 0 && d->n > 0 &&
			   q->n < (1ull << 31) && d->n < (1ull << 31);
	const bool sums = q->max_sum < 65536 + (u64)base * N && d->max_sum < 65536 + (u64)base * N;
	const bool known_bad = (q->cum16_valid < 0 && q->cum_base == base) || (d->cum16_valid < 0 && d->cum_base == base);
	return shape && sums && !known_bad;
}

bool tile_sweep_supported(const DevModel &dm, const mc2_hset *q, const mc2_hset *d, int identity)
{
	const bool off = getenv("MC2_SWEEP_LEGACY") != nullptr; // read per call: bench.py times both forms in one process
	if (off) {
		return false;
	}
	const bool model = dm.fast_epi && (dm.regression != 0) == (identity != 0) && !(dm.need & NEED_LOG) && (dm.need & 7) != 0;
	return model && tile_sweep_shape_ok(q, d);
}

template <int NEED, bool RAW, bool ONE, bool COARSE>
static int launch_form(int grid, cudaStream_t st, const DevModel &dm, const ts::Params &p, const CUtensorMap *m)
{
	const int smem = ts::Smem<NEED, COARSE>::TOTAL;
	MC2_CUDA(cudaFuncSetAttribute(ts::tile_sweep_kernel<NEED, RAW, ONE, COARSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
	ts::tile_sweep_kernel<NEED, RAW, ONE, COARSE><<<grid, ts::Layout<NEED, COARSE>::THREADS, smem, st>>>(dm, p, m[0], m[1], m[2], m[3]);
	return MC2_OK;
}

template <int NEED, bool RAW>
static int launch_need(int grid, cudaStream_t st, const DevModel &dm, const ts::Params &p, const CUtensorMap *m, bool coarse)
{
	if constexpr ((NEED & NEED_EMD) != 0 && !RAW) {
		if (coarse) {
			return launch_form<NEED, false, true, true>(grid, st, dm, p, m);
		}
	}
	return p.n_slabs == 1 ? launch_form<NEED, RAW, true, false>(grid, st, dm, p, m) : launch_form<NEED, RAW, false, false>(grid, st, dm, p, m);
}

int launch_tile_sweep(mc2_ctx *ctx, const DevModel &dm, int need, const mc2_hset *q, u64 q0, u64 q1, const mc2_hset *d, u64 d0, u64 d1,
		      int upper_only, double cutoff, u64 max_out, u64 *d_out_q, u64 *d_out_d, double *d_out_score, u64 *d_counters,
		      u32 *raw_dot, u32 *raw_emd, u32 *raw_sad, int identity, double min_identity)
{
	if (!ctx->d_sched) {
		MC2_CUDA(cudaMalloc(&ctx->d_sched, (ts::MAX_SUPER + 1) * 4));
	}
	u32 *d_sched = (u32 *)ctx->d_sched;
	const bool raw = raw_dot || raw_emd || raw_sad;
	int rc;
	// operands first: a set that cannot be served (a bin below the pseudo-count, a uint16 bin above 255) is known before
	// anything is written, and the caller falls back to the row-streaming kernels
	const int base = tile_base(q, d);
	if ((need & NEED_EMD) || q->eb == 2) {
		rc = ensure_tile_operands(ctx, q, base);
		if (rc == MC2_OK && d != q) rc = ensure_tile_operands(ctx, d, base);
		if (rc == MC2_ERR_UNSUPPORTED) {
			set_error("tile sweep: this set's rows do not fit the tile form");
		}
		if (rc != MC2_OK) return rc;
	}
	ts::Params p;
	memset(&p, 0, sizeof p);
	p.q0 = q0; p.q1 = q1; p.d0 = d0; p.d1 = d1;
	p.upper_only = upper_only;
	p.cutoff = cutoff;
	p.max_out = max_out;
	p.out_q = d_out_q; p.out_d = d_out_d; p.out_score = d_out_score;
	p.counters = d_counters;
	p.err = ctx->d_err;
	p.identity = identity;
	p.min_identity = min_identity;
	p.sbQ = Sideband{q->mag, q->sum, q->sumsq, q->len};
	p.sbD = Sideband{d->mag, d->sum, d->sumsq, d->len};
	p.csQ = q->cumsum; p.csD = d->cumsum;
	p.nqt = (u32)((q1 - q0 + ts::TQ - 1) / ts::TQ);
	p.ndt = (u32)((d1 - d0 + ts::TD - 1) / ts::TD);
	u32 group = 8;
	while ((p.nqt + group - 1) / group > (u32)ts::MAX_SUPER) {
		group *= 2;
	}
	p.group = group;
	p.n_super = (p.nqt + group - 1) / group;
	p.n_slabs = (u32)(q->N / 1024);
	p.sched = d_sched;
	p.raw_dot = raw_dot; p.raw_emd = raw_emd; p.raw_sad = raw_sad;
	// the kernel reads the item count from the last prefix entry; it must fit 32 bits
	if ((u64)p.n_super * group * p.ndt >= (1ull << 32)) {
		set_error("tile sweep: more than 2^32 tiles in one call; split the query range");
		return MC2_ERR_ARG;
	}
	ts::sched_kernel<<<1, 1024, 0, ctx->stream>>>(p, d_sched);
	ctx->launches++;
	CUtensorMap maps[4];
	memset(maps, 0, sizeof maps);
	// the coarse form wherever the screen runs on rows of one slab: its cumulative stage is the 64 samples per row, and
	// the full rows are read for the screen's survivors only.  Raw mode, models without a screen (an identity search
	// with t <= 0 among them) and wider rows take the full form.
	const bool coarse = (need & NEED_EMD) && !raw && p.n_slabs == 1 && dm.scr_ok && q->cum16s && d->cum16s;
	if (coarse) {
		p.cumQ = q->cum16; p.cumD = d->cum16;
		p.smpQ = q->cum16s; p.smpD = d->cum16s;
		rc = make_map(&maps[0], d->cum16s, d->n, 64, 2, ts::TD);
		if (rc != MC2_OK) return rc;
		rc = make_map(&maps[1], q->cum16s, q->n, 64, 2, ts::TQ);
		if (rc != MC2_OK) return rc;
	} else if (need & NEED_EMD) {
		rc = make_map(&maps[0], d->cum16, d->n, d->N, 2, ts::TD);
		if (rc != MC2_OK) return rc;
		rc = make_map(&maps[1], q->cum16, q->n, q->N, 2, ts::TQ);
		if (rc != MC2_OK) return rc;
	}
	if (need & (NEED_DOT | NEED_MIN)) {
		rc = make_map(&maps[2], d->eb == 2 ? (const void *)d->plane8 : d->bins, d->n, d->N, 1, ts::TD);
		if (rc != MC2_OK) return rc;
		rc = make_map(&maps[3], q->eb == 2 ? (const void *)q->plane8 : q->bins, q->n, q->N, 1, ts::TQ);
		if (rc != MC2_OK) return rc;
	}
	const int grid = ctx->sm_count;
	prof_begin(ctx, 3);
	rc = MC2_OK;
	switch (need & 7) {
#define MC2_TS_CASE(n)                                                                                  \
	case n:                                                                                         \
		rc = raw ? launch_need<n, true>(grid, ctx->stream, dm, p, maps, false)    \
			 : launch_need<n, false>(grid, ctx->stream, dm, p, maps, coarse); \
		break;
		MC2_TS_CASE(1)
		MC2_TS_CASE(2)
		MC2_TS_CASE(3)
		MC2_TS_CASE(4)
		MC2_TS_CASE(5)
		MC2_TS_CASE(6)
		MC2_TS_CASE(7)
#undef MC2_TS_CASE
	default:
		set_error("tile sweep: the model needs no reduction");
		rc = MC2_ERR_UNSUPPORTED;
	}
	prof_end(ctx);
	if (rc != MC2_OK) return rc;
	ctx->launches++;
	MC2_CUDA(cudaGetLastError());
	return MC2_OK;
}

} // namespace mc2
