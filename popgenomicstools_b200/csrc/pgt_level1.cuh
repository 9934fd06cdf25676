// pgt_level1.cuh -- level 1: sites -> unit partials.  Direct warp-per-unit kernel, the TMA-staged persistent kernel with its bulk-copy ring (also used by the sliding tile), the vectorised genotype kernel, bp-mode unit bounds
// Part of the one translation unit pgt_scan.cu (device code only; included from there, in this order:
// pgt_kernels_common.cuh, pgt_level1.cuh, pgt_level2.cuh, pgt_slide.cuh).
#ifndef PGT_LEVEL1_CUH
#define PGT_LEVEL1_CUH

// ----------------------------------------------------------------------------- level 1

// One warp per unit, persistent grid-stride over the launch's unit range.  Lane l folds sites
// l, l+32, l+64, ... of the unit in that order (all loads of a unit are issued before the first
// fold: UPL independent loads per column per lane in flight), then the butterfly.
// INDIRECT (bp mode): the unit's site range comes from `bounds` instead of the closed form.
template <class Stat, int UPL, bool INDIRECT>
__global__ void __launch_bounds__(256) k_units(DevPlan P, Cols cols, typename Stat::Acc* __restrict__ units, const uint64_t* __restrict__ bounds) {
	const uint32_t lane = threadIdx.x & 31u;
	const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const uint64_t nwarp = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	uint32_t si = 0xffffffffu;
	pgt_seg sg;
	sg.unit_base = 0;
	sg.nunits = 0;
	for (uint64_t j = P.unit_lo + warp; j < P.unit_hi; j += nwarp) {
		uint64_t i0;
		uint32_t len;
		if (INDIRECT) {
			const uint64_t b0 = bounds[j - P.unit_lo], b1 = bounds[j - P.unit_lo + 1];
			i0 = b0 + lane;
			len = (uint32_t)(b1 - b0);
		} else {
			if (si == 0xffffffffu || j - sg.unit_base >= sg.nunits) {
				si = find_seg<true>(P, j);
				sg = P.segs[si];
			}
			uint64_t st;
			len = pgt_unit_range(P.g, sg.nsites, j - sg.unit_base, &st);
			i0 = sg.site_base + st - P.site_origin + lane;
		}
		PGT_CHECK(len == 0 || (i0 - lane) + len <= P.col_elems);
		typename Stat::Acc acc = Stat::zero();
		if (UPL > 0 && len <= 32u * UPL) {
			typename Stat::Site v[UPL > 0 ? UPL : 1];
#pragma unroll
			for (int t = 0; t < UPL; ++t)
				if (lane + 32u * t < len) v[t] = Stat::load(cols, i0 + 32u * t);
#pragma unroll
			for (int t = 0; t < UPL; ++t)
				if (lane + 32u * t < len) Stat::fold(acc, v[t], cols.minind, cols.cutoff, P.site_origin + i0 + 32u * t);
		} else {
			for (uint32_t x = lane; x < len; x += 32u)
				Stat::fold(acc, Stat::load(cols, i0 + (x - lane)), cols.minind, cols.cutoff, P.site_origin + i0 + (x - lane));
		}
		acc = warp_butterfly<Stat>(acc);
		if (lane == 0) units[j - P.unit_lo] = acc;
	}
}

// Genomes of many contigs (scaffold-level assemblies: 1e3-1e6 segments, down to a few units each): deriving a
// unit's site range from its segment costs every consumer group a 72-byte segment record from L2 per unit or two.
// A one-thread-per-unit kernel writes the unit starts once (8 bytes per unit; units tile the axis, so unit j ends where
// unit j + 1 starts) and level 1 then runs its INDIRECT variant -- the same kernels bp mode uses -- with identical
// units, lanes and results.  starts[t] for t in [0, nunits]: column element index of unit unit_lo + t (the last entry:
// the end of the last unit).
__global__ void __launch_bounds__(256) k_unit_starts(DevPlan P, uint64_t* __restrict__ starts) {
	const uint64_t nu = P.unit_hi - P.unit_lo;
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t <= nu; t += stride) {
		const uint64_t j = P.unit_lo + (t < nu ? t : nu - 1);
		const pgt_seg sg = P.segs[find_seg<true>(P, j)];
		uint64_t st;
		const uint32_t len = pgt_unit_range(P.g, sg.nsites, j - sg.unit_base, &st);
		starts[t] = sg.site_base + st + (t < nu ? 0u : len) - P.site_origin;
	}
}

// ----------------------------------------------------------------------------- level 1, tiled
//
// Persistent CTAs (one per SM) walk tiles of `m` consecutive units.  Warp 0 is the producer: it
// stages the tile's slice of every column in shared memory with 1-D bulk async copies
// (cp.async.bulk -> UBLKCP, completion on an mbarrier), two stages deep, so the bytes in flight
// per SM are one whole tile (64-96 KB) and cost no registers.  Warps 1..15 are consumers: groups
// of G lanes reduce one unit each straight from shared memory (lane g of a group folds sites
// g, g+G, g+2G, ... in that order, then a log2(G)-level butterfly), so the summation order is the
// same function of (W, S, u) as in k_units and does not depend on tiles, CTAs or shards.  G is
// small when units are short (pgt_geom.gw), which keeps all lanes busy for fine windows.
// Only the 16-byte-aligned interior of a slice is bulk-copied; the <16-byte head and tail are
// copied by the producer's lanes, so nothing outside [column, column + n) is ever read.

static constexpr int kTileThreads = 512;
static constexpr int kTileMaxStages = 4;
static constexpr int kTileConsumerWarps = kTileThreads / 32 - 1;
static constexpr int kMaxTileCols = 7;  // of a statistic; the sliding tile stages `pos` as one more (kMaxStageCols)
static constexpr int kMaxStageCols = kMaxTileCols + 1;
static constexpr uint32_t kTileCtlBytes = 384;  // >= sizeof(TileCtl) = 368


// With more segments than this the tiled kernel gets a precomputed tile -> segment table: a CTA's
// consecutive tiles lie gridDim * m units apart, i.e. in different segments once contigs are shorter
// than ~1e6 sites, and the producer then paid two binary searches over the segment table per tile
// (measured: 1e3 contigs 5.5 TB/s, 1e5 contigs 2.6 TB/s, against 7.0 TB/s for 24 contigs).
static constexpr size_t kTileSegTableMin = 32;

struct TileCfg {
	const uint32_t* tile_seg;  // [ntiles] segment of each tile's first unit, or NULL (few segments / bp mode)
	const char* gcol[kMaxStageCols];  // global column pointers (element 0 = site_origin), staging order
	uint32_t elem[kMaxStageCols];     // bytes per site
	uint32_t col_off[kMaxStageCols];  // byte offset of the column's region inside a stage
	uint32_t col_cap[kMaxStageCols];  // capacity of that region in bytes
	uint32_t ncol;
	uint32_t m;            // units per tile
	uint32_t stage_bytes;
	uint32_t nstages;      // 2..kTileMaxStages
	int minind;
	double cutoff;         // XStat
	uint64_t valid_elems;  // elements every column holds from element 0 (bounds the aligned superset copies)
};

struct TileCtl {
	uint64_t full[kTileMaxStages];
	uint64_t empty[kTileMaxStages];
	uint64_t s0[kTileMaxStages];                   // column element index of the tile's first site
	uint32_t ns[kTileMaxStages];                   // elements staged (PGT_BOUNDS checks)
	const char* cp[kTileMaxStages][kMaxStageCols];  // where site s0 of each column lives (shared, or global if unstaged)
};
static_assert(sizeof(TileCtl) <= kTileCtlBytes, "control block");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
	asm volatile(
	    "{\n"
	    ".reg .pred P1;\n"
	    "LAB_WAIT:\n"
	    "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
	    "@P1 bra DONE;\n"
	    "bra LAB_WAIT;\n"
	    "DONE:\n"
	    "}\n" ::"r"(smem_u32(bar)),
	    "r"(parity)
	    : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
	             "r"(bytes), "r"(smem_u32(bar))
	             : "memory");
}

// Producer side of a stage (all 32 lanes of the producer warp; the caller has waited for the stage to
// drain): lane c stages elements [s0, s1) of column c.  The bulk copy covers the 16-byte-aligned SUPERSET
// of the slice whenever that stays inside the column (always, except at the first/last elements of a
// column that is not 16-byte aligned/padded); only then are head/tail bytes copied by hand, so nothing
// outside [column, column + valid_elems) is ever read.
__device__ __forceinline__ void producer_fill_stage(const TileCfg& tc, TileCtl* ctl, unsigned char* stages, uint32_t stg, uint64_t s0,
                                                    uint64_t s1, uint32_t lane) {
	PGT_CHECK(s0 <= s1 && s1 <= tc.valid_elems && stg < tc.nstages);
	// generic-proxy reads of this stage are done; order them before the async-proxy writes
	asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
	unsigned char* stage = stages + (size_t)stg * tc.stage_bytes;
	const uint32_t c = lane < tc.ncol ? lane : 0u;
	const char* A = tc.gcol[c] + s0 * tc.elem[c];
	const uint64_t nbytes = (s1 - s0) * tc.elem[c];
	const uint32_t pad = (uint32_t)((uintptr_t)A & 15u);
	const bool staged = lane < tc.ncol && pad + nbytes + 16u <= tc.col_cap[c];
	unsigned char* region = stage + tc.col_off[c];
	const char* col_lo = tc.gcol[c];
	const char* col_hi = tc.gcol[c] + tc.valid_elems * tc.elem[c];
	const char* B0 = A - pad;  // aligned superset [B0, B1)
	const char* B1 = (const char*)(((uintptr_t)(A + nbytes) + 15u) & ~(uintptr_t)15u);
	uint32_t nh = 0, ntl = 0;
	if (B0 < col_lo) {  // cannot read before the column: copy the head by hand
		B0 += 16;
		nh = 16u - pad;
		if (nh > nbytes) nh = (uint32_t)nbytes;
	}
	if (B1 > col_hi) {  // cannot read past the column: copy the tail by hand
		B1 -= 16;
		ntl = (uint32_t)((A + nbytes) - B1);
		if (B1 < A + nh) ntl = (uint32_t)(nbytes - nh);
	}
	uint32_t tx = (staged && B1 > B0) ? (uint32_t)(B1 - B0) : 0u;
	if (lane < tc.ncol) ctl->cp[stg][c] = staged ? (const char*)(region + pad) : A;
	uint32_t txsum = tx;
#pragma unroll
	for (int m = 16; m >= 1; m >>= 1) txsum += __shfl_xor_sync(0xffffffffu, txsum, m);
	PGT_CHECK(!tx || (B0 >= col_lo && B1 <= col_hi && (uint32_t)(pad + (B0 - A)) + tx <= tc.col_cap[c] && tc.col_off[c] + tc.col_cap[c] <= tc.stage_bytes));
	if (lane == 0) {
		ctl->s0[stg] = s0;
		ctl->ns[stg] = (uint32_t)(s1 - s0);
		mbar_arrive_expect_tx(&ctl->full[stg], txsum);
	}
	__syncwarp();
	if (tx) bulk_g2s(region + pad + (B0 - A), B0, tx, &ctl->full[stg]);
	// rare: hand-copied head / tail bytes
	const uint32_t any = __ballot_sync(0xffffffffu, staged && (nh | ntl));
	for (uint32_t cc = 0; cc < tc.ncol; ++cc) {
		if (!((any >> cc) & 1u)) continue;
		const uint32_t nh_c = __shfl_sync(0xffffffffu, nh, cc), nt_c = __shfl_sync(0xffffffffu, ntl, cc);
		const uint32_t pad_c = __shfl_sync(0xffffffffu, pad, cc);
		const unsigned long long A_c = __shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)A, cc);
		const unsigned long long nb_c = __shfl_sync(0xffffffffu, (unsigned long long)nbytes, cc);
		unsigned char* reg_c = stage + tc.col_off[cc];
		const unsigned char* Ac = (const unsigned char*)(uintptr_t)A_c;
		if (lane < nh_c) reg_c[pad_c + lane] = __ldg(Ac + lane);
		if (lane < nt_c) reg_c[pad_c + (uint32_t)(nb_c - nt_c) + lane] = __ldg(Ac + (nb_c - nt_c) + lane);
	}
	__syncwarp();
	if (lane == 0) mbar_arrive(&ctl->full[stg]);  // control words (and any head/tail bytes) are in place
}

// global site (entry) index where global unit j starts / ends
__device__ __forceinline__ uint64_t unit_bounds_global(const DevPlan& P, uint64_t j, uint64_t* end) {
	const pgt_seg sg = P.segs[find_seg<true>(P, j)];
	uint64_t st;
	const uint32_t len = pgt_unit_range(P.g, sg.nsites, j - sg.unit_base, &st);
	*end = sg.site_base + st + len;
	return sg.site_base + st;
}

__global__ void __launch_bounds__(256) k_tile_segs(DevPlan P, uint32_t m, uint64_t ntiles, uint32_t* __restrict__ tile_seg) {
	const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (t < ntiles) tile_seg[t] = find_seg<true>(P, P.unit_lo + t * m);
}

// hetWindow's 1-byte genotype column inside the tiled kernel: a warp reduces one unit from the staged tile
// with 16-byte loads + byte-SIMD compare / popc (the generic per-site loop would need one load per byte).
// The staged copy keeps the column's alignment modulo 16, so the aligned chunks are the same in shared
// memory and -- for a slice that was too long to stage -- in global memory (generic loads serve both).
// Integer counts: independent of the order, identical to the per-site fold.
// Four genotypes per word.  Both tests end in a word with 0x80 in every byte that counts, and an unsigned
// dp4a against 0x01010101 adds 128 per such byte: the accumulators hold 128 x count (shifted down once per
// unit; a lane sees < 2^25 bytes of a unit).  ~7 integer instructions per word and no POPC, which runs at a
// quarter of the integer rate (the POPC / __vcmpeq4 version needed 13 and was issue-bound at 4.5 TB/s).
__device__ __forceinline__ void het_count_word(uint32_t w, uint32_t& nonmissing128, uint32_t& nhet128) {
	nonmissing128 = __dp4a(~w & 0x80808080u, 0x01010101u, nonmissing128);  // g >= 0  (hetWindow.cpp:78): sign bit clear
	const uint32_t x = w ^ 0x01010101u;                                     // g == 1  (hetWindow.cpp:80): byte of x is zero
	const uint32_t t = (x & 0x7f7f7f7fu) + 0x7f7f7f7fu;                     // bit 7 of t | x is set iff the byte of x is not zero
	nhet128 = __dp4a(~(t | x) & 0x80808080u, 0x01010101u, nhet128);
}
__device__ __forceinline__ void het_unit_from_tile(HetStat::Acc& acc, const char* col, uint32_t rel, uint32_t len, uint32_t lane) {
	const int8_t* A = (const int8_t*)col + rel;
	const int8_t* E = A + len;
	const int8_t* A0 = (const int8_t*)(((uintptr_t)A + 15u) & ~(uintptr_t)15u);  // first aligned chunk inside
	const int8_t* A1 = (const int8_t*)((uintptr_t)E & ~(uintptr_t)15u);          // end of the last aligned chunk
	uint32_t nonmissing = 0, nhet = 0;
	if (A1 > A0) {
		const uint32_t nch = (uint32_t)(A1 - A0) >> 4;
		uint32_t nm128 = 0, h128 = 0;
		for (uint32_t c = lane; c < nch; c += 32u) {
			const uint4 v = *(reinterpret_cast<const uint4*>(A0) + c);
			het_count_word(v.x, nm128, h128);
			het_count_word(v.y, nm128, h128);
			het_count_word(v.z, nm128, h128);
			het_count_word(v.w, nm128, h128);
		}
		nonmissing = nm128 >> 7;
		nhet = h128 >> 7;
		const uint32_t nh = (uint32_t)(A0 - A), nt = (uint32_t)(E - A1);  // < 16 each
		if (lane < nh) {
			const int g = A[lane];
			nonmissing += (g >= 0);
			nhet += (g == 1);
		}
		if (lane >= 16u && lane - 16u < nt) {
			const int g = A1[lane - 16u];
			nonmissing += (g >= 0);
			nhet += (g == 1);
		}
	} else {
		for (uint32_t x = lane; x < len; x += 32u) {  // < 32 bytes without an aligned chunk
			const int g = A[x];
			nonmissing += (g >= 0);
			nhet += (g == 1);
		}
	}
	acc.nonmissing += nonmissing;
	acc.nhet += nhet;
}

template <class Stat, int G, bool INDIRECT>
__global__ void __launch_bounds__(kTileThreads, 1)
    k_units_tiled(DevPlan P, TileCfg tc, typename Stat::Acc* __restrict__ units, const uint64_t* __restrict__ bounds) {
	extern __shared__ __align__(128) unsigned char smem[];
	TileCtl* ctl = reinterpret_cast<TileCtl*>(smem);
	unsigned char* stages = smem + kTileCtlBytes;
	const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
	const uint64_t nunits = P.unit_hi - P.unit_lo;
	const uint64_t ntiles = (nunits + tc.m - 1) / tc.m;

	if (threadIdx.x == 0) {
		for (uint32_t s = 0; s < tc.nstages; ++s) {
			mbar_init(&ctl->full[s], 2);
			mbar_init(&ctl->empty[s], kTileConsumerWarps);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncthreads();

	if (warp == 0) {
		// ------------------------------------------------------------------ producer
		// lane c stages column c: the bulk copy covers the 16-byte-aligned SUPERSET of the slice
		// whenever that stays inside the column (always, except at the first/last elements of a
		// column that is not 16-byte aligned/padded); only then are head/tail bytes copied by hand.
		uint32_t it = 0;
		uint32_t psi = 0xffffffffu;  // cached segment of the producer
		pgt_seg psg;
		psg.unit_base = 0;
		psg.nunits = 0;
		auto unit_span = [&](uint64_t j, uint64_t* end) -> uint64_t {  // global [start, end) of unit j
			if (psi == 0xffffffffu || j - psg.unit_base >= psg.nunits) {
				if (tc.tile_seg && psi != 0xffffffffu && j >= psg.unit_base) {
					do {  // forward from the tile's first segment (set from the table below)
						++psi;
						psg = P.segs[psi];
					} while (j - psg.unit_base >= psg.nunits);
				} else {
					psi = find_seg<true>(P, j);
					psg = P.segs[psi];
				}
			}
			uint64_t st;
			const uint32_t len = pgt_unit_range(P.g, psg.nsites, j - psg.unit_base, &st);
			*end = psg.site_base + st + len;
			return psg.site_base + st;
		};
		for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
			const uint32_t stg = it % tc.nstages;
			// the tile's element range is computed BEFORE waiting for the stage to drain
			const uint64_t j0 = P.unit_lo + t * tc.m;
			const uint64_t j1 = (P.unit_hi - j0 < tc.m) ? P.unit_hi : j0 + tc.m;
			uint64_t s0, s1;  // element range of the tile in the columns
			if (INDIRECT) {
				s0 = bounds[j0 - P.unit_lo];
				s1 = bounds[j1 - P.unit_lo];
			} else {
				uint64_t e;
				if (tc.tile_seg) {
					const uint32_t ts = tc.tile_seg[t];
					if (ts != psi) {
						psi = ts;
						psg = P.segs[psi];
					}
				}
				s0 = unit_span(j0, &e) - P.site_origin;
				unit_span(j1 - 1, &e);
				s1 = e - P.site_origin;
			}
			if (it >= tc.nstages) mbar_wait(&ctl->empty[stg], ((it / tc.nstages) - 1u) & 1u);
			producer_fill_stage(tc, ctl, stages, stg, s0, s1, lane);
		}
	} else {
		// ------------------------------------------------------------------ consumers
		constexpr uint32_t GPW = 32u / G;  // groups per warp
		const uint32_t gl = lane % G;      // lane inside its group
		const uint32_t wgroup0 = (warp - 1u) * GPW;
		constexpr uint32_t NGROUPS = kTileConsumerWarps * GPW;
		uint32_t si = 0xffffffffu;
		pgt_seg sg;
		sg.unit_base = 0;
		sg.nunits = 0;
		uint32_t it = 0;
		for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
			const uint32_t stg = it % tc.nstages;
			mbar_wait(&ctl->full[stg], (it / tc.nstages) & 1u);
			const uint64_t s0 = ctl->s0[stg];
			const char* cp[kMaxTileCols];
#pragma unroll
			for (int c = 0; c < kMaxTileCols; ++c) cp[c] = ctl->cp[stg][c];
			const uint64_t j0 = P.unit_lo + t * tc.m;
			const uint32_t cnt = (uint32_t)((P.unit_hi - j0 < tc.m) ? (P.unit_hi - j0) : tc.m);
			// Units are dealt to the consumer groups round-robin by GLOBAL unit index, so the group that
			// gets the extra unit rotates from tile to tile and warps that finish early run ahead
			// into the next stage: no warp is systematically idle.
			const uint32_t rot = (uint32_t)((t * tc.m) % NGROUPS);
			const uint32_t myg = wgroup0 + lane / G;
			const uint32_t first = myg >= rot ? myg - rot : myg + NGROUPS - rot;
			for (uint32_t base = 0; base < cnt; base += NGROUPS) {  // warp-uniform trip count
				const uint32_t ul = base + first;
				const bool active = ul < cnt;
				const uint64_t j = j0 + (active ? ul : 0u);
				uint32_t rel, len;
				if (INDIRECT) {
					const uint64_t b0 = bounds[j - P.unit_lo], b1 = bounds[j - P.unit_lo + 1];
					rel = (uint32_t)(b0 - s0);
					len = (uint32_t)(b1 - b0);
				} else {
					if (si == 0xffffffffu || j - sg.unit_base >= sg.nunits) {
						if (tc.tile_seg) {  // forward from the tile's first segment
							if (si == 0xffffffffu || j < sg.unit_base || j - sg.unit_base >= sg.nunits + (uint64_t)tc.m) {
								si = tc.tile_seg[t];
								sg = P.segs[si];
							}
							while (j - sg.unit_base >= sg.nunits) {
								++si;
								sg = P.segs[si];
							}
						} else {
							si = find_seg<true>(P, j);
							sg = P.segs[si];
						}
					}
					uint64_t st;
					len = pgt_unit_range(P.g, sg.nsites, j - sg.unit_base, &st);
					rel = (uint32_t)(sg.site_base + st - P.site_origin - s0);
				}
				if (!active) len = 0;
				PGT_CHECK(len == 0 || (rel + len <= ctl->ns[stg] && j >= P.unit_lo && j < P.unit_hi));
				typename Stat::Acc acc = Stat::zero();
				if constexpr (std::is_same<Stat, HetStat>::value && G == 32) {
					het_unit_from_tile(acc, cp[0], rel, len, lane);
				} else {
					for (uint32_t x = gl; x < len; x += G)
						Stat::fold(acc, Stat::load_tile(cp, rel + x), tc.minind, tc.cutoff, P.site_origin + s0 + rel + x);
				}
				acc = group_butterfly<Stat, G>(acc);
				if (active && gl == 0) units[j - P.unit_lo] = acc;
			}
			__syncwarp();
			if (lane == 0) mbar_arrive(&ctl->empty[stg]);
		}
	}
}

// hetWindow's 1-byte genotype column: a warp per unit, lanes take 16-byte aligned chunks
// (LDG.128) and count with byte-SIMD + popc; the partial chunks at the two ends of the unit are
// read byte by byte, so nothing outside [unit start, unit end) is touched.  Integer counts: the
// result is independent of the order, identical to the generic kernels.
// volatile asm: the eight loads of a round stay back to back (the compiler otherwise interleaves
// them with the counting and keeps only ~3 in flight)
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
	uint4 v;
	asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
	return v;
}
template <bool INDIRECT>
__global__ void __launch_bounds__(256, 4) k_units_het_vec(DevPlan P, const int8_t* __restrict__ geno, HetStat::Acc* __restrict__ units,
                                                        const uint64_t* __restrict__ bounds) {
	const uint32_t lane = threadIdx.x & 31u;
	const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const uint64_t nwarp = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	uint32_t si = 0xffffffffu;
	pgt_seg sg;
	sg.unit_base = 0;
	sg.nunits = 0;
	for (uint64_t j = P.unit_lo + warp; j < P.unit_hi; j += nwarp) {
		uint64_t i0;
		uint32_t len;
		if (INDIRECT) {
			const uint64_t b0 = bounds[j - P.unit_lo], b1 = bounds[j - P.unit_lo + 1];
			i0 = b0;
			len = (uint32_t)(b1 - b0);
		} else {
			if (si == 0xffffffffu || j - sg.unit_base >= sg.nunits) {
				si = find_seg<true>(P, j);
				sg = P.segs[si];
			}
			uint64_t st;
			len = pgt_unit_range(P.g, sg.nsites, j - sg.unit_base, &st);
			i0 = sg.site_base + st - P.site_origin;
		}
		const int8_t* A = geno + i0;
		const int8_t* E = A + len;
		PGT_CHECK(len == 0 || i0 + len <= P.col_elems);
		const int8_t* A0 = (const int8_t*)(((uintptr_t)A + 15u) & ~(uintptr_t)15u);  // first aligned chunk inside
		const int8_t* A1 = (const int8_t*)((uintptr_t)E & ~(uintptr_t)15u);          // end of the last aligned chunk
		uint32_t nonmissing = 0, nhet = 0;
		if (A1 > A0) {
			uint32_t nm128 = 0, h128 = 0;
			const uint32_t nch = (uint32_t)(A1 - A0) >> 4;
			// 8 x 16 bytes in flight per lane (one 4096-site unit = one round); chunks past the end read
			// as 0x80 bytes = missing genotypes, which count for nothing
			const uint4 kMissing = make_uint4(0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u);
			for (uint32_t c0 = lane; c0 < nch; c0 += 256u) {
				uint4 v[8];
#pragma unroll
				for (int q = 0; q < 8; ++q) {  // unconditional loads (index clamped) so that all 8 are issued back to back
					const uint32_t c = c0 + 32u * q;
					v[q] = ldg_stream_u4(reinterpret_cast<const uint4*>(A0) + (c < nch ? c : nch - 1u));
				}
#pragma unroll
				for (int q = 0; q < 8; ++q) {
					if (c0 + 32u * q >= nch) v[q] = kMissing;
					het_count_word(v[q].x, nm128, h128);
					het_count_word(v[q].y, nm128, h128);
					het_count_word(v[q].z, nm128, h128);
					het_count_word(v[q].w, nm128, h128);
				}
			}
			nonmissing = nm128 >> 7;
			nhet = h128 >> 7;
			const uint32_t nh = (uint32_t)(A0 - A), nt = (uint32_t)(E - A1);  // < 16 each
			if (lane < nh) {
				const int g = __ldg(A + lane);
				nonmissing += (g >= 0);
				nhet += (g == 1);
			}
			if (lane >= 16u && lane - 16u < nt) {
				const int g = __ldg(A1 + (lane - 16u));
				nonmissing += (g >= 0);
				nhet += (g == 1);
			}
		} else {
			for (uint32_t x = lane; x < len; x += 32u) {  // < 32 bytes without an aligned chunk
				const int g = __ldg(A + x);
				nonmissing += (g >= 0);
				nhet += (g == 1);
			}
		}
		HetStat::Acc acc{nonmissing, nhet};
		acc = warp_butterfly<HetStat>(acc);
		if (lane == 0) units[j - P.unit_lo] = acc;
	}
}

// bp mode: the first site at or after global bp entry e of chromosome c (e inside the axis), as an index relative to
// the columns' element 0: a lower_bound of e's 1-based position in chromosome c's slice of `pos`, clipped to the
// `ndata` sites this call holds.
__device__ __forceinline__ uint64_t bp_entry_site(const DevPlan& P, const uint32_t* __restrict__ pos, uint64_t ndata, uint32_t c, uint64_t e) {
	const uint32_t p = (uint32_t)(e - P.off[c]) + 1u;
	uint64_t lo = P.site_off[c], hi = P.site_off[c + 1];
	if (lo < P.site_origin) lo = P.site_origin;
	if (hi > P.site_origin + ndata) hi = P.site_origin + ndata;
	if (hi < lo) hi = lo;
	while (lo < hi) {
		const uint64_t mid = lo + ((hi - lo) >> 1);
		if (__ldg(pos + (mid - P.site_origin)) < p) lo = mid + 1;
		else hi = mid;
	}
	if (lo < P.site_origin) lo = P.site_origin;
	if (lo > P.site_origin + ndata) lo = P.site_origin + ndata;
	return lo - P.site_origin;
}

// bp mode: bounds[t] = index (relative to the columns' element 0) of the first site at or after
// the first bp of unit unit_lo+t, t in [0, unit_hi-unit_lo]; the unit's bp -> (chromosome, pos) is
// closed form, the site is a lower_bound in that chromosome's slice of `pos`.
__global__ void __launch_bounds__(256) k_bp_bounds(DevPlan P, const uint32_t* __restrict__ pos, uint64_t ndata, uint64_t* __restrict__ bounds) {
	const uint64_t nb = P.unit_hi - P.unit_lo + 1;
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nb; t += stride) {
		const uint64_t j = P.unit_lo + t;
		uint64_t res;
		if (j >= P.nunits_total) {
			res = P.site_off[P.ncontig];
			if (res < P.site_origin) res = P.site_origin;
			if (res > P.site_origin + ndata) res = P.site_origin + ndata;
			res -= P.site_origin;
		} else {
			const pgt_seg sg = P.segs[find_seg<true>(P, j)];
			uint64_t st;
			pgt_unit_range(P.g, sg.nsites, j - sg.unit_base, &st);
			const uint64_t e = sg.site_base + st;  // global bp entry
			res = bp_entry_site(P, pos, ndata, find_contig(P.off, sg.first_contig, sg.ncontig, e), e);
		}
		bounds[t] = res;
	}
}

// bp mode: the first and last site this call holds of every chromosome must lie on the chromosome (1 <= pos <= length);
// *bad receives the smallest global index of a site that does not (left as it is when all do).  Chromosomes t0, t0 + stride, ...
__device__ __forceinline__ void bp_check_positions(const DevPlan& P, const uint32_t* __restrict__ pos, uint64_t ndata, uint64_t t0, uint64_t stride,
                                                   unsigned long long* __restrict__ bad) {
	for (uint64_t c = t0; c < P.ncontig; c += stride) {
		uint64_t lo = P.site_off[c], hi = P.site_off[c + 1];
		if (lo < P.site_origin) lo = P.site_origin;
		if (hi > P.site_origin + ndata) hi = P.site_origin + ndata;
		if (hi <= lo) continue;
		const uint64_t len = P.off[c + 1] - P.off[c];
		if (__ldg(pos + (lo - P.site_origin)) < 1u) atomicMin(bad, (unsigned long long)lo);
		else if (__ldg(pos + (hi - 1 - P.site_origin)) > len) atomicMin(bad, (unsigned long long)(hi - 1));
	}
}

// bp mode, pgt_scan_bp_sites: the number of sites on the entries of every window [win_lo, win_hi) -- the difference of
// the lower bounds of its first entry and of the entry after its last, the same searches k_bp_bounds makes for the
// units at the window's two edges.  Also the position check: the first and last site this call holds of every
// chromosome must lie on the chromosome (1 <= pos <= length); *bad receives the smallest global index of a site that
// does not (left as it is when all do).
__global__ void __launch_bounds__(256) k_bp_sites(DevPlan P, const uint32_t* __restrict__ pos, uint64_t ndata, uint32_t* __restrict__ nsites,
                                                  unsigned long long* __restrict__ bad) {
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	const uint64_t t0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint64_t axis_end = P.off[P.ncontig];
	uint32_t si = 0xffffffffu;
	pgt_seg sg;
	sg.win_base = 0;
	sg.nwin = 0;
	for (uint64_t w = P.win_lo + t0; w < P.win_hi; w += stride) {
		if (si == 0xffffffffu || w - sg.win_base >= sg.nwin) {
			si = find_seg<false>(P, w);
			sg = P.segs[si];
		}
		uint64_t fs;
		const uint32_t n = pgt_window_sites(P.g, sg, w - sg.win_base, &fs);
		const uint64_t e0 = sg.site_base + fs, e1 = e0 + n;
		const uint64_t s0 = bp_entry_site(P, pos, ndata, find_contig(P.off, sg.first_contig, sg.ncontig, e0), e0);
		uint64_t s1;
		if (e1 >= axis_end) {
			s1 = P.site_off[P.ncontig];
			s1 = (s1 < P.site_origin ? P.site_origin : (s1 > P.site_origin + ndata ? P.site_origin + ndata : s1)) - P.site_origin;
		} else {
			s1 = bp_entry_site(P, pos, ndata, find_contig(P.off, 0, P.ncontig, e1), e1);
		}
		PGT_CHECK(s0 <= s1 && s1 <= ndata);
		nsites[w - P.win_lo] = (uint32_t)(s1 - s0);
	}
	bp_check_positions(P, pos, ndata, t0, stride, bad);
}

// bp mode, the position check alone (pgt_scan_plan_extreme)
__global__ void __launch_bounds__(256) k_bp_pos_check(DevPlan P, const uint32_t* __restrict__ pos, uint64_t ndata, unsigned long long* __restrict__ bad) {
	bp_check_positions(P, pos, ndata, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, (uint64_t)gridDim.x * blockDim.x, bad);
}

#endif  // PGT_LEVEL1_CUH
