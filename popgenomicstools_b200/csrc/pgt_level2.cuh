// pgt_level2.cuh -- level 2: unit partials -> window rows.  Warp per window, thread per window for fine windows, the per-site map (W = S = 1), scan mode (block prefix / suffix scans)
// Part of the one translation unit pgt_scan.cu (device code only; included from there, in this order:
// pgt_kernels_common.cuh, pgt_level1.cuh, pgt_level2.cuh, pgt_slide.cuh).
#ifndef PGT_LEVEL2_CUH
#define PGT_LEVEL2_CUH

// ----------------------------------------------------------------------------- level 2

template <class Stat>
__device__ __forceinline__ void emit_window(const DevPlan& P, const pgt_seg& sg, uint64_t w, uint64_t k, const typename Stat::Acc& acc,
                                            const uint32_t* __restrict__ pos, const typename Stat::Out& out, uint64_t o, bool have_edges = false,
                                            uint32_t edge_start = 0, uint32_t edge_end = 0);

// two batches of 32 rows of every output column, staged in shared memory so that a block writes its rows with
// full-width stores (double-buffered: one barrier per batch).  staged(): rows of the same columns as `out`, pointing into
// the stage; store(): rows [half, half + nrows) of the stage to rows [o - lane, ...) of `out`, column f by warp f % 8.
template <class Out>
struct RowStage;
template <>
struct RowStage<pgt_windows> {
	uint32_t u[9][64];  // label, start_pos, end_pos, mid_pos, nsites, nhet, nonmissing, neffective, nskip
	double d[5][64];    // sum_a, sum_b, fst, het, dxy
	__device__ __forceinline__ pgt_windows staged(const pgt_windows& out) {
		pgt_windows st;
		st.label = out.label ? u[0] : nullptr;
		st.start_pos = out.start_pos ? u[1] : nullptr;
		st.end_pos = out.end_pos ? u[2] : nullptr;
		st.mid_pos = out.mid_pos ? u[3] : nullptr;
		st.nsites = out.nsites ? u[4] : nullptr;
		st.nhet = out.nhet ? u[5] : nullptr;
		st.nonmissing = out.nonmissing ? u[6] : nullptr;
		st.neffective = out.neffective ? u[7] : nullptr;
		st.nskip = out.nskip ? u[8] : nullptr;
		st.sum_a = out.sum_a ? d[0] : nullptr;
		st.sum_b = out.sum_b ? d[1] : nullptr;
		st.fst = out.fst ? d[2] : nullptr;
		st.het = out.het ? d[3] : nullptr;
		st.dxy = out.dxy ? d[4] : nullptr;
		st.dxy_global = nullptr;
		return st;
	}
	__device__ __forceinline__ void store(const pgt_windows& out, uint32_t half, uint64_t o, uint32_t nrows, uint32_t wi, uint32_t lane) const {
		uint32_t* const gu[9] = {out.label, out.start_pos, out.end_pos, out.mid_pos, out.nsites, out.nhet, out.nonmissing, out.neffective, out.nskip};
		double* const gd[5] = {out.sum_a, out.sum_b, out.fst, out.het, out.dxy};
#pragma unroll
		for (int f = 0; f < 9; ++f)
			if ((f & 7) == (int)wi && gu[f] && lane < nrows) gu[f][o] = u[f][half + lane];
#pragma unroll
		for (int f = 0; f < 5; ++f)
			if (((f + 9) & 7) == (int)wi && gd[f] && lane < nrows) gd[f][o] = d[f][half + lane];
	}
};
template <>
struct RowStage<XRows> {
	uint32_t u[8][64];  // label, start_pos, end_pos, mid_pos, nsites, ext_pos, nbig, xnsites
	uint64_t s[64];     // ext_site
	double d[2][64];    // ext_value, prop
	__device__ __forceinline__ XRows staged(const XRows& out) {
		XRows st;
		st.label = out.label ? u[0] : nullptr;
		st.start_pos = out.start_pos ? u[1] : nullptr;
		st.end_pos = out.end_pos ? u[2] : nullptr;
		st.mid_pos = out.mid_pos ? u[3] : nullptr;
		st.nsites = out.nsites ? u[4] : nullptr;
		st.ext_pos = out.ext_pos ? u[5] : nullptr;
		st.nbig = out.nbig ? u[6] : nullptr;
		st.xnsites = out.xnsites ? u[7] : nullptr;
		st.ext_site = out.ext_site ? s : nullptr;
		st.ext_value = out.ext_value ? d[0] : nullptr;
		st.prop = out.prop ? d[1] : nullptr;
		st.score = out.score;
		st.pos = out.pos;
		st.site_origin = out.site_origin;
		return st;
	}
	__device__ __forceinline__ void store(const XRows& out, uint32_t half, uint64_t o, uint32_t nrows, uint32_t wi, uint32_t lane) const {
		uint32_t* const gu[8] = {out.label, out.start_pos, out.end_pos, out.mid_pos, out.nsites, out.ext_pos, out.nbig, out.xnsites};
		double* const gd[2] = {out.ext_value, out.prop};
		if (lane < nrows) {
#pragma unroll
			for (int f = 0; f < 8; ++f)
				if (f == (int)wi && gu[f]) gu[f][o] = u[f][half + lane];
			if (wi == 0 && out.ext_site) out.ext_site[o] = s[half + lane];
#pragma unroll
			for (int f = 0; f < 2; ++f)
				if (f + 1 == (int)wi && gd[f]) gd[f][o] = d[f][half + lane];
		}
	}
};

// One warp per window: lane l adds unit partials l, l+32, ... (from +0.0, so a window of
// -0.0 values sums to +0.0 exactly as the reference's `double asum = 0`), then the butterfly.
// units_base = global index of units[0].
// A block owns a contiguous run of windows and walks it 32 rows at a time: warp i computes rows i, i+8, i+16, i+24 of
// the batch into shared memory, then the block stores the batch column by column, 128 / 256 bytes per store -- one row
// at a time from lane 0 was eight 4- or 8-byte stores per window, which is what a shard pays for when its rows live in
// another GPU's HBM (one NVLink packet per store).
template <class Stat>
__global__ void __launch_bounds__(256) k_windows(DevPlan P, const typename Stat::Acc* __restrict__ units, uint64_t units_base,
                                                  const uint32_t* __restrict__ pos, typename Stat::Out out) {
	__shared__ RowStage<typename Stat::Out> rows;
	const uint32_t lane = threadIdx.x & 31u, wi = threadIdx.x >> 5;
	// The per-window work is a chain of dependent memory round trips; keep it short: the segment is
	// cached (w only grows, so it changes a few dozen times per warp instead of costing a binary
	// search in global memory per window), and lane 0 fetches the two edge positions BEFORE the
	// partials are summed, so that gather overlaps the partial loads instead of following them.
	// Every block takes a contiguous run of windows, so the segment only ever moves forward by a step or
	// two: one binary search per warp, then a walk (genomes of 1e5 contigs with W larger than the contigs
	// paid a 17-probe search in L2 per window: 0.86 ms for 1e5 windows).
	uint32_t si = 0xffffffffu;
	pgt_seg sg;
	sg.win_base = 0;
	sg.nwin = 0;
	const uint64_t nwin_all = P.win_hi - P.win_lo;
	const uint64_t per = (nwin_all + gridDim.x - 1) / gridDim.x;
	const uint64_t w_begin = P.win_lo + (uint64_t)blockIdx.x * per;
	const uint64_t w_end = w_begin + per < P.win_hi ? w_begin + per : P.win_hi;
	const typename Stat::Out staged = rows.staged(out);  // the same columns as `out`, 32 rows each, in shared memory
	uint32_t half = 0;  // which 32 rows of the stage this batch uses
	for (uint64_t b0 = w_begin; b0 < w_end; b0 += 32u, half ^= 32u) {  // block-uniform
		const uint32_t nrows = (uint32_t)(w_end - b0 < 32u ? w_end - b0 : 32u);
		for (uint32_t r = wi; r < nrows; r += 8u) {
			const uint64_t w = b0 + r;
			if (si == 0xffffffffu) {
				si = find_seg<false>(P, w);
				sg = P.segs[si];
			}
			while (w - sg.win_base >= sg.nwin) {  // also skips segments without windows
				++si;
				sg = P.segs[si];
			}
			const uint64_t k = w - sg.win_base;
			uint64_t fu;
			const uint64_t cnt = pgt_window_units(P.g, sg, k, &fu);
			uint32_t sp = 0, ep = 0;
			if (lane == 0 && pos && P.mode != PGT_MODE_BP) {
				uint64_t fs;
				const uint32_t nsites = pgt_window_sites(P.g, sg, k, &fs);
				sp = __ldg(pos + (sg.site_base + fs - P.site_origin));
				ep = __ldg(pos + (sg.site_base + fs + nsites - 1 - P.site_origin));
			}
			const typename Stat::Acc* up = units + (sg.unit_base + fu - units_base);
			PGT_CHECK(sg.unit_base + fu >= P.unit_lo && sg.unit_base + fu + cnt <= P.unit_hi && w >= P.win_lo && w < P.win_hi);
			typename Stat::Acc acc = Stat::zero();
			for (uint64_t x = lane; x < cnt; x += 128u) {  // four partials per lane in flight; added in index order
				typename Stat::Acc v[4];
#pragma unroll
				for (int q = 0; q < 4; ++q)
					if (x + 32u * q < cnt) v[q] = up[x + 32u * q];
#pragma unroll
				for (int q = 0; q < 4; ++q)
					if (x + 32u * q < cnt) Stat::add(acc, v[q]);
			}
			acc = warp_butterfly<Stat>(acc);
			if (lane == 0) emit_window<Stat>(P, sg, w, k, acc, pos, staged, half + r, true, sp, ep);
		}
		__syncthreads();
		rows.store(out, half, b0 - P.win_lo + lane, nrows, wi, lane);
		// no second barrier: the next batch fills the other half, and the barrier after it orders this store before the refill
	}
}

// Fine windows (<= 32 units each): one THREAD per window, outputs written coalesced.  The value is
// bit-identical to k_windows: leaf i is (+0.0 + unit i) for i < cnt and +0.0 beyond, combined in
// the butterfly's order V(i, s) = V(i, 2s) + V(i + s, 2s), evaluated depth-first so only log2(P2)
// partials are live.
template <class Stat, int P2, int S>
struct SmallTree {
	static __device__ __forceinline__ typename Stat::Acc eval(const typename Stat::Acc* __restrict__ up, uint32_t i, uint32_t cnt) {
		typename Stat::Acc a = SmallTree<Stat, P2, S * 2>::eval(up, i, cnt);
		if (i + S < cnt) Stat::add(a, SmallTree<Stat, P2, S * 2>::eval(up, i + S, cnt));  // adding the +0.0 subtree is the identity
		return a;
	}
};
template <class Stat, int P2>
struct SmallTree<Stat, P2, P2> {
	static __device__ __forceinline__ typename Stat::Acc eval(const typename Stat::Acc* __restrict__ up, uint32_t i, uint32_t cnt) {
		typename Stat::Acc a = Stat::zero();
		if (i < cnt) Stat::add(a, up[i]);
		return a;
	}
};

template <class Stat>
__device__ __forceinline__ void emit_window(const DevPlan& P, const pgt_seg& sg, uint64_t w, uint64_t k, const typename Stat::Acc& acc,
                                            const uint32_t* __restrict__ pos, const typename Stat::Out& out, uint64_t o, bool have_edges,
                                            uint32_t edge_start, uint32_t edge_end) {
	uint64_t fs;
	const uint32_t nsites = pgt_window_sites(P.g, sg, k, &fs);
	const uint64_t first = sg.site_base + fs, last = first + nsites - 1;
	const uint32_t label = find_contig(P.off, sg.first_contig, sg.ncontig, last);
	if (out.label) out.label[o] = label;
	if (out.nsites) out.nsites[o] = nsites;
	uint32_t sp = 0, ep = 0;
	bool have = false;
	if (P.mode == PGT_MODE_BP) {
		// dxyWindow.cpp:190 prints the bp position of the first / last buffer entry
		const uint32_t cf = find_contig(P.off, sg.first_contig, sg.ncontig, first);
		sp = (uint32_t)(first - P.off[cf]) + 1u;
		ep = (uint32_t)(last - P.off[label]) + 1u;
		have = true;
	} else if (pos) {
		PGT_CHECK(first >= P.site_origin && last - P.site_origin < P.col_elems);
		sp = have_edges ? edge_start : __ldg(pos + (first - P.site_origin));  // the caller may have fetched them early
		ep = have_edges ? edge_end : __ldg(pos + (last - P.site_origin));
		have = true;
	}
	if (have) {
		if (out.start_pos) out.start_pos[o] = sp;
		if (out.end_pos) out.end_pos[o] = ep;
		if (out.mid_pos) out.mid_pos[o] = (sp + ep) / 2u;  // uint32 arithmetic, fstWindow.cpp:73
	}
	Stat::emit(out, o, acc);
}

template <class Stat, int P2>
__global__ void __launch_bounds__(256) k_windows_small(DevPlan P, const typename Stat::Acc* __restrict__ units, uint64_t units_base,
                                                        const uint32_t* __restrict__ pos, typename Stat::Out out) {
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	uint32_t si = 0xffffffffu;
	pgt_seg sg;
	sg.win_base = 0;
	sg.nwin = 0;
	for (uint64_t w = P.win_lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < P.win_hi; w += stride) {
		if (si == 0xffffffffu || w - sg.win_base >= sg.nwin) {
			si = find_seg<false>(P, w);
			sg = P.segs[si];
		}
		const uint64_t k = w - sg.win_base;
		uint64_t fu;
		const uint32_t cnt = (uint32_t)pgt_window_units(P.g, sg, k, &fu);
		PGT_CHECK(cnt <= (uint32_t)P2 && sg.unit_base + fu >= P.unit_lo && sg.unit_base + fu + cnt <= P.unit_hi);
		const typename Stat::Acc acc = SmallTree<Stat, P2, 1>::eval(units + (sg.unit_base + fu - units_base), 0u, cnt);
		emit_window<Stat>(P, sg, w, k, acc, pos, out, w - P.win_lo);
	}
}

// ----------------------------------------------------------------------------- dxyWindow's global line
//
// Block partial triples {sum of dxy, neffective, nskip} (counts carried as doubles: exact below 2^53), reduced by
// k_global_final (pgt_slide.cuh).  The per-site kernels below add their own sites' values on the way -- their windows ARE
// the sites -- so the dxy columns are read once; scans with a unit array reduce the unit partials, the sliding tile takes a
// pass over the columns (k_global_partial / k_global_sites).
static constexpr int kGlobalBlocks = 256;  // fixed (part of the summation order of the global line)
static constexpr int kGlobalMaxPartials = 4096;  // block partial triples the workspace holds (per-site kernels: one per block)

__device__ __forceinline__ void block_reduce_global(double d, unsigned long long ne, unsigned long long nk, double* __restrict__ out3) {
	__shared__ double s_d[32];
	__shared__ unsigned long long s_e[32], s_k[32];
#pragma unroll
	for (int m = 16; m >= 1; m >>= 1) {
		d = __dadd_rn(d, shfl_xor_f64(d, m));
		ne += __shfl_xor_sync(0xffffffffu, ne, m);
		nk += __shfl_xor_sync(0xffffffffu, nk, m);
	}
	if ((threadIdx.x & 31u) == 0) {
		s_d[threadIdx.x >> 5] = d;
		s_e[threadIdx.x >> 5] = ne;
		s_k[threadIdx.x >> 5] = nk;
	}
	__syncthreads();
	if (threadIdx.x < 32) {
		const uint32_t nw = blockDim.x >> 5;
		d = threadIdx.x < nw ? s_d[threadIdx.x] : 0.0;
		ne = threadIdx.x < nw ? s_e[threadIdx.x] : 0ull;
		nk = threadIdx.x < nw ? s_k[threadIdx.x] : 0ull;
#pragma unroll
		for (int m = 16; m >= 1; m >>= 1) {
			d = __dadd_rn(d, shfl_xor_f64(d, m));
			ne += __shfl_xor_sync(0xffffffffu, ne, m);
			nk += __shfl_xor_sync(0xffffffffu, nk, m);
		}
		if (threadIdx.x == 0) {
			out3[0] = d;
			out3[1] = (double)ne;
			out3[2] = (double)nk;
		}
	}
}

// what a window accumulator contributes to the global line (nothing for fst / het)
template <class Stat>
struct GlobalTerm {
	static constexpr bool has = false;
	static __device__ __forceinline__ void add(const typename Stat::Acc&, double&, unsigned long long&, unsigned long long&) {}
};
template <>
struct GlobalTerm<DxyStat> {
	static constexpr bool has = true;
	static __device__ __forceinline__ void add(const DxyStat::Acc& a, double& d, unsigned long long& ne, unsigned long long& nk) {
		d = __dadd_rn(d, a.dxy);
		ne += a.neff;
		nk += a.nskip;
	}
};
template <>
struct GlobalTerm<FusedStat> {
	static constexpr bool has = true;
	static __device__ __forceinline__ void add(const FusedStat::Acc& a, double& d, unsigned long long& ne, unsigned long long& nk) {
		GlobalTerm<DxyStat>::add(a.dxy, d, ne, nk);
	}
};

// W = S = 1 (the tools' default arguments): every window is one site, so the window table is an
// elementwise map of the columns; level 1 is skipped and the per-site statistic is evaluated here.
// Output-bound (36-76 bytes of rows per 1-41 bytes of site): a thread takes four windows per turn and issues
// their column loads together before the first row is stored; the label comes from a cached contig range
// instead of a binary search per window.
template <class Stat>
__global__ void __launch_bounds__(256) k_windows_persite(DevPlan P, Cols cols, typename Stat::Out out, double* __restrict__ gpart) {
	constexpr int U = 4;
	double gd = 0.0;  // this thread's share of the global line (gpart != NULL: one partial triple per block)
	unsigned long long gne = 0, gnk = 0;
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	uint32_t si = 0xffffffffu;
	pgt_seg sg;
	sg.win_base = 0;
	sg.nwin = 0;
	uint32_t lc = 0;
	uint64_t lc_lo = 1, lc_hi = 0;  // sites of contig lc: [lc_lo, lc_hi); empty = nothing cached
	for (uint64_t w0 = P.win_lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w0 < P.win_hi; w0 += U * stride) {
		uint64_t site[U];
		typename Stat::Site v[U];
		uint32_t ps[U];
#pragma unroll
		for (int q = 0; q < U; ++q) {
			const uint64_t w = w0 + q * stride;
			site[q] = ~0ull;
			if (w >= P.win_hi) continue;
			if (si == 0xffffffffu || w - sg.win_base >= sg.nwin) {
				si = find_seg<false>(P, w);
				sg = P.segs[si];
			}
			site[q] = sg.site_base + (w - sg.win_base);  // window k of a segment is its site k
		}
#pragma unroll
		for (int q = 0; q < U; ++q) {
			if (site[q] == ~0ull) continue;
			PGT_CHECK(site[q] >= P.site_origin && site[q] - P.site_origin < P.col_elems);
			v[q] = Stat::load(cols, site[q] - P.site_origin);
			ps[q] = cols.pos ? __ldg(cols.pos + (site[q] - P.site_origin)) : 0u;
		}
#pragma unroll
		for (int q = 0; q < U; ++q) {
			if (site[q] == ~0ull) continue;
			const uint64_t o = w0 + q * stride - P.win_lo;
			if (site[q] < lc_lo || site[q] >= lc_hi) {
				lc = find_contig(P.off, 0, P.ncontig, site[q]);
				lc_lo = P.off[lc];
				lc_hi = P.off[lc + 1];
			}
			typename Stat::Acc acc = Stat::zero();
			Stat::fold(acc, v[q], cols.minind, cols.cutoff, site[q]);
			if (GlobalTerm<Stat>::has && gpart) GlobalTerm<Stat>::add(acc, gd, gne, gnk);
			if (out.label) out.label[o] = lc;
			if (out.nsites) out.nsites[o] = 1u;
			if (cols.pos) {
				if (out.start_pos) out.start_pos[o] = ps[q];
				if (out.end_pos) out.end_pos[o] = ps[q];
				if (out.mid_pos) out.mid_pos[o] = (ps[q] + ps[q]) / 2u;  // uint32 arithmetic, fstWindow.cpp:73
			}
			Stat::emit(out, o, acc);
		}
	}
	if (GlobalTerm<Stat>::has && gpart) block_reduce_global(gd, gne, gnk, gpart + 3 * blockIdx.x);  // gpart is grid-uniform
}

// The same map with FOUR CONSECUTIVE windows per thread and 128-bit loads and stores: the scalar kernel above spends ~130
// instructions per window on 64-bit addresses, NULL checks and predicates for eight 4- or 8-byte stores (ncu: issue-bound
// at 4.6 TB/s where a plain fill reaches 7.5 TB/s).  Preconditions, checked on the host (else the scalar kernel runs): the
// scan's windows lie in ONE segment (always so for W = S = 1: the reference's buffer is exactly full at every contig
// change, so all contigs chain up), and every column / output pointer is 16-byte aligned at the scan's first window.
// site0 = column element index of window win_lo.
// Four doubles are one 256-bit access (LDG/STG.E.ENL2.256, sm_100) when the address allows it: a warp then covers 1 KB of
// full 32-byte sectors per instruction.  As two 128-bit halves each instruction touched every other half-sector
// (ncu: 26 of 32 bytes per sector used by the stores of the per-site kernel).
__device__ __forceinline__ void ld4(const double* p, double* v) {
	if ((reinterpret_cast<uintptr_t>(p) & 31u) == 0) {
		asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p));
		return;
	}
	const double2 a = __ldg(reinterpret_cast<const double2*>(p)), b = __ldg(reinterpret_cast<const double2*>(p) + 1);
	v[0] = a.x;
	v[1] = a.y;
	v[2] = b.x;
	v[3] = b.y;
}
__device__ __forceinline__ void ld4(const int32_t* p, int* v) {
	const int4 a = __ldg(reinterpret_cast<const int4*>(p));
	v[0] = a.x;
	v[1] = a.y;
	v[2] = a.z;
	v[3] = a.w;
}
__device__ __forceinline__ void ld4(const uint32_t* p, uint32_t* v) {
	const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
	v[0] = a.x;
	v[1] = a.y;
	v[2] = a.z;
	v[3] = a.w;
}
__device__ __forceinline__ void ld4(const int8_t* p, int* v) {
	const uint32_t a = __ldg(reinterpret_cast<const uint32_t*>(p));
	v[0] = (int)(int8_t)(a & 0xffu);
	v[1] = (int)(int8_t)((a >> 8) & 0xffu);
	v[2] = (int)(int8_t)((a >> 16) & 0xffu);
	v[3] = (int)(int8_t)(a >> 24);
}
__device__ __forceinline__ void st4(uint32_t* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
	if (p) *reinterpret_cast<uint4*>(p) = make_uint4(a, b, c, d);
}
__device__ __forceinline__ void st4(double* p, double a, double b, double c, double d) {
	if (!p) return;
	if ((reinterpret_cast<uintptr_t>(p) & 31u) == 0) {
		asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
		return;
	}
	reinterpret_cast<double2*>(p)[0] = make_double2(a, b);
	reinterpret_cast<double2*>(p)[1] = make_double2(c, d);
}
// sites i .. i+3 of the statistic's columns
__device__ __forceinline__ void load4(const Cols& c, uint64_t i, FstStat::Site* s) {
	double a[4], b[4];
	ld4(c.a + i, a);
	ld4(c.b + i, b);
#pragma unroll
	for (int q = 0; q < 4; ++q) s[q] = FstStat::Site{a[q], b[q]};
}
__device__ __forceinline__ void load4(const Cols& c, uint64_t i, HetStat::Site* s) {
	int g[4];
	ld4(c.g + i, g);
#pragma unroll
	for (int q = 0; q < 4; ++q) s[q] = HetStat::Site{g[q]};
}
__device__ __forceinline__ void load4(const Cols& c, uint64_t i, DxyStat::Site* s) {
	double f1[4], f2[4];
	int n1[4], n2[4];
	ld4(c.f1 + i, f1);
	ld4(c.f2 + i, f2);
	ld4(c.n1 + i, n1);
	ld4(c.n2 + i, n2);
#pragma unroll
	for (int q = 0; q < 4; ++q) s[q] = DxyStat::Site{f1[q], f2[q], n1[q], n2[q]};
}
__device__ __forceinline__ void load4(const Cols& c, uint64_t i, FusedStat::Site* s) {
	FstStat::Site f[4];
	DxyStat::Site d[4];
	HetStat::Site h[4];
	load4(c, i, f);
	load4(c, i, d);
	load4(c, i, h);
#pragma unroll
	for (int q = 0; q < 4; ++q) s[q] = FusedStat::Site{f[q], d[q], h[q]};
}
// rows o .. o+3 of the statistic's output columns (the values of Stat::emit, four at a time)
__device__ __forceinline__ void emit4(const pgt_windows& out, uint64_t o, const FstStat::Acc* a) {
	st4(out.sum_a ? out.sum_a + o : nullptr, a[0].a, a[1].a, a[2].a, a[3].a);
	st4(out.sum_b ? out.sum_b + o : nullptr, a[0].b, a[1].b, a[2].b, a[3].b);
	if (out.fst) {
		double f[4];
#pragma unroll
		for (int q = 0; q < 4; ++q) f[q] = a[q].b != 0.0 ? __ddiv_rn(a[q].a, a[q].b) : 0.0;
		st4(out.fst + o, f[0], f[1], f[2], f[3]);
	}
}
__device__ __forceinline__ void emit4(const pgt_windows& out, uint64_t o, const HetStat::Acc* a) {
	st4(out.nhet ? out.nhet + o : nullptr, a[0].nhet, a[1].nhet, a[2].nhet, a[3].nhet);
	st4(out.nonmissing ? out.nonmissing + o : nullptr, a[0].nonmissing, a[1].nonmissing, a[2].nonmissing, a[3].nonmissing);
	if (out.het) {
		double h[4];
#pragma unroll
		for (int q = 0; q < 4; ++q) h[q] = a[q].nonmissing ? (double)a[q].nhet : 0.0;  // one site: nhet / 1
		st4(out.het + o, h[0], h[1], h[2], h[3]);
	}
}
__device__ __forceinline__ void emit4(const pgt_windows& out, uint64_t o, const DxyStat::Acc* a) {
	st4(out.dxy ? out.dxy + o : nullptr, a[0].dxy, a[1].dxy, a[2].dxy, a[3].dxy);
	st4(out.neffective ? out.neffective + o : nullptr, a[0].neff, a[1].neff, a[2].neff, a[3].neff);
	st4(out.nskip ? out.nskip + o : nullptr, a[0].nskip, a[1].nskip, a[2].nskip, a[3].nskip);
}
__device__ __forceinline__ void emit4(const pgt_windows& out, uint64_t o, const FusedStat::Acc* a) {
	FstStat::Acc f[4];
	DxyStat::Acc d[4];
	HetStat::Acc h[4];
#pragma unroll
	for (int q = 0; q < 4; ++q) {
		f[q] = a[q].fst;
		d[q] = a[q].dxy;
		h[q] = a[q].het;
	}
	emit4(out, o, f);
	emit4(out, o, d);
	emit4(out, o, h);
}

template <class Stat>
__global__ void __launch_bounds__(256) k_windows_persite4(DevPlan P, Cols cols, pgt_windows out, uint64_t site0, double* __restrict__ gpart) {
	double gd = 0.0;  // this thread's share of the global line (gpart != NULL: one partial triple per block)
	unsigned long long gne = 0, gnk = 0;
	const uint64_t nwin = P.win_hi - P.win_lo;
	const uint64_t ngroups = (nwin + 3) / 4;
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	uint32_t lc = 0;
	uint64_t lc_lo = 1, lc_hi = 0;  // global sites of contig lc: [lc_lo, lc_hi); empty = nothing cached
	// The loads of a thread's NEXT turn are issued before the rows of this turn are stored, so a warp always has column
	// loads in flight behind its store burst (the rows are 36-76 bytes per 1-41 bytes read: without this a warp sat out a
	// full DRAM round trip per turn with nothing outstanding).
	typename Stat::Site v[4];
	uint32_t ps[4] = {0u, 0u, 0u, 0u};
	{
		const uint64_t g0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
		if (g0 < ngroups && nwin - 4 * g0 >= 4) {
			PGT_CHECK(site0 + 4 * g0 + 4 <= P.col_elems);
			load4(cols, site0 + 4 * g0, v);
			if (cols.pos) ld4(cols.pos + site0 + 4 * g0, ps);
		}
	}
	for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
		const uint64_t o = 4 * g, i = site0 + o, gs = P.site_origin + i;
		if (nwin - o >= 4) {
			typename Stat::Site vn[4];
			uint32_t pn[4] = {0u, 0u, 0u, 0u};
			const uint64_t gn = g + stride;
			const bool more = gn < ngroups && nwin - 4 * gn >= 4;
			if (more) {
				PGT_CHECK(site0 + 4 * gn + 4 <= P.col_elems);
				load4(cols, site0 + 4 * gn, vn);
				if (cols.pos) ld4(cols.pos + site0 + 4 * gn, pn);
			}
			uint32_t lab[4];
#pragma unroll
			for (int q = 0; q < 4; ++q) {
				if (gs + q < lc_lo || gs + q >= lc_hi) {  // (rare: at most once per contig and thread)
					lc = find_contig(P.off, 0, P.ncontig, gs + q);
					lc_lo = P.off[lc];
					lc_hi = P.off[lc + 1];
				}
				lab[q] = lc;
			}
			typename Stat::Acc acc[4];
#pragma unroll
			for (int q = 0; q < 4; ++q) {
				acc[q] = Stat::zero();
				Stat::fold(acc[q], v[q], cols.minind, cols.cutoff, gs + q);
				if (GlobalTerm<Stat>::has && gpart) GlobalTerm<Stat>::add(acc[q], gd, gne, gnk);
			}
			st4(out.label ? out.label + o : nullptr, lab[0], lab[1], lab[2], lab[3]);
			st4(out.nsites ? out.nsites + o : nullptr, 1u, 1u, 1u, 1u);
			if (cols.pos) {
				st4(out.start_pos ? out.start_pos + o : nullptr, ps[0], ps[1], ps[2], ps[3]);
				st4(out.end_pos ? out.end_pos + o : nullptr, ps[0], ps[1], ps[2], ps[3]);
				// (start + end) / 2 in uint32 arithmetic, fstWindow.cpp:73
				st4(out.mid_pos ? out.mid_pos + o : nullptr, (ps[0] + ps[0]) / 2u, (ps[1] + ps[1]) / 2u, (ps[2] + ps[2]) / 2u, (ps[3] + ps[3]) / 2u);
			}
			emit4(out, o, acc);
			if (more) {
#pragma unroll
				for (int q = 0; q < 4; ++q) {
					v[q] = vn[q];
					ps[q] = pn[q];
				}
			}
		} else {
			for (uint64_t q = 0; o + q < nwin; ++q) {  // the last one to three windows of the scan
				PGT_CHECK(i + q < P.col_elems);
				typename Stat::Acc acc = Stat::zero();
				Stat::fold(acc, Stat::load(cols, i + q), cols.minind, cols.cutoff, gs + q);
				if (GlobalTerm<Stat>::has && gpart) GlobalTerm<Stat>::add(acc, gd, gne, gnk);
				const uint32_t ps = cols.pos ? __ldg(cols.pos + i + q) : 0u;
				lc = find_contig(P.off, 0, P.ncontig, gs + q);
				if (out.label) out.label[o + q] = lc;
				if (out.nsites) out.nsites[o + q] = 1u;
				if (cols.pos) {
					if (out.start_pos) out.start_pos[o + q] = ps;
					if (out.end_pos) out.end_pos[o + q] = ps;
					if (out.mid_pos) out.mid_pos[o + q] = (ps + ps) / 2u;
				}
				Stat::emit(out, o + q, acc);
			}
		}
	}
	if (GlobalTerm<Stat>::has && gpart) block_reduce_global(gd, gne, gnk, gpart + 3 * blockIdx.x);  // gpart is grid-uniform
}

// ----------------------------------------------------------------------------- level 2, scan mode
//
// Fine steps with long windows (e.g. W = 1000, S = 1): summing W/S unit partials per window
// would cost O(n * W / S^2).  Instead the unit array is cut into blocks of B = wunits units
// (aligned to the segment's first unit), and an inclusive prefix scan PRE and suffix scan SUF are
// taken inside every block.  A window covers at most two adjacent blocks, so
//     window = SUF[first unit] + PRE[last unit]          (van Herk / Gil-Werman)
// -- two reads per window, only additions of true partial sums (no subtraction, no cancellation).
// Order inside a block: chunks of 256 units; warp shuffle scan, warp totals, running carry.

template <class Acc>
__device__ __forceinline__ Acc shfl_up_acc(const Acc& v, unsigned delta) {
	static_assert(sizeof(Acc) % 4 == 0, "Acc is made of 32-bit words");
	uint32_t w[sizeof(Acc) / 4];
	memcpy(w, &v, sizeof(Acc));
#pragma unroll
	for (unsigned i = 0; i < sizeof(Acc) / 4; ++i) w[i] = __shfl_up_sync(0xffffffffu, w[i], delta);
	Acc r;
	memcpy(&r, w, sizeof(Acc));
	return r;
}

// one direction of the block scan: items x0 + i (forward) or x1 - 1 - i (backward), i = 0..n-1
template <class Stat, bool BACKWARD>
__device__ __forceinline__ void cta_scan_dir(const typename Stat::Acc* __restrict__ in, typename Stat::Acc* __restrict__ outp, uint64_t x0, uint64_t x1,
                                             typename Stat::Acc* s_wtot, typename Stat::Acc* s_carry) {
	typedef typename Stat::Acc Acc;
	const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
	const uint64_t n = x1 - x0;
	if (threadIdx.x == 0) *s_carry = Stat::zero();
	__syncthreads();
	for (uint64_t base = 0; base < n; base += blockDim.x) {
		const uint64_t i = base + threadIdx.x;
		const bool ok = i < n;
		const uint64_t idx = BACKWARD ? (x1 - 1 - i) : (x0 + i);
		Acc v = Stat::zero();
		if (ok) Stat::add(v, in[idx]);
		// inclusive scan inside the warp
#pragma unroll
		for (unsigned d = 1; d < 32; d <<= 1) {
			Acc o = shfl_up_acc(v, d);
			if (lane >= d) {
				Acc t = o;          // earlier items first: t = earlier + v
				Stat::add(t, v);
				v = t;
			}
		}
		if (lane == 31) s_wtot[warp] = v;
		__syncthreads();
		Acc pre = *s_carry;  // everything before this chunk
		for (uint32_t w = 0; w < warp; ++w) Stat::add(pre, s_wtot[w]);
		Stat::add(pre, v);
		if (ok) outp[idx] = pre;
		__syncthreads();
		if (threadIdx.x == blockDim.x - 1) *s_carry = pre;  // inclusive total through this chunk
		__syncthreads();
	}
}

template <class Stat>
__global__ void __launch_bounds__(256) k_block_scan(DevPlan P, typename Stat::Acc* __restrict__ units, typename Stat::Acc* __restrict__ pre,
                                                     uint64_t units_base, uint64_t blk_lo, uint64_t blk_hi) {
	__shared__ typename Stat::Acc s_wtot[8];
	__shared__ typename Stat::Acc s_carry;
	const uint64_t B = P.g.wunits;
	for (uint64_t gb = blk_lo + blockIdx.x; gb < blk_hi; gb += gridDim.x) {
		const pgt_seg sg = P.segs[find_seg_by_block(P, gb)];
		const uint64_t lb = gb - sg.blk_base;
		uint64_t u0 = sg.unit_base + lb * B;
		uint64_t u1 = sg.unit_base + ((lb + 1) * B < sg.nunits ? (lb + 1) * B : sg.nunits);
		// clip to the units this scan computed (shards): see DESIGN.md, the clipped values are never used
		if (u0 < P.unit_lo) u0 = P.unit_lo;
		if (u1 > P.unit_hi) u1 = P.unit_hi;
		if (u1 <= u0) continue;
		PGT_CHECK(u0 >= units_base && u0 >= P.unit_lo && u1 <= P.unit_hi);
		cta_scan_dir<Stat, false>(units, pre, u0 - units_base, u1 - units_base, s_wtot, &s_carry);  // PRE (reads raw units)
		cta_scan_dir<Stat, true>(units, units, u0 - units_base, u1 - units_base, s_wtot, &s_carry);  // SUF in place
	}
}

template <class Stat>
__global__ void __launch_bounds__(256) k_windows_hgw(DevPlan P, const typename Stat::Acc* __restrict__ suf, const typename Stat::Acc* __restrict__ pre,
                                                      uint64_t units_base, const uint32_t* __restrict__ pos, typename Stat::Out out) {
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	const uint64_t B = P.g.wunits;
	uint32_t si = 0xffffffffu;
	pgt_seg sg;
	sg.win_base = 0;
	sg.nwin = 0;
	for (uint64_t w = P.win_lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < P.win_hi; w += stride) {
		if (si == 0xffffffffu || w - sg.win_base >= sg.nwin) {
			si = find_seg<false>(P, w);
			sg = P.segs[si];
		}
		const uint64_t k = w - sg.win_base;
		uint64_t fu;
		const uint64_t cnt = pgt_window_units(P.g, sg, k, &fu);
		const uint64_t lu = fu + cnt - 1;  // segment-local first / last unit
		const uint64_t gf = sg.unit_base + fu - units_base, gl = sg.unit_base + lu - units_base;
		PGT_CHECK(sg.unit_base + fu >= P.unit_lo && sg.unit_base + lu < P.unit_hi);
		typename Stat::Acc acc = Stat::zero();
		if (fu / B == lu / B) {
			// inside one block: block-aligned start (PRE up to the last unit), or it runs to the block /
			// segment end (SUF from the first unit)
			if (fu % B == 0) Stat::add(acc, pre[gl]);
			else Stat::add(acc, suf[gf]);
		} else {
			Stat::add(acc, suf[gf]);
			Stat::add(acc, pre[gl]);
		}
		emit_window<Stat>(P, sg, w, k, acc, pos, out, w - P.win_lo);
	}
}

#endif  // PGT_LEVEL2_CUH
