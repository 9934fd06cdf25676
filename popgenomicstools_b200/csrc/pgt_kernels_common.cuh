// pgt_kernels_common.cuh -- device-side plan, search helpers, the PGT_BOUNDS check and the statistics (what one site contributes, how partials combine, what a window row holds)
// Part of the one translation unit pgt_scan.cu (device code only; included from there, in this order:
// pgt_kernels_common.cuh, pgt_level1.cuh, pgt_level2.cuh, pgt_slide.cuh).
#ifndef PGT_KERNELS_COMMON_CUH
#define PGT_KERNELS_COMMON_CUH

// -DPGT_BOUNDS (make -C csrc bounds -> libpgtscan_bounds.so): every index a kernel forms from the plan is checked
// against the extent it must stay in -- column slices against the elements the caller's columns hold, positions
// inside a shared-memory stage against the staged slice, unit / window / block indices against this launch's ranges
// -- and a violation traps (the launch fails with an error instead of reading or writing out of bounds).  The GPU
// test-suite is run against this build with PGT_LIB=.../libpgtscan_bounds.so (tools/run_bounds_gpu.sh).
#ifdef PGT_BOUNDS
#define PGT_CHECK(cond)                                                                             \
	do {                                                                                            \
		if (!(cond)) {                                                                              \
			printf("PGT_BOUNDS violated at %s:%d: %s\n", __FILE__, __LINE__, #cond);                \
			__trap();                                                                               \
		}                                                                                           \
	} while (0)
#else
#define PGT_CHECK(cond) ((void)0)
#endif

// ----------------------------------------------------------------------------- device plan

struct Cols {
	const uint32_t* pos;
	const double* a;
	const double* b;
	const int8_t* g;
	const double* f1;
	const double* f2;
	const int32_t* n1;
	const int32_t* n2;
	const double* score;  // extreme scan over a window plan (XStat)
	int minind;
	double cutoff;  // XStat
};

struct DevPlan {
	pgt_geom g;
	const pgt_seg* segs;
	const uint64_t* off;       // contig offsets on the plan axis (sites, or bp entries)
	const uint64_t* site_off;  // bp mode: cumulative site counts per chromosome (global site indices)
	uint32_t nseg;
	uint32_t ncontig;
	uint64_t unit_lo, unit_hi;  // global unit range reduced by this launch
	uint64_t win_lo, win_hi;    // global window range of this scan
	uint64_t site_origin;       // global index of element 0 of the columns
	uint64_t nunits_total;
	uint64_t col_elems;         // elements the columns hold from element 0 (PGT_BOUNDS checks; ~0 = unknown)
	int mode;
};

// last segment with key <= x, key = unit_base (BY_UNIT) or win_base
template <bool BY_UNIT>
__device__ __forceinline__ uint32_t find_seg(const DevPlan& P, uint64_t x) {
	uint32_t lo = 0, hi = P.nseg;
	while (hi - lo > 1) {
		uint32_t mid = lo + ((hi - lo) >> 1);
		uint64_t key = BY_UNIT ? P.segs[mid].unit_base : P.segs[mid].win_base;
		if (key <= x) lo = mid;
		else hi = mid;
	}
	return lo;
}
// last segment with blk_base <= x AND at least one scan block
__device__ __forceinline__ uint32_t find_seg_by_block(const DevPlan& P, uint64_t x) {
	uint32_t lo = 0, hi = P.nseg;
	while (hi - lo > 1) {
		uint32_t mid = lo + ((hi - lo) >> 1);
		if (P.segs[mid].blk_base <= x) lo = mid;
		else hi = mid;
	}
	return lo;
}

// contig c in [c0, c0+nc) with off[c] <= x < off[c+1]
__device__ __forceinline__ uint32_t find_contig(const uint64_t* off, uint32_t c0, uint32_t nc, uint64_t x) {
	uint32_t lo = c0, hi = c0 + nc;
	while (hi - lo > 1) {
		uint32_t mid = lo + ((hi - lo) >> 1);
		if (off[mid] <= x) lo = mid;
		else hi = mid;
	}
	return lo;
}

__device__ __forceinline__ double shfl_xor_f64(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ uint32_t shfl_xor_u32(uint32_t v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }

// ----------------------------------------------------------------------------- statistics
//
// A Stat describes: the per-site record loaded from the columns (Site), the unit partial (Acc,
// stored as-is in the unit array), how one site is folded into a lane's partial (the per-site
// statistic; fold also gets dxyWindow's -minind, the extreme scan's cutoff and the site's global
// index, which only XStat reads), the combine used by the butterflies, and the window epilogue
// into the rows of type Out.

// --- fstWindow: asum += a; bsum += b (fstWindow.cpp:80-83); fst = bsum != 0 ? asum/bsum : 0 (:85)
struct FstStat {
	typedef pgt_windows Out;
	struct Acc {
		double a, b;
	};
	struct Site {
		double a, b;
	};
	static __device__ __forceinline__ Acc zero() { return Acc{0.0, 0.0}; }
	static __device__ __forceinline__ Site load(const Cols& c, uint64_t i) { return Site{__ldg(c.a + i), __ldg(c.b + i)}; }
	// tile columns in staging order (a, b); generic loads: the tile lives in shared memory
	static __device__ __forceinline__ Site load_tile(const char* const* cp, uint32_t i) {
		return Site{((const double*)cp[0])[i], ((const double*)cp[1])[i]};
	}
	static __device__ __forceinline__ void fold(Acc& acc, const Site& s, int, double, uint64_t) {
		acc.a = __dadd_rn(acc.a, s.a);
		acc.b = __dadd_rn(acc.b, s.b);
	}
	static __device__ __forceinline__ void add(Acc& acc, const Acc& o) {
		acc.a = __dadd_rn(acc.a, o.a);
		acc.b = __dadd_rn(acc.b, o.b);
	}
	static __device__ __forceinline__ Acc shfl_xor(const Acc& v, int m) { return Acc{shfl_xor_f64(v.a, m), shfl_xor_f64(v.b, m)}; }
	static __device__ __forceinline__ void emit(const pgt_windows& out, uint64_t o, const Acc& acc) {
		if (out.sum_a) out.sum_a[o] = acc.a;
		if (out.sum_b) out.sum_b[o] = acc.b;
		if (out.fst) out.fst[o] = acc.b != 0.0 ? __ddiv_rn(acc.a, acc.b) : 0.0;
	}
};

// --- hetWindow: nonmissing += (g >= 0); nhet += (g == 1) (hetWindow.cpp:77-82); h = nhet/nonmissing (:84)
struct HetStat {
	typedef pgt_windows Out;
	struct Acc {
		uint32_t nonmissing, nhet;
	};
	struct Site {
		int g;
	};
	static __device__ __forceinline__ Acc zero() { return Acc{0u, 0u}; }
	static __device__ __forceinline__ Site load(const Cols& c, uint64_t i) { return Site{(int)__ldg(c.g + i)}; }
	static __device__ __forceinline__ Site load_tile(const char* const* cp, uint32_t i) { return Site{(int)((const int8_t*)cp[0])[i]}; }
	static __device__ __forceinline__ void fold(Acc& acc, const Site& s, int, double, uint64_t) {
		acc.nonmissing += (s.g >= 0);
		acc.nhet += (s.g == 1);
	}
	static __device__ __forceinline__ void add(Acc& acc, const Acc& o) {
		acc.nonmissing += o.nonmissing;
		acc.nhet += o.nhet;
	}
	static __device__ __forceinline__ Acc shfl_xor(const Acc& v, int m) { return Acc{shfl_xor_u32(v.nonmissing, m), shfl_xor_u32(v.nhet, m)}; }
	static __device__ __forceinline__ void emit(const pgt_windows& out, uint64_t o, const Acc& acc) {
		if (out.nhet) out.nhet[o] = acc.nhet;
		if (out.nonmissing) out.nonmissing[o] = acc.nonmissing;
		// (one non-missing site -- every window of the tools' default W = S = 1 -- divides by 1: the ~40-instruction IEEE
		// division is skipped, the value is the same)
		if (out.het)
			out.het[o] = acc.nonmissing > 1u ? __ddiv_rn((double)acc.nhet, (double)acc.nonmissing) : (acc.nonmissing ? (double)acc.nhet : 0.0);
	}
};

// --- dxyWindow: per-site dxy (dxyWindow.cpp:381) with explicit non-fused IEEE ops so the value is
// bit-identical to the x86-64 reference (no FMA there); window fold dxyWindow.cpp:179-186:
// v >= 0 -> dxy += v, ++neffective; v == -9 -> ++nskip.
__device__ __forceinline__ double dxy_site_value(double f1, double f2, int n1, int n2, int minind) {
	return (n1 >= minind && n2 >= minind) ? __dadd_rn(__dmul_rn(f1, __dsub_rn(1.0, f2)), __dmul_rn(f2, __dsub_rn(1.0, f1))) : -9.0;
}
struct DxyStat {
	typedef pgt_windows Out;
	struct Acc {
		double dxy;
		uint32_t neff, nskip;
	};
	struct Site {
		double f1, f2;
		int n1, n2;
	};
	static __device__ __forceinline__ Acc zero() { return Acc{0.0, 0u, 0u}; }
	static __device__ __forceinline__ Site load(const Cols& c, uint64_t i) {
		return Site{__ldg(c.f1 + i), __ldg(c.f2 + i), __ldg(c.n1 + i), __ldg(c.n2 + i)};
	}
	static __device__ __forceinline__ Site load_tile(const char* const* cp, uint32_t i) {
		return Site{((const double*)cp[0])[i], ((const double*)cp[1])[i], ((const int32_t*)cp[2])[i], ((const int32_t*)cp[3])[i]};
	}
	static __device__ __forceinline__ void fold(Acc& acc, const Site& s, int minind, double, uint64_t) {
		const double v = dxy_site_value(s.f1, s.f2, s.n1, s.n2, minind);
		if (v >= 0.0) {
			acc.dxy = __dadd_rn(acc.dxy, v);
			++acc.neff;
		} else if (v == -9.0) {
			++acc.nskip;
		}
	}
	static __device__ __forceinline__ void add(Acc& acc, const Acc& o) {
		acc.dxy = __dadd_rn(acc.dxy, o.dxy);
		acc.neff += o.neff;
		acc.nskip += o.nskip;
	}
	static __device__ __forceinline__ Acc shfl_xor(const Acc& v, int m) {
		return Acc{shfl_xor_f64(v.dxy, m), shfl_xor_u32(v.neff, m), shfl_xor_u32(v.nskip, m)};
	}
	static __device__ __forceinline__ void emit(const pgt_windows& out, uint64_t o, const Acc& acc) {
		if (out.dxy) out.dxy[o] = acc.dxy;
		if (out.neffective) out.neffective[o] = acc.neff;
		if (out.nskip) out.nskip[o] = acc.nskip;
	}
};

// --- fused fst + dxy + het over one site axis (BASELINE config 5): one pass, 41 B/site
struct FusedStat {
	typedef pgt_windows Out;
	struct Acc {
		FstStat::Acc fst;
		DxyStat::Acc dxy;
		HetStat::Acc het;
	};
	struct Site {
		FstStat::Site fst;
		DxyStat::Site dxy;
		HetStat::Site het;
	};
	static __device__ __forceinline__ Acc zero() { return Acc{FstStat::zero(), DxyStat::zero(), HetStat::zero()}; }
	static __device__ __forceinline__ Site load(const Cols& c, uint64_t i) { return Site{FstStat::load(c, i), DxyStat::load(c, i), HetStat::load(c, i)}; }
	// staging order: a, b, f1, f2, n1, n2, geno
	static __device__ __forceinline__ Site load_tile(const char* const* cp, uint32_t i) {
		return Site{FstStat::load_tile(cp, i), DxyStat::load_tile(cp + 2, i), HetStat::load_tile(cp + 6, i)};
	}
	static __device__ __forceinline__ void fold(Acc& acc, const Site& s, int minind, double, uint64_t) {
		FstStat::fold(acc.fst, s.fst, minind, 0.0, 0);
		DxyStat::fold(acc.dxy, s.dxy, minind, 0.0, 0);
		HetStat::fold(acc.het, s.het, minind, 0.0, 0);
	}
	static __device__ __forceinline__ void add(Acc& acc, const Acc& o) {
		FstStat::add(acc.fst, o.fst);
		DxyStat::add(acc.dxy, o.dxy);
		HetStat::add(acc.het, o.het);
	}
	static __device__ __forceinline__ Acc shfl_xor(const Acc& v, int m) {
		return Acc{FstStat::shfl_xor(v.fst, m), DxyStat::shfl_xor(v.dxy, m), HetStat::shfl_xor(v.het, m)};
	}
	static __device__ __forceinline__ void emit(const pgt_windows& out, uint64_t o, const Acc& acc) {
		FstStat::emit(out, o, acc.fst);
		DxyStat::emit(out, o, acc.dxy);
		HetStat::emit(out, o, acc.het);
	}
};

// --- fst + het together: what one of the two crews of the fused sliding tile computes (pgt_slide.cuh); every
// component is folded, combined and emitted exactly as by FstStat / HetStat alone.  Staged columns as FusedStat.
struct FstHetStat {
	typedef pgt_windows Out;
	struct Acc {
		FstStat::Acc fst;
		HetStat::Acc het;
	};
	struct Site {
		FstStat::Site fst;
		HetStat::Site het;
	};
	static __device__ __forceinline__ Acc zero() { return Acc{FstStat::zero(), HetStat::zero()}; }
	static __device__ __forceinline__ Site load_tile(const char* const* cp, uint32_t i) {
		return Site{FstStat::load_tile(cp, i), HetStat::load_tile(cp + 6, i)};
	}
	static __device__ __forceinline__ void fold(Acc& acc, const Site& s, int minind, double, uint64_t) {
		FstStat::fold(acc.fst, s.fst, minind, 0.0, 0);
		HetStat::fold(acc.het, s.het, minind, 0.0, 0);
	}
	static __device__ __forceinline__ void add(Acc& acc, const Acc& o) {
		FstStat::add(acc.fst, o.fst);
		HetStat::add(acc.het, o.het);
	}
	static __device__ __forceinline__ void emit(const pgt_windows& out, uint64_t o, const Acc& acc) {
		FstStat::emit(out, o, acc.fst);
		HetStat::emit(out, o, acc.het);
	}
};

// --- most extreme score over a window plan (pgt_scan_plan_extreme, ihsWindow / xpehhWindow statistics): the first
// site of largest key (|v|, v or -v; a NaN key is -inf), sites past the cutoff, sites.  The accumulator is a total
// order on (key, -site) plus two counts, so every butterfly, tree, scan and shard order gives the same bits.
enum { XMODE_ABS = 0, XMODE_MAX = 1, XMODE_MIN = 2 };

// Rows of an extreme scan: the geometry columns of pgt_windows (same meanings), the pgt_xwindows columns
// (xnsites = its nsites: score sites), and where ext_value / ext_pos are gathered from (score / pos[ext_site -
// site_origin]).
struct XRows {
	uint32_t *label, *start_pos, *end_pos, *mid_pos, *nsites;
	double* ext_value;
	uint32_t* ext_pos;
	uint64_t* ext_site;
	uint32_t *nbig, *xnsites;
	double* prop;
	const double* score;
	const uint32_t* pos;
	uint64_t site_origin;
};

template <int MODE>
struct XStat {
	typedef XRows Out;
	// The key of the extreme site rides in the partial, not its score: a lane's fold is then one compare and two
	// selects on registers (the score is gathered once per window in the epilogue, as its position).
	struct Acc {
		double key;
		uint64_t site;
		uint32_t nbig, n;
	};
	struct Site {
		double v;
	};
	static __device__ __forceinline__ double key(double v) {
		const double k = MODE == XMODE_ABS ? fabs(v) : (MODE == XMODE_MAX ? v : -v);
		return k != k ? -CUDART_INF : k;
	}
	// identity: key -inf ties with any real site's key at worst, and then the smaller index wins
	static __device__ __forceinline__ Acc zero() { return Acc{-CUDART_INF, ~0ull, 0u, 0u}; }
	static __device__ __forceinline__ Site load(const Cols& c, uint64_t i) { return Site{__ldg(c.score + i)}; }
	static __device__ __forceinline__ Site load_tile(const char* const* cp, uint32_t i) { return Site{((const double*)cp[0])[i]}; }
	// beyond the cutoff (strict; NaN never is)
	static __device__ __forceinline__ bool big(double v, double cutoff) {
		return MODE == XMODE_ABS ? fabs(v) > cutoff : (MODE == XMODE_MAX ? v > cutoff : v < cutoff);
	}
	static __device__ __forceinline__ void fold(Acc& acc, const Site& s, int, double cutoff, uint64_t site) {
		const double k = key(s.v);
		if (k > acc.key || (k == acc.key && site < acc.site)) {
			acc.key = k;
			acc.site = site;
		}
		acc.nbig += big(s.v, cutoff) ? 1u : 0u;
		++acc.n;
	}
	static __device__ __forceinline__ void add(Acc& acc, const Acc& o) {
		if (o.key > acc.key || (o.key == acc.key && o.site < acc.site)) {
			acc.key = o.key;
			acc.site = o.site;
		}
		acc.nbig += o.nbig;
		acc.n += o.n;
	}
	static __device__ __forceinline__ Acc shfl_xor(const Acc& v, int m) {
		return Acc{shfl_xor_f64(v.key, m), (uint64_t)__shfl_xor_sync(0xffffffffu, (unsigned long long)v.site, m), shfl_xor_u32(v.nbig, m),
		           shfl_xor_u32(v.n, m)};
	}
	static __device__ __forceinline__ void emit(const XRows& out, uint64_t o, const Acc& acc) {
		if (out.ext_value) out.ext_value[o] = acc.n ? __ldg(out.score + (acc.site - out.site_origin)) : CUDART_NAN;
		if (out.ext_site) out.ext_site[o] = acc.site;
		if (out.ext_pos) out.ext_pos[o] = acc.n ? __ldg(out.pos + (acc.site - out.site_origin)) : 0u;
		if (out.nbig) out.nbig[o] = acc.nbig;
		if (out.xnsites) out.xnsites[o] = acc.n;
		if (out.prop) out.prop[o] = acc.n ? __ddiv_rn((double)acc.nbig, (double)acc.n) : CUDART_NAN;
	}
};
template <class Stat>
struct IsXStat : std::false_type {};
template <int MODE>
struct IsXStat<XStat<MODE>> : std::true_type {};

template <class Stat>
__device__ __forceinline__ typename Stat::Acc warp_butterfly(typename Stat::Acc acc) {
#pragma unroll
	for (int m = 16; m >= 1; m >>= 1) Stat::add(acc, Stat::shfl_xor(acc, m));
	return acc;
}
// butterfly inside aligned groups of G lanes
template <class Stat, int G>
__device__ __forceinline__ typename Stat::Acc group_butterfly(typename Stat::Acc acc) {
#pragma unroll
	for (int m = G / 2; m >= 1; m >>= 1) Stat::add(acc, Stat::shfl_xor(acc, m));
	return acc;
}

#endif  // PGT_KERNELS_COMMON_CUH
