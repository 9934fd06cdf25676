// pgt_extreme.cu -- bp-window "most extreme score" scans (ihsWindow / xpehhWindow hot path):
// host window bookkeeping + sm_100a kernels + C ABI (include/pgt_extreme.h).
//
// The reference walks the file once, keeping (winstart, winend, nsites, nbig, best) and printing
// a row at every flush (/root/reference/ihsWindow.cpp:93-187, xpehhWindow.cpp:87-193).  Here:
//
//   pgt_xplan_create  : the flush bookkeeping alone -- integer compares on the position column,
//                       one independent state machine per chromosome run (threads across runs).
//                       Result: windows = contiguous site ranges (CSR `xoff`), possibly empty,
//                       each cut every U sites from its start into reduction *units*.
//   k_xunits<MODE,G>  : level 1.  The site axis is dealt to groups of G lanes in equal chunks; a
//                       group reduces every unit that STARTS in its chunk: lane-strided 8-byte
//                       streaming loads (8 in flight per lane), per-site key (|v|, v or -v) and
//                       cutoff test in registers, then a G-lane shuffle butterfly on
//                       (key, site index) -- larger key wins, equal keys keep the smaller index,
//                       which is exactly "the first extreme wins" of the reference's strict
//                       comparisons (ihsWindow.cpp:166) and makes the reduction order-free, so any
//                       G / U / sharding gives identical results.  A window that is a single unit
//                       is finished right here (epilogue fused); longer windows leave a 16-byte
//                       partial per unit.
//   k_xwindows<MODE>  : level 2.  Thread per window: writes the "NA" defaults of empty windows,
//                       combines the partials of multi-unit windows (windows of more than 32
//                       units are combined by the whole warp).
//
// Every score is read from HBM once (8 B/site); positions are touched only at the extreme site.
// No CPU fallback: without a CUDA device pgt_scan_extreme fails with PGT_ERR_CUDA.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <limits>
#include <new>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/pgt_synth.h"
#include "pgt_cuda.h"

static const uint32_t kDefaultUnit = 2048;

// pgt_tune("xgroup", G): force the lanes-per-unit of the extreme scan's level 1 (0 = auto; 4, 8, 16, 32)
int g_tune_xgroup = 0;
int g_tune_xsmall = 0;  // 0 auto, 1 never the small-window kernel (k_xsmall), 2 whenever the longest window allows it

// ----------------------------------------------------------------------------- host plan

struct pgt_xplan {
	uint32_t W = 0, U = 0;
	uint64_t nsites = 0, nwin = 0, nunits = 0;
	uint64_t max_window_sites = 0;            // longest window (chooses the small-window kernel)
	std::vector<uint32_t> label, start, end;  // per window
	std::vector<uint64_t> xoff;               // nwin+1: window w holds sites [xoff[w], xoff[w+1])
	std::vector<uint64_t> unit0;              // nwin+1: first unit of window w
	unsigned char* d_tables = nullptr;        // caller-owned device copy of xoff | unit0 (pgt_xplan_bind_device)
};

namespace {

struct RunRows {
	std::vector<uint32_t> start, end;
	std::vector<uint64_t> first;
	int err = 0;
	uint64_t err_site = 0;
};

// One chromosome run [lo, hi) of the position column through the reference's window bookkeeping.
// ihsWindow.cpp:98-99 (initial window, not clipped), :130-144 (chromosome change: flush, pad to
// chrlen, reset + clip), :145-157 (flush when pos >= winend, empty windows while pos > winend),
// :179-186 (last window + padding).  uint32 arithmetic as in the reference.
void run_windows(const uint32_t* pos, uint64_t lo, uint64_t hi, bool first_run, uint32_t L, uint32_t W, RunRows* out) {
	uint32_t ws = 1;
	uint32_t we = ws + (W - 1);
	if (!first_run && L && we > L) we = L;
	uint64_t wfirst = lo;
	uint64_t n = 0;
	auto emit = [&](uint64_t first) {
		out->start.push_back(ws);
		out->end.push_back(we);
		out->first.push_back(first);
	};
	auto advance = [&]() {
		ws = we + 1;
		we = ws + (W - 1);
		if (L && we > L) we = L;
	};
	for (uint64_t i = lo; i < hi; ++i) {
		const uint32_t p = pos[i];
		if ((i != lo || first_run) && p >= we) {  // the first site of a later run is never tested (:130 vs :145)
			emit(wfirst);
			advance();
			n = 0;
			while (p > we) {
				if (L && we >= L) {  // winend is pinned at chrlen: the reference never leaves this loop
					out->err = 1;
					out->err_site = i;
					return;
				}
				emit(i);
				advance();
			}
		}
		if (n == 0) wfirst = i;
		++n;
	}
	emit(wfirst);
	while (we < L) {
		advance();
		emit(hi);
	}
}

}  // namespace

extern "C" int pgt_xplan_create(pgt_xplan** out, const uint32_t* pos, const uint64_t* contig_offsets, const uint32_t* contig_len,
                                uint32_t ncontig, uint32_t winsize, uint32_t unit_sites) {
	if (!out) return pgt_set_error(PGT_ERR_ARGS, "pgt_xplan_create: plan pointer is NULL");
	*out = nullptr;
	if (winsize < 1) return pgt_set_error(PGT_ERR_ARGS, "Window size must be a positive integer");
	if (!contig_offsets || ncontig == 0) return pgt_set_error(PGT_ERR_ARGS, "pgt_xplan_create: no contigs");
	for (uint32_t c = 0; c < ncontig; ++c)
		if (contig_offsets[c + 1] <= contig_offsets[c] || contig_offsets[0] != 0)
			return pgt_set_error(PGT_ERR_ARGS, "pgt_xplan_create: contig_offsets must start at 0 and increase strictly");
	const uint64_t n = contig_offsets[ncontig];
	if (!pos) return pgt_set_error(PGT_ERR_ARGS, "pgt_xplan_create: pos is NULL (host position column required)");
	pgt_xplan* P = new (std::nothrow) pgt_xplan;
	if (!P) return pgt_set_error(PGT_ERR_NOMEM, "pgt_xplan_create: out of memory");
	P->W = winsize;
	P->U = unit_sites ? unit_sites : kDefaultUnit;
	P->nsites = n;
	try {
		std::vector<RunRows> rows(ncontig);
		unsigned nt = n > (1u << 20) ? std::min<unsigned>(std::min<unsigned>(std::thread::hardware_concurrency(), 32u), ncontig) : 1;
		if (nt < 1) nt = 1;
		std::atomic<uint32_t> next{0};
		auto work = [&]() {
			for (;;) {
				const uint32_t c = next.fetch_add(1);
				if (c >= ncontig) break;
				try {
					run_windows(pos, contig_offsets[c], contig_offsets[c + 1], c == 0, contig_len ? contig_len[c] : 0u, winsize, &rows[c]);
				} catch (const std::bad_alloc&) {  // e.g. -winsize 1 over gigabase gaps: rows do not fit
					rows[c].err = 2;
				}
			}
		};
		if (nt == 1) work();
		else {
			std::vector<std::thread> th;
			for (unsigned t = 0; t < nt; ++t) th.emplace_back(work);
			for (auto& x : th) x.join();
		}
		uint64_t nwin = 0;
		for (uint32_t c = 0; c < ncontig; ++c) {
			if (rows[c].err == 2) {
				delete P;
				return pgt_set_error(PGT_ERR_NOMEM, "pgt_xplan_create: out of memory for the window table");
			}
			if (rows[c].err) {
				const uint64_t i = rows[c].err_site;
				delete P;
				return pgt_set_error(PGT_ERR_INPUT, "site " + std::to_string(i) + " (position " + std::to_string(pos[i]) +
				                                        ") lies beyond its chromosome length " + std::to_string(contig_len[c]));
			}
			nwin += rows[c].start.size();
		}
		P->nwin = nwin;
		P->label.reserve(nwin);
		P->start.reserve(nwin);
		P->end.reserve(nwin);
		P->xoff.reserve(nwin + 1);
		for (uint32_t c = 0; c < ncontig; ++c) {
			P->label.insert(P->label.end(), rows[c].start.size(), c);
			P->start.insert(P->start.end(), rows[c].start.begin(), rows[c].start.end());
			P->end.insert(P->end.end(), rows[c].end.begin(), rows[c].end.end());
			P->xoff.insert(P->xoff.end(), rows[c].first.begin(), rows[c].first.end());
			RunRows().start.swap(rows[c].start);
			RunRows().end.swap(rows[c].end);
			RunRows().first.swap(rows[c].first);
		}
		P->xoff.push_back(n);
		P->unit0.resize(nwin + 1);
		uint64_t u = 0;
		for (uint64_t w = 0; w < nwin; ++w) {
			P->unit0[w] = u;
			u += (P->xoff[w + 1] - P->xoff[w] + P->U - 1) / P->U;
			P->max_window_sites = std::max(P->max_window_sites, P->xoff[w + 1] - P->xoff[w]);
		}
		P->unit0[nwin] = u;
		P->nunits = u;
	} catch (const std::bad_alloc&) {
		delete P;
		return pgt_set_error(PGT_ERR_NOMEM, "pgt_xplan_create: out of memory for the window table");
	}
	*out = P;
	return PGT_OK;
}

extern "C" void pgt_xplan_destroy(pgt_xplan* plan) { delete plan; }
extern "C" uint64_t pgt_xplan_num_windows(const pgt_xplan* plan) { return plan ? plan->nwin : 0; }
extern "C" uint64_t pgt_xplan_num_units(const pgt_xplan* plan) { return plan ? plan->nunits : 0; }
extern "C" uint64_t pgt_xplan_num_sites(const pgt_xplan* plan) { return plan ? plan->nsites : 0; }

extern "C" int pgt_xplan_windows(const pgt_xplan* plan, uint32_t* label, uint32_t* start, uint32_t* end, uint64_t* first_site,
                                 uint32_t* nsites) {
	if (!plan) return pgt_set_error(PGT_ERR_ARGS, "pgt_xplan_windows: plan is NULL");
	const uint64_t n = plan->nwin;
	if (label) memcpy(label, plan->label.data(), n * sizeof(uint32_t));
	if (start) memcpy(start, plan->start.data(), n * sizeof(uint32_t));
	if (end) memcpy(end, plan->end.data(), n * sizeof(uint32_t));
	if (first_site) memcpy(first_site, plan->xoff.data(), n * sizeof(uint64_t));
	if (nsites)
		for (uint64_t w = 0; w < n; ++w) nsites[w] = (uint32_t)(plan->xoff[w + 1] - plan->xoff[w]);
	return PGT_OK;
}

extern "C" int pgt_xplan_shard(const pgt_xplan* plan, uint32_t shard, uint32_t nshards, uint64_t* w_lo, uint64_t* w_hi,
                               uint64_t* site_lo, uint64_t* site_hi) {
	if (!plan) return pgt_set_error(PGT_ERR_ARGS, "pgt_xplan_shard: plan is NULL");
	if (nshards == 0 || shard >= nshards) return pgt_set_error(PGT_ERR_ARGS, "pgt_xplan_shard: shard out of range");
	// cut r = first window whose first site is >= r * nsites / nshards (windows never split)
	auto cut = [&](uint32_t r) -> uint64_t {
		if (r == 0) return 0;
		if (r >= nshards) return plan->nwin;
		const uint64_t target = (uint64_t)((unsigned __int128)plan->nsites * r / nshards);
		return (uint64_t)(std::lower_bound(plan->xoff.begin(), plan->xoff.begin() + plan->nwin, target) - plan->xoff.begin());
	};
	const uint64_t lo = cut(shard), hi = cut(shard + 1);
	if (w_lo) *w_lo = lo;
	if (w_hi) *w_hi = hi;
	if (site_lo) *site_lo = plan->xoff[lo];
	if (site_hi) *site_hi = plan->xoff[hi];
	return PGT_OK;
}

// ----------------------------------------------------------------------------- device side

enum { XMODE_ABS = 0, XMODE_MAX = 1, XMODE_MIN = 2 };

// unit partials, SoA (20 B per unit): signed score and global site index of the unit's first
// extreme, sites beyond the cutoff
struct XPartials {
	double* val;
	uint64_t* idx;
	uint32_t* nbig;
};

struct XDev {
	const uint64_t* xoff;   // nw+1 entries for windows w_lo..w_hi: global site indices
	const uint64_t* unit0;  // nw+1 entries: global unit indices
	uint64_t unit_base;     // unit0[w_lo]: partials are indexed by unit - unit_base
	uint64_t nw;
	uint64_t site_lo, site_hi;  // sites of the range
	uint64_t origin;            // global index of element 0 of score / pos
	uint32_t U;
	double cutoff;
};

// key: larger = more extreme.  NaN never beats anything (x > NaN and NaN > x are false in the
// reference's comparisons); the one case where the reference keeps a NaN -- it is the first site
// of the window (updateMax on nsites == 0, ihsWindow.cpp:161-164) -- is handled explicitly.
template <int MODE>
__device__ __forceinline__ double x_key(double v) {
	double k = MODE == XMODE_ABS ? fabs(v) : (MODE == XMODE_MAX ? v : -v);
	return k != k ? -CUDART_INF : k;
}
template <int MODE>
__device__ __forceinline__ bool x_big(double v, double cutoff) {
	return MODE == XMODE_ABS ? fabs(v) > cutoff : (MODE == XMODE_MAX ? v > cutoff : v < cutoff);
}

struct XAcc {
	double key;
	double val;
	uint64_t idx;
	uint32_t nbig;
};
// (key, idx) lexicographic: larger key wins, equal keys keep the smaller site index = the first
// extreme in file order, whatever the evaluation order
__device__ __forceinline__ void x_take(XAcc& a, double k, double v, uint64_t i) {
	if (k > a.key || (k == a.key && i < a.idx)) {
		a.key = k;
		a.val = v;
		a.idx = i;
	}
}

// last window w in [0, nw) with xoff[w] <= s
__device__ __forceinline__ uint64_t x_window_of(const XDev& P, uint64_t s) {
	uint64_t lo = 0, hi = P.nw;
	while (hi - lo > 1) {
		const uint64_t mid = lo + ((hi - lo) >> 1);
		if (P.xoff[mid] <= s) lo = mid;
		else hi = mid;
	}
	return lo;
}

// Level 1: pure streaming.  Window bounds and unit indices are fetched one window ahead, the only
// store per unit takes its data from registers, so a group's next unit never waits on anything
// but its own score loads.
template <int MODE, int G>
__global__ void __launch_bounds__(256) k_xunits(XDev P, uint64_t chunk, const double* __restrict__ score, XPartials part) {
	const uint32_t lane = threadIdx.x & 31u;
	const uint32_t gl = lane & (G - 1);  // lane inside the group
	const uint32_t gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(uint32_t)(G - 1)));
	const uint64_t group = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
	const uint64_t c_lo = P.site_lo + group * chunk;
	if (c_lo >= P.site_hi) return;
	const uint64_t c_hi = c_lo + chunk < P.site_hi ? c_lo + chunk : P.site_hi;
	uint64_t w = x_window_of(P, c_lo);
	uint64_t w_st = P.xoff[w];
	uint64_t w_end = P.xoff[w + 1];
	uint64_t w_end2 = P.xoff[w + 2 <= P.nw ? w + 2 : P.nw];  // one window ahead
	uint64_t u0 = P.unit0[w], u0n = P.unit0[w + 1];
	uint64_t st = w_st + (c_lo - w_st + P.U - 1) / P.U * P.U;  // first unit starting at or after c_lo
	for (;;) {
		while (st >= w_end) {  // next non-empty window
			++w;
			if (w >= P.nw) return;
			w_st = w_end;
			w_end = w_end2;
			u0 = u0n;
			w_end2 = P.xoff[w + 2 <= P.nw ? w + 2 : P.nw];
			u0n = P.unit0[w + 1];
			st = w_st;
		}
		if (st >= c_hi) return;
		const uint32_t len = (uint32_t)(w_end - st < P.U ? w_end - st : P.U);
		XAcc a{-CUDART_INF, 0.0, ~0ull, 0u};
		const double* __restrict__ p = score + (st - P.origin);  // element 0 of `score` is global site P.origin
		bool first_nan = false;  // lane gl == 0 sees the window's first site when st == w_st
		uint32_t x = gl;
		for (; x + 7u * G < len; x += 8u * G) {  // full rounds: 8 loads in flight per lane
			double v[8];
#pragma unroll
			for (int q = 0; q < 8; ++q) v[q] = __ldcs(p + x + q * G);
			if (x == 0) first_nan = v[0] != v[0];
#pragma unroll
			for (int q = 0; q < 8; ++q) {
				x_take(a, x_key<MODE>(v[q]), v[q], st + x + q * G);
				a.nbig += x_big<MODE>(v[q], P.cutoff) ? 1u : 0u;
			}
		}
		if (x < len) {  // ragged last round, predicated: still all of its loads in flight at once
			double v[7];
#pragma unroll
			for (int q = 0; q < 7; ++q) v[q] = x + q * G < len ? __ldcs(p + x + q * G) : CUDART_NAN;
			if (x == 0) first_nan = v[0] != v[0];
#pragma unroll
			for (int q = 0; q < 7; ++q) {
				if (x + q * G < len) {
					x_take(a, x_key<MODE>(v[q]), v[q], st + x + q * G);
					a.nbig += x_big<MODE>(v[q], P.cutoff) ? 1u : 0u;
				}
			}
		}
#pragma unroll
		for (int m = G >> 1; m > 0; m >>= 1) {
			const double ko = __shfl_xor_sync(gmask, a.key, m);
			const double vo = __shfl_xor_sync(gmask, a.val, m);
			const uint64_t io = __shfl_xor_sync(gmask, a.idx, m);
			a.nbig += __shfl_xor_sync(gmask, a.nbig, m);
			x_take(a, ko, vo, io);
		}
		if (gl == 0) {
			if (st == w_st && first_nan) {  // a NaN on the window's first site stays the extreme
				a.val = p[0];
				a.idx = st;
			}
			const uint64_t j = u0 + (st - w_st) / P.U - P.unit_base;
			part.val[j] = a.val;
			part.idx[j] = a.idx;
			part.nbig[j] = a.nbig;
		}
		st += len;
	}
}

__device__ __forceinline__ void x_emit(uint64_t w, double val, uint64_t best, uint32_t nbig, uint64_t n, uint64_t origin,
                                       const uint32_t* __restrict__ pos, const pgt_xwindows& out) {
	if (out.ext_value) out.ext_value[w] = val;
	if (out.ext_pos) out.ext_pos[w] = pos ? pos[best - origin] : 0u;
	if (out.ext_site) out.ext_site[w] = best;
	if (out.nbig) out.nbig[w] = nbig;
	if (out.nsites) out.nsites[w] = (uint32_t)n;
	if (out.prop) out.prop[w] = (double)nbig / (double)(uint32_t)n;  // ihsWindow.cpp:79: double / unsigned
}

// the reference's "NA NA NA 0" row of an empty window (ihsWindow.cpp:82)
__device__ __forceinline__ void x_emit_empty(uint64_t w, const pgt_xwindows& out) {
	if (out.ext_value) out.ext_value[w] = CUDART_NAN;
	if (out.ext_pos) out.ext_pos[w] = 0u;
	if (out.ext_site) out.ext_site[w] = ~0ull;
	if (out.nbig) out.nbig[w] = 0u;
	if (out.nsites) out.nsites[w] = 0u;
	if (out.prop) out.prop[w] = CUDART_NAN;
}

// Level 2: thread per window.  Empty windows get the "NA" defaults, single-unit windows copy their
// partial, windows of 2..32 units are combined by their thread, longer ones by the whole warp.
template <int MODE>
__global__ void __launch_bounds__(256) k_xwindows(XDev P, const uint32_t* __restrict__ pos, XPartials part, pgt_xwindows out) {
	const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t lane = threadIdx.x & 31u;
	const bool valid = w < P.nw;
	uint64_t n = 0, u0 = 0, nu = 0, first = 0;
	if (valid) {
		first = P.xoff[w];
		n = P.xoff[w + 1] - first;
		u0 = P.unit0[w] - P.unit_base;
		nu = P.unit0[w + 1] - P.unit_base - u0;
	}
	if (valid && n == 0) {
		x_emit_empty(w, out);
	} else if (valid && nu <= 32) {
		const double v0 = part.val[u0];
		XAcc a{x_key<MODE>(v0), v0, part.idx[u0], part.nbig[u0]};
		if (!(v0 != v0 && a.idx == first)) {  // unless the first site is a NaN (it then stays)
			for (uint64_t j = 1; j < nu; ++j) {
				const double v = part.val[u0 + j];
				x_take(a, x_key<MODE>(v), v, part.idx[u0 + j]);
			}
		}
		for (uint64_t j = 1; j < nu; ++j) a.nbig += part.nbig[u0 + j];
		x_emit(w, a.val, a.idx, a.nbig, n, P.origin, pos, out);
	}
	uint32_t todo = __ballot_sync(0xffffffffu, valid && nu > 32);
	while (todo) {
		const int src = __ffs(todo) - 1;
		todo &= todo - 1;
		const uint64_t wb = __shfl_sync(0xffffffffu, w, src);
		const uint64_t ub = __shfl_sync(0xffffffffu, u0, src);
		const uint64_t nub = __shfl_sync(0xffffffffu, nu, src);
		const uint64_t nb = __shfl_sync(0xffffffffu, n, src);
		const uint64_t fb = __shfl_sync(0xffffffffu, first, src);
		XAcc a{-CUDART_INF, 0.0, ~0ull, 0u};
		for (uint64_t j = lane; j < nub; j += 32) {
			const double v = part.val[ub + j];
			x_take(a, x_key<MODE>(v), v, part.idx[ub + j]);
			a.nbig += part.nbig[ub + j];
		}
#pragma unroll
		for (int m = 16; m > 0; m >>= 1) {
			const double ko = __shfl_xor_sync(0xffffffffu, a.key, m);
			const double vo = __shfl_xor_sync(0xffffffffu, a.val, m);
			const uint64_t io = __shfl_xor_sync(0xffffffffu, a.idx, m);
			a.nbig += __shfl_xor_sync(0xffffffffu, a.nbig, m);
			x_take(a, ko, vo, io);
		}
		if (lane == 0) {
			const double v0 = part.val[ub];
			if (v0 != v0 && part.idx[ub] == fb) {
				a.val = v0;
				a.idx = fb;
			}
			x_emit(wb, a.val, a.idx, a.nbig, nb, P.origin, pos, out);
		}
	}
}

// Short windows (tens of sites: dense windows over sparse SNP sets): the two-level scheme pays a unit partial, a second
// read of the window table and a butterfly per 33-site window (r01: 3.3 ms per 1e9 sites at 33 sites per window).  Here a
// CTA stages a tile of consecutive sites in shared memory with coalesced loads -- batch t = the windows whose first site
// lies in [site_lo + t*kXTileStep, +kXTileStep), found by two binary searches in xoff; their sites span less than
// kXTileStep + kXMaxSmallWindow <= kXTileSites -- and ONE THREAD walks each window in file order: the reference's own
// loop (first site taken unconditionally, then strictly-greater comparisons, ihsWindow.cpp:159-173), so NaN handling
// needs no special case, and the finished row is written straight to the output columns (no partials, no level 2).
static constexpr uint32_t kXTileSites = 12288;        // 96 KB of scores per CTA: two CTAs per SM
static constexpr uint32_t kXMaxSmallWindow = 2048;    // plans whose longest window exceeds this keep the two-level scheme
static constexpr uint32_t kXTileStep = kXTileSites - kXMaxSmallWindow;

// first window w in [0, nw] with xoff[w] >= s (nw if none)
__device__ __forceinline__ uint64_t x_lower_window(const XDev& P, uint64_t s) {
	uint64_t lo = 0, hi = P.nw;
	while (lo < hi) {
		const uint64_t mid = lo + ((hi - lo) >> 1);
		if (P.xoff[mid] < s) lo = mid + 1;
		else hi = mid;
	}
	return lo;
}

// batch -> first window, one thread per batch (a binary search over millions of windows is ~25 dependent trips to L2 /
// HBM: done per tile inside k_xsmall it cost more than the tile itself).  bw[nbatches] = nw: the last batch also takes
// the windows that start at site_hi (trailing empty windows).
__global__ void __launch_bounds__(256) k_xbatches(XDev P, uint64_t nbatches, uint64_t* __restrict__ bw) {
	const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (t < nbatches) bw[t] = x_lower_window(P, P.site_lo + t * kXTileStep);
	else if (t == nbatches) bw[t] = P.nw;
}

template <int MODE>
__global__ void __launch_bounds__(256) k_xsmall(XDev P, uint64_t nbatches, const uint64_t* __restrict__ bw, const double* __restrict__ score,
                                                 const uint32_t* __restrict__ pos, pgt_xwindows out) {
	extern __shared__ __align__(16) double x_tile[];
	for (uint64_t t = blockIdx.x; t < nbatches; t += gridDim.x) {
		const uint64_t w_lo = bw[t], w_hi = bw[t + 1];
		if (w_hi > w_lo) {
			const uint64_t s_lo = P.xoff[w_lo], s_hi = P.xoff[w_hi];
			const uint32_t n = (uint32_t)(s_hi - s_lo);  // < kXTileStep + kXMaxSmallWindow
			const double* __restrict__ src = score + (s_lo - P.origin);
			// the whole tile in flight at once and at no register cost: 8-byte asynchronous copies straight into shared
			// memory (with register-staged loads, 16 KB in flight per CTA, the kernel ran at 1.6 TB/s)
			const uint32_t tile_addr = (uint32_t)__cvta_generic_to_shared(x_tile);
			for (uint32_t i = threadIdx.x; i < n; i += 256u)
				asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(tile_addr + i * 8u), "l"(src + i) : "memory");
			asm volatile("cp.async.wait_all;" ::: "memory");
			__syncthreads();
			for (uint64_t w = w_lo + threadIdx.x; w < w_hi; w += 256u) {
				const uint64_t a = P.xoff[w], b = P.xoff[w + 1];
				const uint32_t len = (uint32_t)(b - a);
				if (len == 0) {
					x_emit_empty(w, out);
					continue;
				}
				const double* __restrict__ p = x_tile + (a - s_lo);
				double best = p[0];
				double bkey = MODE == XMODE_ABS ? fabs(best) : (MODE == XMODE_MAX ? best : -best);  // NaN stays NaN: nothing beats it
				uint32_t bi = 0, nbig = x_big<MODE>(best, P.cutoff) ? 1u : 0u;
				for (uint32_t j = 1; j < len; ++j) {
					const double v = p[j];
					const double k = MODE == XMODE_ABS ? fabs(v) : (MODE == XMODE_MAX ? v : -v);
					if (k > bkey) {  // strictly greater: the first extreme stays on ties; false for NaN on either side
						bkey = k;
						best = v;
						bi = j;
					}
					nbig += x_big<MODE>(v, P.cutoff) ? 1u : 0u;
				}
				x_emit(w, best, a + bi, nbig, len, P.origin, pos, out);
			}
		}
		__syncthreads();  // the tile is reused by the next batch
	}
}

__global__ void k_synth_score(uint64_t seed, uint64_t site0, uint64_t n, double* __restrict__ score) {
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) score[i] = pgt_synth_score(seed, site0 + i);
}

extern "C" int pgt_synth_score(uint64_t seed, uint64_t site0, uint64_t n, double* score, void* stream) {
	if (n == 0) return PGT_OK;
	if (!score) return pgt_set_error(PGT_ERR_ARGS, "pgt_synth_score: NULL column");
	const uint64_t want = (n + 255) / 256;
	k_synth_score<<<(unsigned)std::min<uint64_t>(want, 148ull * 16ull), 256, 0, (cudaStream_t)stream>>>(seed, site0, n, score);
	pgt_count_launch();
	PGT_CUDA(cudaGetLastError());
	return PGT_OK;
}

// ----------------------------------------------------------------------------- host side of a scan

namespace {

struct XLayout {
	uint64_t w_lo = 0, w_hi = 0, nw = 0, site_lo = 0, site_hi = 0, nsite = 0, unit_lo = 0, nunit = 0;
	bool resident = false;  // window tables are bound on the device (pgt_xplan_bind_device)
	size_t off_xoff = 0, off_unit0 = 0, p_val = 0, p_idx = 0, p_nbig = 0, off_score = 0, off_outs = 0, total = 0;
};

int x_layout(const pgt_xplan* plan, const pgt_range* range, pgt_mem mem, XLayout* L) {
	if (!plan) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme: plan is NULL");
	uint64_t lo = 0, hi = plan->nwin;
	if (range && !(range->w_lo == 0 && range->w_hi == 0)) {
		lo = range->w_lo;
		hi = range->w_hi;
	}
	if (lo > hi || hi > plan->nwin) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme: window range out of bounds");
	L->w_lo = lo;
	L->w_hi = hi;
	L->nw = hi - lo;
	L->site_lo = plan->xoff[lo];
	L->site_hi = plan->xoff[hi];
	L->nsite = L->site_hi - L->site_lo;
	L->unit_lo = plan->unit0[lo];
	L->nunit = plan->unit0[hi] - plan->unit0[lo];
	L->resident = plan->d_tables != nullptr;
	size_t o = 0;
	if (!L->resident) {
		L->off_xoff = o;
		o += align_up((L->nw + 1) * sizeof(uint64_t), 256);
		L->off_unit0 = o;
		o += align_up((L->nw + 1) * sizeof(uint64_t), 256);
	}
	L->p_val = o;
	o += align_up(L->nunit * sizeof(double), 256);
	L->p_idx = o;
	o += align_up(L->nunit * sizeof(uint64_t), 256);
	L->p_nbig = o;
	o += align_up(L->nunit * sizeof(uint32_t), 256);
	if (mem == PGT_MEM_HOST) {
		L->off_score = o;
		o += align_up(L->nsite * sizeof(double), 256);
		// staged outputs: one block per field in for_each_xfield order, none for ext_pos (gathered on the host)
		L->off_outs = o;
		pgt_xwindows t{};
		for_each_xfield([&](auto*& p) { o += (void*)&p == (void*)&t.ext_pos ? 0 : align_up(L->nw * sizeof(*p), 256); }, t);
	}
	L->total = o + 256;
	return PGT_OK;
}

template <int MODE, int G>
void x_launch_units(const XDev& P, uint64_t nsite, const double* score, const XPartials& part, cudaStream_t st) {
	// site axis dealt in equal chunks to groups of G lanes: at least 64 sites per lane, at most
	// one wave of resident CTAs (grid = multiple of the SM count)
	int per_sm = 0;
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_xunits<MODE, G>, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
	const uint64_t max_groups = (uint64_t)num_sms() * (uint64_t)per_sm * 256ull / G;
	uint64_t chunk = (nsite + max_groups - 1) / max_groups;
	const uint64_t min_chunk = 64ull * G;
	if (chunk < min_chunk) chunk = min_chunk;
	const uint64_t groups = (nsite + chunk - 1) / chunk;
	const uint64_t threads = groups * G;
	const unsigned grid = (unsigned)((threads + 255) / 256);
	k_xunits<MODE, G><<<grid, 256, 0, st>>>(P, chunk, score, part);
	pgt_count_launch();
}

template <int MODE>
int x_run(const XDev& P, uint64_t nsite, uint64_t nunit, const double* score, const uint32_t* pos, const XPartials& part,
          const pgt_xwindows& out, bool small, cudaStream_t st) {
	if (small && P.nw) {
		// short windows: tile of sites in shared memory, a thread per window, rows written directly (k_xsmall)
		const uint64_t nbatches = (P.site_hi - P.site_lo) / kXTileStep + 1;
		const size_t smem = (size_t)kXTileSites * sizeof(double);
		PGT_CUDA(cudaFuncSetAttribute(k_xsmall<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		ProfScope prof(2, st);
		uint64_t* bw = part.idx;  // the partials are not used on this path: >= nw entries, and nw >= nbatches + 1 (checked by the caller)
		k_xbatches<<<(unsigned)((nbatches + 256) / 256), 256, 0, st>>>(P, nbatches, bw);
		pgt_count_launch();
		k_xsmall<MODE><<<one_wave_grid(k_xsmall<MODE>, 256, nbatches, smem), 256, smem, st>>>(P, nbatches, bw, score, pos, out);
		pgt_count_launch();
		PGT_CUDA(cudaGetLastError());
		return PGT_OK;
	}
	if (nsite) {
		ProfScope prof(2, st);
		// lanes per unit from the mean unit length: short windows get narrow groups, so that every
		// lane still streams several rounds of 8 loads per unit
		const uint64_t mean = nunit ? nsite / nunit : 0;
		// measured on B200 (profiles/r01c_extreme_xgroup_sweep.txt): best at ~32-64 sites per lane
		int g = mean >= 1024 ? 32 : (mean >= 512 ? 16 : (mean >= 160 ? 8 : 4));
		if (g_tune_xgroup >= 4) g = g_tune_xgroup;
		switch (g) {
			case 32: x_launch_units<MODE, 32>(P, nsite, score, part, st); break;
			case 16: x_launch_units<MODE, 16>(P, nsite, score, part, st); break;
			case 8: x_launch_units<MODE, 8>(P, nsite, score, part, st); break;
			default: x_launch_units<MODE, 4>(P, nsite, score, part, st); break;
		}
		PGT_CUDA(cudaGetLastError());
	}
	if (P.nw) {
		ProfScope prof(3, st);
		k_xwindows<MODE><<<(unsigned)((P.nw + 255) / 256), 256, 0, st>>>(P, pos, part, out);
		pgt_count_launch();
		PGT_CUDA(cudaGetLastError());
	}
	return PGT_OK;
}

}  // namespace

extern "C" size_t pgt_xplan_device_bytes(const pgt_xplan* plan) {
	return plan ? table_pair_bytes((plan->nwin + 1) * sizeof(uint64_t), (plan->nwin + 1) * sizeof(uint64_t)) : 0;
}

extern "C" int pgt_xplan_bind_device(pgt_xplan* plan, void* buffer, size_t bytes, void* stream) {
	if (!plan) return pgt_set_error(PGT_ERR_ARGS, "pgt_xplan_bind_device: plan is NULL");
	if (!buffer) {
		plan->d_tables = nullptr;
		return PGT_OK;
	}
	if (bytes < pgt_xplan_device_bytes(plan)) return pgt_set_error(PGT_ERR_NOMEM, "pgt_xplan_bind_device: buffer too small");
	const size_t tb = (plan->nwin + 1) * sizeof(uint64_t);
	return bind_table_pair(buffer, plan->xoff.data(), tb, plan->unit0.data(), tb, stream, &plan->d_tables);
}

extern "C" size_t pgt_scan_extreme_workspace_bytes(const pgt_xplan* plan, const pgt_range* range, pgt_mem mem) {
	XLayout L;
	if (x_layout(plan, range, mem, &L) != PGT_OK) return 0;
	return L.total;
}

extern "C" int pgt_scan_extreme(const pgt_xplan* plan, const pgt_range* range, pgt_xstat stat, double cutoff, const uint32_t* pos,
                                const double* score, const pgt_xwindows* out, void* workspace, size_t workspace_bytes, pgt_mem mem,
                                void* stream) {
	if (stat != PGT_XSTAT_IHS && stat != PGT_XSTAT_XPEHH) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme: unknown statistic");
	if (mem != PGT_MEM_DEVICE && mem != PGT_MEM_HOST) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme: unknown memory kind");
	if (!out) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme: out is NULL");
	XLayout L;
	int rc = x_layout(plan, range, mem, &L);
	if (rc != PGT_OK) return rc;
	if (L.nw == 0) return PGT_OK;
	if (!score && L.nsite) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme: score column is NULL");
	if (out->ext_pos && !pos) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme: ext_pos requested but pos is NULL");
	if (!workspace || workspace_bytes < L.total) return pgt_set_error(PGT_ERR_NOMEM, "pgt_scan_extreme: workspace too small");
	const uint64_t origin = range ? range->site_origin : 0;
	if (origin > L.site_lo) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme: site_origin lies after the first site of the window range");
	int ndev = 0;
	{
		cudaError_t e = cudaGetDeviceCount(&ndev);
		if (e != cudaSuccess || ndev == 0) return cuda_fail(e != cudaSuccess ? e : cudaErrorNoDevice, "pgt_scan_extreme: no usable CUDA device");
	}
	cudaStream_t st = (cudaStream_t)stream;
	unsigned char* ws = (unsigned char*)(((uintptr_t)workspace + 255) / 256 * 256);

	XDev P;
	if (L.resident) {  // tables bound once with pgt_xplan_bind_device: nothing to upload
		const uint64_t* t = (const uint64_t*)plan->d_tables;
		P.xoff = t + L.w_lo;
		P.unit0 = (const uint64_t*)(plan->d_tables + align_up((plan->nwin + 1) * sizeof(uint64_t), 256)) + L.w_lo;
	} else {
		uint64_t* d_xoff = (uint64_t*)(ws + L.off_xoff);
		uint64_t* d_unit0 = (uint64_t*)(ws + L.off_unit0);
		PGT_CUDA(cudaMemcpyAsync(d_xoff, plan->xoff.data() + L.w_lo, (L.nw + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
		PGT_CUDA(cudaMemcpyAsync(d_unit0, plan->unit0.data() + L.w_lo, (L.nw + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
		P.xoff = d_xoff;
		P.unit0 = d_unit0;
	}
	P.unit_base = L.unit_lo;
	P.nw = L.nw;
	P.site_lo = L.site_lo;
	P.site_hi = L.site_hi;
	P.U = plan->U;
	P.cutoff = cutoff;
	XPartials part{(double*)(ws + L.p_val), (uint64_t*)(ws + L.p_idx), (uint32_t*)(ws + L.p_nbig)};
	const int mode = stat == PGT_XSTAT_IHS ? XMODE_ABS : (cutoff < 0 ? XMODE_MIN : XMODE_MAX);  // xpehhWindow.cpp:171

	pgt_xwindows dout;
	const double* d_score;
	const uint32_t* d_pos;
	if (mem == PGT_MEM_DEVICE) {
		P.origin = origin;
		d_score = score;
		d_pos = pos;
		dout = *out;
	} else {
		// host columns: stage the scores of the range; positions stay on the host (gathered there
		// from ext_site after the scan)
		P.origin = L.site_lo;
		double* stage = (double*)(ws + L.off_score);
		if (L.nsite) PGT_CUDA(cudaMemcpyAsync(stage, score + (L.site_lo - origin), L.nsite * sizeof(double), cudaMemcpyHostToDevice, st));
		d_score = stage;
		d_pos = nullptr;
		memset(&dout, 0, sizeof(dout));
		size_t o = L.off_outs;  // the blocks of x_layout; ext_site is staged for ext_pos too
		for_each_xfield(
		    [&](auto*& d, auto* h) {
			    if ((void*)&d == (void*)&dout.ext_pos) return;
			    if (h || ((void*)&d == (void*)&dout.ext_site && out->ext_pos)) d = (std::remove_reference_t<decltype(d)>)(ws + o);
			    o += align_up(L.nw * sizeof(*d), 256);
		    },
		    dout, *out);
	}
	// short windows (a function of the plan only: longest window <= 2048 sites, fewer than 160 sites per unit on average)
	// Measured (1e9 sites, profiles/r02z_extreme_small_windows.txt): 33 sites per window 2.79 ms against 3.32 ms for
	// the two-level scheme, 100 sites per window 2.31 against 2.08 ms (a thread per window leaves most of a CTA idle once
	// windows are long): chosen below 48 sites per window.  (The batch table lives in the unit-partial area, one entry
	// per batch + 1: tiny scans keep the two-level scheme.)
	const bool small = g_tune_xsmall != 1 && plan->max_window_sites <= kXMaxSmallWindow && plan->nunits > 0 &&
	                   (g_tune_xsmall == 2 || plan->nsites / plan->nunits < 48) && L.nunit >= L.nsite / kXTileStep + 2;
	switch (mode) {
		case XMODE_ABS: rc = x_run<XMODE_ABS>(P, L.nsite, L.nunit, d_score, d_pos, part, dout, small, st); break;
		case XMODE_MAX: rc = x_run<XMODE_MAX>(P, L.nsite, L.nunit, d_score, d_pos, part, dout, small, st); break;
		default: rc = x_run<XMODE_MIN>(P, L.nsite, L.nunit, d_score, d_pos, part, dout, small, st); break;
	}
	if (rc != PGT_OK) return rc;
	if (mem == PGT_MEM_HOST) {
		std::vector<uint64_t> site_tmp;
		uint64_t* h_site = out->ext_site;
		if (!h_site && out->ext_pos) {
			site_tmp.resize(L.nw);
			h_site = site_tmp.data();
		}
		pgt_xwindows host = *out;  // (ext_pos: gathered below)
		host.ext_site = h_site;
		host.ext_pos = nullptr;
		cudaError_t e = cudaSuccess;
		auto back = [&](auto* h, auto* d) {
			if (e == cudaSuccess && h) e = cudaMemcpyAsync(h, d, L.nw * sizeof(*h), cudaMemcpyDeviceToHost, st);
		};
		for_each_xfield(back, host, dout);
		if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(window table -> host)");
		PGT_CUDA(cudaStreamSynchronize(st));
		if (out->ext_pos) {
			for (uint64_t w = 0; w < L.nw; ++w) out->ext_pos[w] = h_site[w] == ~0ull ? 0u : pos[h_site[w] - origin];
		}
	}
	return PGT_OK;
}
