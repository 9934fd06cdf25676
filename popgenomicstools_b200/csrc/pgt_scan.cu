// pgt_scan.cu -- CUDA (sm_100a) implementation of the windowed site-statistic scan + C ABI.
//
// Replaces calcWindow of the reference (/root/reference/fstWindow.cpp:69-107,
// hetWindow.cpp:66-105, dxyWindow.cpp:172-209) -- a sequential re-sum of a W-entry buffer per
// window followed by a slide-by-copy -- with a one-pass reduction over columnar site arrays:
//
//   level 1  k_units<Stat>   : every site is read from HBM exactly once; the per-site statistic
//                              is evaluated in registers and reduced (lane-strided partial sums +
//                              warp-shuffle butterfly) into one partial per *unit* (pgt_geom.h).
//   level 2  k_windows<Stat> : every window is the sum of its consecutive unit partials (the
//                              carry across overlapping windows: W/S-fold overlap costs re-reads
//                              of small partials from L2, never of sites), plus the epilogue
//                              (ratio, position gather at the two window edges, label lookup).
//   (dxy)    k_global_*      : dxyWindow's global line from the same unit partials (two stages).
//   (bp)     k_bp_bounds     : dxyWindow -fixedsite 0: the reference materialises one buffer entry
//                              per bp (dxyWindow.cpp:365-372); here units live on the bp axis and
//                              each unit's site range is found by binary search in `pos` (sparse,
//                              O(#sites) instead of O(chromosome length)).
//
//   (fine)   k_slide<Stat>   : fine steps under long windows (W = 1000, S = 1): windows formed straight
//                              from the sites in shared memory, no unit array (pgt_slide.cuh).
//
// Device code lives in pgt_kernels_common.cuh (plan, statistics), pgt_level1.cuh, pgt_level2.cuh and
// pgt_slide.cuh, all included below into this one translation unit; this file holds the host side: layout of
// the caller-owned workspace, kernel selection and launches, host-memory mode, the C ABI entry points.
// There is no CPU fallback: every entry point fails with PGT_ERR_CUDA when no device is usable.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "pgt_cuda.h"

// ----------------------------------------------------------------------------- utilities

static std::atomic<uint64_t> g_launches{0};
extern "C" uint64_t pgt_kernel_launch_count(void) { return g_launches.load(); }
void pgt_count_launch() { g_launches++; }

extern "C" int pgt_device_count(void) {
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
	return n;
}
extern "C" int pgt_set_device(int device) {
	PGT_CUDA(cudaSetDevice(device));
	return PGT_OK;
}
extern "C" int pgt_host_alloc(void** p, size_t bytes) {
	if (!p) return pgt_set_error(PGT_ERR_ARGS, "pgt_host_alloc: NULL");
	PGT_CUDA(cudaHostAlloc(p, bytes, cudaHostAllocPortable));  // page-locked for every device of the process (pgt_scan_sharded)
	return PGT_OK;
}
extern "C" int pgt_host_free(void* p) {
	PGT_CUDA(cudaFreeHost(p));
	return PGT_OK;
}
extern "C" int pgt_device_alloc(void** p, size_t bytes) {
	if (!p) return pgt_set_error(PGT_ERR_ARGS, "pgt_device_alloc: NULL");
	PGT_CUDA(cudaMalloc(p, bytes ? bytes : 1));
	return PGT_OK;
}
extern "C" int pgt_device_free(void* p) {
	PGT_CUDA(cudaFree(p));
	return PGT_OK;
}
// ---- result tables shared between the processes of one box (one process per GPU, SURVEY.md §8e): rank 0 exports
// its table (pgt_device_alloc memory), the others map it and pass pointers into it as their `out` arrays, so the
// window kernels write each shard's rows straight into rank 0's HBM over NVLink -- no gather step at all.
extern "C" int pgt_ipc_export(const void* devptr, void* handle, size_t handle_bytes) {
	if (!devptr || !handle || handle_bytes < sizeof(cudaIpcMemHandle_t)) return pgt_set_error(PGT_ERR_ARGS, "pgt_ipc_export: need a device pointer and 64 bytes for the handle");
	cudaIpcMemHandle_t h;
	PGT_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(devptr)));
	memcpy(handle, &h, sizeof(h));
	return PGT_OK;
}
extern "C" int pgt_ipc_open(const void* handle, void** devptr) {
	if (!handle || !devptr) return pgt_set_error(PGT_ERR_ARGS, "pgt_ipc_open: NULL");
	cudaIpcMemHandle_t h;
	memcpy(&h, handle, sizeof(h));
	PGT_CUDA(cudaIpcOpenMemHandle(devptr, h, cudaIpcMemLazyEnablePeerAccess));
	return PGT_OK;
}
extern "C" int pgt_ipc_close(void* devptr) {
	PGT_CUDA(cudaIpcCloseMemHandle(devptr));
	return PGT_OK;
}
extern "C" int pgt_host_register(void* p, size_t bytes) {
	PGT_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterDefault));
	return PGT_OK;
}
extern "C" int pgt_host_unregister(void* p) {
	PGT_CUDA(cudaHostUnregister(p));
	return PGT_OK;
}

// ---- optional per-kernel timing (bench.py roofline): CUDA events on the launching stream (ProfScope, pgt_cuda.h)
struct ProfEvent {
	cudaEvent_t a, b;
	int kind;
};
static std::atomic<bool> g_profile{false};
static std::mutex g_prof_mutex;  // scans may run from several host threads while profiling is on
static std::vector<ProfEvent> g_prof_events;
static double g_prof_ms[4] = {0, 0, 0, 0};
static uint64_t g_prof_n[4] = {0, 0, 0, 0};

bool pgt_profile_enabled() { return g_profile; }
void pgt_profile_push(int kind, void* ev_a, void* ev_b) {
	std::lock_guard<std::mutex> lk(g_prof_mutex);
	g_prof_events.push_back(ProfEvent{(cudaEvent_t)ev_a, (cudaEvent_t)ev_b, kind});
}

extern "C" int pgt_profile(int enable) {
	g_profile = enable != 0;
	return PGT_OK;
}

// synchronise all recorded events and fold them into the per-kind totals
static int prof_drain() {
	std::lock_guard<std::mutex> lk(g_prof_mutex);
	for (ProfEvent& e : g_prof_events) {
		float t = 0;
		cudaError_t err = cudaEventSynchronize(e.b);
		if (err == cudaSuccess) err = cudaEventElapsedTime(&t, e.a, e.b);
		cudaEventDestroy(e.a);
		cudaEventDestroy(e.b);
		if (err != cudaSuccess) {
			g_prof_events.clear();
			return cuda_fail(err, "pgt_profile_read");
		}
		g_prof_ms[e.kind & 3] += t;
		g_prof_n[e.kind & 3]++;
	}
	g_prof_events.clear();
	return PGT_OK;
}
static int prof_read(int k0, double* units_ms, uint64_t* units_launches, double* windows_ms, uint64_t* windows_launches) {
	PGT_TRY(prof_drain());
	if (units_ms) *units_ms = g_prof_ms[k0];
	if (units_launches) *units_launches = g_prof_n[k0];
	if (windows_ms) *windows_ms = g_prof_ms[k0 + 1];
	if (windows_launches) *windows_launches = g_prof_n[k0 + 1];
	g_prof_ms[k0] = g_prof_ms[k0 + 1] = 0;
	g_prof_n[k0] = g_prof_n[k0 + 1] = 0;
	return PGT_OK;
}
extern "C" int pgt_profile_read(double* units_ms, uint64_t* units_launches, double* windows_ms, uint64_t* windows_launches) {
	return prof_read(0, units_ms, units_launches, windows_ms, windows_launches);
}
extern "C" int pgt_profile_read_extreme(double* units_ms, uint64_t* units_launches, double* windows_ms, uint64_t* windows_launches) {
	return prof_read(2, units_ms, units_launches, windows_ms, windows_launches);
}

// tuning knobs (tests / experiments, pgt_tune):
//   level1: 0 auto, 1 force the direct kernel (k_units; only valid when pgt_geom.gw == 32), 2 force the tiled kernel
//   level2: 0 auto, 1 force warp-per-window, 2 force scan mode (k_block_scan + k_windows_hgw)
static int g_tune_level1 = 0;
static int g_tune_level2 = 0;
static int g_tune_stages = 2;      // tiled kernel: shared-memory stages (2..4)
static int g_tune_stage_kb = 110;  // tiled kernel: KB per stage (stages * stage_kb <= 224)
extern int g_tune_xgroup;          // extreme scan (pgt_extreme.cu): lanes per unit, 0 = auto
extern int g_tune_xsmall;          // extreme scan: 0 auto, 1 never / 2 always (if the longest window fits) the small-window kernel
//   unittable: 0 auto (unit-start table for plans of more than 32 segments, device mode), 1 never, 2 always
static int g_tune_unittable = 0;
static constexpr size_t kUnitTableMinSegs = 33;  // measured (profiles/r02o_*): better from 1e3 contigs on, 3.8x at 1e6; few-contig genomes keep the closed form
//   fused2: 0 auto (fused sliding tile with one block per step: two crews, k_slide_fused2), 1 the single-crew k_slide<FusedStat>
static int g_tune_fused2 = 0;
//   persite: 0 auto (W = S = 1: four windows per thread with 128-bit accesses when everything is aligned), 1 always the scalar kernel
static int g_tune_persite = 0;
//   slide: 0 auto, 1 never use the sliding-tile kernel (k_slide), 2 use it whenever it fits shared memory (any W <= 1048)
static int g_tune_slide = 0;
// 0: the sliding tile also takes dxyWindow's global line when its runs own exactly the line's sites; 1: always a separate pass
static int g_tune_slideglobal = 0;

// Grid of a grid-stride kernel that wants `want` blocks: at most 8 per SM.
static unsigned capped_grid(uint64_t want) {
	const uint64_t cap = (uint64_t)num_sms() * 8;
	return (unsigned)(want < cap ? want : cap);
}

#include "pgt_kernels_common.cuh"
#include "pgt_level1.cuh"
#include "pgt_level2.cuh"
#include "pgt_slide.cuh"

// ----------------------------------------------------------------------------- host side of a scan

static const uint64_t kSlabSites = 1ull << 22;  // PGT_MEM_HOST: sites (entries) staged per slab
static const uint64_t kSlabSlack = 8192;         // >= 2 units

// One input column: where its pointer lives inside Cols, and its bytes per site.
struct ColDesc {
	size_t member;  // offsetof(Cols, ...)
	uint32_t elem;
};

// The extreme-score statistic (XStat) inside the host code: not a pgt_stat of the ABI (pgt_scan rejects it), only a
// key of the per-statistic tables below.
static constexpr pgt_stat kStatExtreme = (pgt_stat)16;

// The columns a statistic reads, in staging order -- pos first in bp mode, then a b f1 f2 n1 n2 g score.  The tiled and
// sliding-tile kernels read their staged columns in this order.
static int stat_columns(pgt_stat stat, pgt_mode mode, ColDesc* d) {
	int n = 0;
	if (mode == PGT_MODE_BP) d[n++] = {offsetof(Cols, pos), 4};
	if (stat == PGT_STAT_FST || stat == PGT_STAT_FUSED) {
		d[n++] = {offsetof(Cols, a), 8};
		d[n++] = {offsetof(Cols, b), 8};
	}
	if (stat == PGT_STAT_DXY || stat == PGT_STAT_FUSED) {
		d[n++] = {offsetof(Cols, f1), 8};
		d[n++] = {offsetof(Cols, f2), 8};
		d[n++] = {offsetof(Cols, n1), 4};
		d[n++] = {offsetof(Cols, n2), 4};
	}
	if (stat == PGT_STAT_HET || stat == PGT_STAT_FUSED) d[n++] = {offsetof(Cols, g), 1};
	if (stat == kStatExtreme) d[n++] = {offsetof(Cols, score), 8};
	return n;
}
static const void* col_ptr(const Cols& c, const ColDesc& d) {
	const void* p;
	memcpy(&p, (const char*)&c + d.member, sizeof(p));
	return p;
}
static void set_col_ptr(Cols* c, const ColDesc& d, const void* p) { memcpy((char*)c + d.member, &p, sizeof(p)); }

static Cols cols_from(const pgt_columns& c, int minind) { return Cols{c.pos, c.a, c.b, c.geno, c.f1, c.f2, c.n1, c.n2, nullptr, minind, 0.0}; }

template <class Stat>
static constexpr pgt_stat kStatOf = IsXStat<Stat>::value                 ? kStatExtreme
                                    : std::is_same<Stat, FstStat>::value ? PGT_STAT_FST
                                    : std::is_same<Stat, HetStat>::value ? PGT_STAT_HET
                                    : std::is_same<Stat, DxyStat>::value ? PGT_STAT_DXY
                                                                         : PGT_STAT_FUSED;

static size_t acc_bytes(pgt_stat stat) {
	if (stat == kStatExtreme) return sizeof(XStat<XMODE_ABS>::Acc);
	switch (stat) {
		case PGT_STAT_FST: return sizeof(FstStat::Acc);
		case PGT_STAT_HET: return sizeof(HetStat::Acc);
		case PGT_STAT_DXY: return sizeof(DxyStat::Acc);
		default: return sizeof(FusedStat::Acc);
	}
}

// Sliding-tile scan (k_slide): shared-memory shape, and whether the geometry takes that path at all.
struct SlideShape {
	uint32_t E, wpb, G, wp, nstages, stage_bytes, sf_off, pr_off, pos_off, stage_off, ncol;
	uint32_t col_off[kMaxStageCols], col_cap[kMaxStageCols];
	size_t smem;
};
// (sized with the position column staged, whether or not a scan passes positions: the choice of path must
// not depend on it)
static void slide_footprint(const pgt_geom& g, pgt_stat stat, SlideShape* sh) {
	const SlideTeam tm = slide_team(g.W);
	sh->E = tm.E;
	sh->wpb = tm.wpb;
	sh->G = tm.G;
	sh->wp = (uint32_t)align_up(g.W, 32);
	ColDesc d[8];
	const int nc = stat_columns(stat, PGT_MODE_SITES, d);
	uint32_t o = 0;
	for (int c = 0; c <= nc; ++c) {  // column nc = pos (uint32); a stage holds the G blocks of a step
		sh->col_off[c] = o;
		sh->col_cap[c] = (uint32_t)align_up((size_t)tm.G * g.W * (c < nc ? d[c].elem : 4) + 48, 16);
		o += sh->col_cap[c];
	}
	sh->ncol = (uint32_t)nc;
	sh->stage_bytes = (uint32_t)align_up(o, 128);
	const uint32_t accb = (uint32_t)align_up((size_t)tm.G * sh->wp * acc_bytes(stat), 128);
	sh->sf_off = kTileCtlBytes + kSlideWtBytes;
	sh->pr_off = sh->sf_off + 2 * accb;              // SUF: two halves (step parity)
	sh->pos_off = sh->pr_off + accb;
	sh->stage_off = sh->pos_off + 2 * tm.G * sh->wp * 4;  // positions: two halves
}
static bool slide_shape(const pgt_geom& g, pgt_mode mode, pgt_stat stat, SlideShape* sh) {
	if (mode != PGT_MODE_SITES || g_tune_slide == 1) return false;
	if (g.W > (uint32_t)kSlideConsumers * kSlideMaxE) return false;
	if (g_tune_slide != 2) {
		// auto: no piece of a step reaches a sector of doubles (units of < 32 sites) under windows of many
		// units -- where level 2 would otherwise run its block scans over a unit array as large as the input
		if (g.ueff >= 32 || g.wunits <= 32) return false;
	}
	const size_t half = 113u * 1024u, full = 226u * 1024u;
	// One rule for all statistics (the fused scan must equal the three single scans bit for bit): the block
	// of the widest one -- fused, 41 B/site staged twice + two 40-byte accumulators per site -- has to fit,
	// which bounds W at 1048 sites.
	slide_footprint(g, PGT_STAT_FUSED, sh);
	if (sh->stage_off + 2 * (size_t)sh->stage_bytes > full) return false;
	slide_footprint(g, stat, sh);
	// two CTAs per SM when three (or two) stages fit half the shared memory, else one CTA with up to four
	for (uint32_t ns : {3u, 2u}) {
		if (sh->stage_off + (size_t)ns * sh->stage_bytes <= half) {
			sh->nstages = ns;
			sh->smem = sh->stage_off + (size_t)ns * sh->stage_bytes;
			return true;
		}
	}
	for (uint32_t ns : {4u, 3u, 2u}) {
		if (sh->stage_off + (size_t)ns * sh->stage_bytes <= full) {
			sh->nstages = ns;
			sh->smem = sh->stage_off + (size_t)ns * sh->stage_bytes;
			return true;
		}
	}
	return false;
}

// The kernel path of a scan of `stat` over `plan` (PGT_PATH_*), and for the sliding tile its shape.  The path fixes
// the summation order, so it is a function of (W, S, unit, statistic) and the tuning knobs only -- never of the input
// size, the window range or the shard.
static int scan_path(const pgt_plan* plan, pgt_stat stat, SlideShape* sh) {
	if (stat != kStatExtreme && slide_shape(plan->g, plan->mode, stat, sh)) return PGT_PATH_SLIDE;
	if (plan->mode == PGT_MODE_SITES && plan->g.W == 1 && plan->g.S == 1 && g_tune_level2 != 1) return PGT_PATH_PERSITE;
	return PGT_PATH_UNITS;
}

struct Layout {
	uint64_t w_lo, w_hi, u_lo, u_hi, g_hi, origin;
	size_t segs_off, off_off, siteoff_off, gpart_off, units_off, pre_off, bounds_off, stage_off, outs_off, tileseg_off, flag_off, total;
	uint64_t tileseg_cap;  // entries of the tile -> segment table (0 = not used: few segments)
	bool hgw;              // level 2 in scan mode
	bool unit_table;       // very many segments: level 1 reads unit starts from a table (k_unit_starts) instead of the segment records
	// PGT_PATH_UNITS: level 1 (unit partials) + level 2.  PGT_PATH_SLIDE (fine steps: k_slide) and PGT_PATH_PERSITE
	// (W = S = 1: k_windows_persite) form the windows straight from the sites: no unit array, no level 2.
	int path;
	SlideShape slide;             // PGT_PATH_SLIDE
	uint64_t gsite_lo, gsite_hi;  // global sites this scan owns for dxyWindow's global line
	size_t gslab_off;             // host mode without units: one global-line triple per slab
	uint64_t out_slab_rows;       // host mode without units: rows of each of the two slab-sized output tables
	uint64_t gslab_cap;
	uint64_t blk_lo, blk_hi;  // scan blocks covering [u_lo, u_hi)
	size_t stage_col_bytes[8];
	uint64_t slab_sites;
};

static int make_layout(const pgt_plan* plan, const pgt_range* range, pgt_stat stat, pgt_mem mem, Layout* L) {
	if (!plan) return pgt_set_error(PGT_ERR_ARGS, "plan is NULL");
	if (stat != kStatExtreme && ((int)stat < 0 || (int)stat > (int)PGT_STAT_FUSED)) return pgt_set_error(PGT_ERR_ARGS, "unknown statistic");
	uint64_t lo = 0, hi = plan->nwin, org = plan->off[0];
	if (range) {
		if (range->w_hi != 0 || range->w_lo != 0) {
			lo = range->w_lo;
			hi = range->w_hi;
		}
		org = range->site_origin;
	}
	if (lo > hi || hi > plan->nwin) return pgt_set_error(PGT_ERR_ARGS, "window range out of bounds");
	memset(L, 0, sizeof(*L));
	L->w_lo = lo;
	L->w_hi = hi;
	L->origin = org;
	uint64_t f, c;
	// units reduced: from the first unit of window w_lo (axis head for w_lo == 0) to the last unit
	// of window w_hi-1 (axis tail for w_hi == nwin); units owned for the global line end where
	// the next shard's first window starts.
	if (hi == lo && plan->nwin != 0) {
		L->u_lo = L->u_hi = L->g_hi = 0;
	} else {
		if (lo == 0) L->u_lo = 0;
		else {
			pgt_plan_window_units(plan, lo, &f, &c);
			L->u_lo = f;
		}
		if (hi == plan->nwin) L->u_hi = L->g_hi = plan->nunits;
		else {
			pgt_plan_window_units(plan, hi - 1, &f, &c);
			L->u_hi = f + c;
			pgt_plan_window_units(plan, hi, &f, &c);
			L->g_hi = f;
		}
	}
	// sites owned for the global line (same boundaries as the units [u_lo, g_hi))
	L->gsite_lo = pgt_plan_unit_start(plan, L->u_lo);
	L->gsite_hi = pgt_plan_unit_start(plan, L->g_hi);
	L->path = scan_path(plan, stat, &L->slide);
	const bool nounits = L->path != PGT_PATH_UNITS;
	const uint64_t nunits = nounits ? 0 : L->u_hi - L->u_lo;
	size_t o = 0;
	L->segs_off = o;
	o += align_up(plan->segs.size() * sizeof(pgt_seg) + 8, 256);
	L->off_off = o;
	o += align_up(plan->off.size() * sizeof(uint64_t), 256);
	L->siteoff_off = o;
	if (plan->mode == PGT_MODE_BP) o += align_up(plan->off.size() * sizeof(uint64_t), 256);
	L->gpart_off = o;
	o += align_up((size_t)kGlobalMaxPartials * 3 * sizeof(double), 256);
	L->units_off = o;
	o += align_up((size_t)nunits * acc_bytes(stat) + 8, 256);
	// level 2 in scan mode when summing wunits partials per window would dominate (fine steps, long windows)
	{
		// costs in partial reads/writes; the totals are exact for the whole plan (genomes of many short
		// contigs have windows far shorter than wunits and at least one scan block per segment) and
		// scaled to the window range of a shard
		const double frac = plan->nwin ? (double)(hi - lo) / (double)plan->nwin : 0.0;
		const double direct = (double)plan->window_units_total * frac;
		const double scan = 4.0 * (3.0 * (double)plan->scan_units_total * frac + 2.0 * (double)(hi - lo));
		L->hgw = plan->g.wunits > 32 && direct > scan;
		if (g_tune_level2 == 1) L->hgw = false;
		if (g_tune_level2 == 2 && plan->g.wunits >= 2) L->hgw = true;
	}
	if (nounits) L->hgw = false;
	L->pre_off = o;
	L->blk_lo = L->blk_hi = 0;
	// PRE array: reserved whenever scan mode is possible, so the workspace size does not depend on the
	// (tunable) kernel choice
	if (plan->g.wunits >= 2 && nunits) o += align_up((size_t)nunits * acc_bytes(stat) + 8, 256);
	if (L->hgw && nunits) {
		const pgt_seg& s0 = plan->segs[pgt_plan_seg_of_unit(plan, L->u_lo)];
		const pgt_seg& s1 = plan->segs[pgt_plan_seg_of_unit(plan, L->u_hi - 1)];
		L->blk_lo = s0.blk_base + (L->u_lo - s0.unit_base) / plan->g.wunits;
		L->blk_hi = s1.blk_base + (L->u_hi - 1 - s1.unit_base) / plan->g.wunits + 1;
	}
	L->bounds_off = o;
	L->unit_table = plan->mode == PGT_MODE_SITES && mem == PGT_MEM_DEVICE && nunits > 0 &&
	                (g_tune_unittable == 2 || (g_tune_unittable == 0 && plan->segs.size() >= kUnitTableMinSegs));
	if (plan->mode == PGT_MODE_BP || L->unit_table) o += align_up((size_t)(nunits + 1) * sizeof(uint64_t), 256);
	L->stage_off = o;
	L->outs_off = o;
	if (mem == PGT_MEM_HOST) {
		L->slab_sites = std::min<uint64_t>(kSlabSites, std::max<uint64_t>(plan->nsites, 1)) + kSlabSlack;
		ColDesc d[8];
		const int nc = stat_columns(stat, plan->mode, d);
		for (int i = 0; i < nc; ++i) L->stage_col_bytes[i] = align_up((size_t)L->slab_sites * d[i].elem, 256);
		for (int s = 0; s < 2; ++s)
			for (int i = 0; i < nc; ++i) o += L->stage_col_bytes[i];
		L->outs_off = o;
		// staged per-window outputs + global[3]: the whole table, or (no unit array: the windows are produced
		// slab by slab) two tables of at most one slab's windows -- a window starts at its own site
		L->out_slab_rows = std::min<uint64_t>(hi - lo, L->slab_sites);
		if (nounits) o += 2 * 12 * align_up((size_t)L->out_slab_rows * 8 + 8, 256);
		else o += 12 * align_up((size_t)(hi - lo) * 8 + 8, 256);
		L->gslab_off = o;
		L->gslab_cap = nounits ? plan->nsites / (L->slab_sites - kSlabSlack - std::min<uint64_t>(plan->g.W, L->slab_sites - kSlabSlack - 1)) + 16 : 0;
		o += align_up((size_t)L->gslab_cap * 3 * sizeof(double), 256);
	}
	// tile -> first segment table of the tiled level-1 kernel (genomes of many contigs, see k_tile_segs)
	L->tileseg_off = o;
	L->tileseg_cap = plan->segs.size() > kTileSegTableMin ? nunits / 8 + 1024 : 0;
	o += align_up((size_t)L->tileseg_cap * sizeof(uint32_t), 256);
	// extreme scan of a bp plan in device memory: the position check's flag
	L->flag_off = o;
	if (stat == kStatExtreme && plan->mode == PGT_MODE_BP && mem == PGT_MEM_DEVICE) o += 256;
	L->total = o + 256;
	return PGT_OK;
}

extern "C" int pgt_plan_scan_path(const pgt_plan* plan, pgt_stat stat) {
	if (!plan) return pgt_set_error(PGT_ERR_ARGS, "pgt_plan_scan_path: plan is NULL");
	if ((int)stat < 0 || (int)stat > (int)PGT_STAT_FUSED) return pgt_set_error(PGT_ERR_ARGS, "unknown statistic");
	SlideShape sh;
	return scan_path(plan, stat, &sh);
}

extern "C" size_t pgt_plan_device_bytes(const pgt_plan* plan) {
	if (!plan) return 0;
	return table_pair_bytes(plan->segs.size() * sizeof(pgt_seg), plan->off.size() * sizeof(uint64_t));
}

extern "C" int pgt_plan_bind_device(pgt_plan* plan, void* buffer, size_t bytes, void* stream) {
	if (!plan) return pgt_set_error(PGT_ERR_ARGS, "pgt_plan_bind_device: plan is NULL");
	if (!buffer) {
		plan->d_tables = nullptr;
		return PGT_OK;
	}
	if (bytes < pgt_plan_device_bytes(plan)) return pgt_set_error(PGT_ERR_NOMEM, "pgt_plan_bind_device: buffer too small");
	return bind_table_pair(buffer, plan->segs.data(), plan->segs.size() * sizeof(pgt_seg), plan->off.data(), plan->off.size() * sizeof(uint64_t),
	                       stream, &plan->d_tables);
}

extern "C" size_t pgt_scan_workspace_bytes(const pgt_plan* plan, const pgt_range* range, pgt_stat stat, pgt_mem mem) {
	if ((int)stat < 0 || (int)stat > (int)PGT_STAT_FUSED) return 0;
	Layout L;
	if (make_layout(plan, range, stat, mem, &L) != PGT_OK) return 0;
	return L.total;
}

extern "C" int pgt_tune(const char* key, int value) {
	if (key && strcmp(key, "level1") == 0) g_tune_level1 = value;
	else if (key && strcmp(key, "level2") == 0 && value >= 0 && value <= 2) g_tune_level2 = value;
	else if (key && strcmp(key, "slide") == 0 && value >= 0 && value <= 2) g_tune_slide = value;
	else if (key && strcmp(key, "fused2") == 0 && value >= 0 && value <= 1) g_tune_fused2 = value;
	else if (key && strcmp(key, "slideglobal") == 0 && value >= 0 && value <= 1) g_tune_slideglobal = value;
	else if (key && strcmp(key, "persite") == 0 && value >= 0 && value <= 1) g_tune_persite = value;
	else if (key && strcmp(key, "unittable") == 0 && value >= 0 && value <= 2) g_tune_unittable = value;
	else if (key && strcmp(key, "stages") == 0 && value >= 2 && value <= kTileMaxStages) g_tune_stages = value;
	else if (key && strcmp(key, "stage_kb") == 0 && value >= 8 && value <= 110) g_tune_stage_kb = value;
	else if (key && strcmp(key, "xsmall") == 0 && value >= 0 && value <= 2) g_tune_xsmall = value;
	else if (key && strcmp(key, "xgroup") == 0 && (value == 0 || value == 4 || value == 8 || value == 16 || value == 32)) g_tune_xgroup = value;
	else return pgt_set_error(PGT_ERR_ARGS, "pgt_tune: unknown key");
	return PGT_OK;
}

// the statistic's columns of `c` for the tiled and sliding-tile kernels, in staging order
struct StatCols {
	const void* ptr[kMaxTileCols];
	uint32_t elem[kMaxTileCols];
	uint32_t n;
};
template <class Stat>
static StatCols tile_columns(const Cols& c) {
	ColDesc d[8];
	StatCols sc;
	sc.n = (uint32_t)stat_columns(kStatOf<Stat>, PGT_MODE_SITES, d);
	for (uint32_t i = 0; i < sc.n; ++i) {
		sc.ptr[i] = col_ptr(c, d[i]);
		sc.elem[i] = d[i].elem;
	}
	return sc;
}

// what the tiled level-1 kernel stages: bytes per site, and `nstages` stages of at most `stage_bytes` each
// (pgt_tune "stages" / "stage_kb", at most 224 KB in all)
struct TileBudget {
	uint32_t bps, nstages, stage_bytes;
};
static TileBudget tile_budget(const StatCols& sc) {
	TileBudget b{0, (uint32_t)g_tune_stages, (uint32_t)g_tune_stage_kb * 1024u};
	for (uint32_t c = 0; c < sc.n; ++c) b.bps += sc.elem[c];
	if (b.nstages * b.stage_bytes > 224u * 1024u) b.stage_bytes = 224u * 1024u / b.nstages;
	return b;
}

template <class Stat, bool INDIRECT>
static int launch_units_tiled(const DevPlan& P, const StatCols& sc, const TileBudget& tb, const Cols& cols, typename Stat::Acc* units,
                              const uint64_t* bounds, uint64_t valid_elems, uint32_t* tileseg, uint64_t tileseg_cap, cudaStream_t st) {
	const uint64_t nunits = P.unit_hi - P.unit_lo;
	const int nsm = num_sms();
	// `nstages` stages of <= `stage_kb` KB; tiles of whole units; at least ~4 tiles per SM when the input allows
	uint32_t tsites = (tb.stage_bytes - 48u * sc.n) / tb.bps;
	if (tsites > 16384u && tb.bps > 1) tsites = 16384u;  // (the 1-byte genotype column alone fills a stage with ~110 K sites)
	uint32_t m = tsites / P.g.ueff;
	if (m < 1) m = 1;
	{
		// A tile's units are dealt to NG consumer groups; a tile of m units takes ceil(m / NG) rounds.
		// When the last round would be mostly idle (measured: dxy, m = 18 over 15 warps, 6.29 TB/s;
		// m = 15, 6.80 TB/s) a smaller tile of whole rounds wins; a nearly full last round (fst,
		// m = 27 of 30) is better left alone: the larger tile keeps more bytes in flight.
		const uint32_t ng = (uint32_t)kTileConsumerWarps * (32u / P.g.gw);
		if (m > ng && m % ng != 0 && (double)m / (double)((m + ng - 1) / ng * ng) < 0.8) m = m / ng * ng;
	}
	const uint32_t cap_sites = m * P.g.ueff;  // sites a stage can hold (what the shared-memory regions are sized for)
	if (INDIRECT && nunits) {
		// bp mode: a unit is a bp range and holds anything from 0 to ueff sites.  Sizing tiles for the
		// dense worst case makes them nearly empty on sparse data (SNP-only MAFs: ~3 % full, and the
		// per-tile cost dominated: 5.6 ms for 1e8 sites over 3e9 bp).  Size them for the average
		// density instead; a tile whose slice does not fit is read straight from global memory by
		// the consumers (`staged` in the kernel), so dense stretches stay correct.
		const double avg = (double)valid_elems / (double)nunits;  // sites per unit
		const double want = 0.75 * (double)cap_sites / (avg > 1e-3 ? avg : 1e-3);
		const uint32_t m_sparse = want > 65536.0 ? 65536u : (uint32_t)want;
		if (m_sparse > m) m = m_sparse;
	}
	const uint64_t want_tiles = (uint64_t)nsm * 4;
	if ((nunits + m - 1) / m < want_tiles) {
		uint64_t mm = (nunits + want_tiles - 1) / want_tiles;
		m = (uint32_t)(mm < 1 ? 1 : mm);
	}
	TileCfg tc;
	memset(&tc, 0, sizeof(tc));
	tc.ncol = sc.n;
	tc.m = m;
	tc.nstages = tb.nstages;
	tc.minind = cols.minind;
	tc.cutoff = cols.cutoff;
	tc.valid_elems = valid_elems;
	uint32_t o = 0;
	for (uint32_t c = 0; c < sc.n; ++c) {
		tc.gcol[c] = (const char*)sc.ptr[c];
		tc.elem[c] = sc.elem[c];
		tc.col_off[c] = o;
		tc.col_cap[c] = (uint32_t)align_up((size_t)cap_sites * sc.elem[c] + 48, 16);
		o += tc.col_cap[c];
	}
	tc.stage_bytes = (uint32_t)align_up(o, 128);
	const size_t smem = kTileCtlBytes + tb.nstages * (size_t)tc.stage_bytes;
	void (*kern)(DevPlan, TileCfg, typename Stat::Acc*, const uint64_t*);
	switch (P.g.gw) {
		case 1: kern = k_units_tiled<Stat, 1, INDIRECT>; break;
		case 2: kern = k_units_tiled<Stat, 2, INDIRECT>; break;
		case 4: kern = k_units_tiled<Stat, 4, INDIRECT>; break;
		case 8: kern = k_units_tiled<Stat, 8, INDIRECT>; break;
		case 16: kern = k_units_tiled<Stat, 16, INDIRECT>; break;
		default: kern = k_units_tiled<Stat, 32, INDIRECT>; break;
	}
	PGT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	const uint64_t ntiles = (nunits + m - 1) / m;
	const unsigned grid = (unsigned)(ntiles < (uint64_t)nsm ? ntiles : (uint64_t)nsm);
	{
		ProfScope prof(0, st);
		if (!INDIRECT && tileseg && ntiles <= tileseg_cap && ntiles > grid) {  // many segments: tile -> segment table first
			k_tile_segs<<<(unsigned)((ntiles + 255) / 256), 256, 0, st>>>(P, m, ntiles, tileseg);
			g_launches++;
			tc.tile_seg = tileseg;
		}
		kern<<<grid, kTileThreads, smem, st>>>(P, tc, units, bounds);
	}
	g_launches++;
	PGT_CUDA(cudaGetLastError());
	return PGT_OK;
}

// valid_elems: number of elements every column is known to hold from element 0
template <class Stat>
static int launch_units(const DevPlan& P, const Cols& cols, typename Stat::Acc* units, const uint64_t* bounds, uint64_t valid_elems,
                        uint32_t* tileseg, uint64_t tileseg_cap, cudaStream_t st) {
	const uint64_t nunits = P.unit_hi - P.unit_lo;
	if (nunits == 0) return PGT_OK;
	// Kernel choice.  The direct kernel reduces every unit with a full warp, so it implements the
	// summation order only when gw == 32 (long units); short units always take the tiled kernel.
	// For long units both kernels give bit-identical results and the choice is purely a speed
	// matter (measured on B200, profiles/): the TMA-staged tiled kernel wins on big inputs
	// (no sector over-fetch, bytes in flight without registers), the direct kernel on small ones
	// (no pipeline fill) and for the 1-byte genotype column.
	const StatCols sc = tile_columns<Stat>(cols);
	const TileBudget tb = tile_budget(sc);
	const uint64_t approx_bytes = nunits * (uint64_t)P.g.ueff * tb.bps;
	// (hetWindow's 1-byte column stays on the vectorised direct kernel: measured at 3e9 sites, 4096-site units,
	// 6.14 TB/s direct against 5.44 TB/s through the ring -- both were issue-bound on the byte counting, 4.5 and
	// 4.3 TB/s, until it went from POPC to dp4a; the ring's het consumer remains for forced / short-unit runs)
	// (the extreme score too: at 1e9 sites, 50000/10000 the direct kernel took 2.01 ms against 2.30 ms through the ring,
	// dense bp 100000/10000 1.79 against 1.93 ms; profiles/r05b_plan_extreme_probe.jsonl)
	bool tiled = P.g.gw != 32 || (tb.bps > 1 && !IsXStat<Stat>::value && approx_bytes >= (256ull << 20));
	if (g_tune_level1 == 2) tiled = true;
	if (g_tune_level1 == 1 && P.g.gw == 32) tiled = false;
	// a tile holds whole units: very long units (unit_sites up to 4096) may not fit a stage;
	// they always have gw == 32, so the direct kernel applies
	if ((uint64_t)P.g.ueff * tb.bps + 64ull * kMaxTileCols > tb.stage_bytes) tiled = false;
	if (tiled)
		return bounds ? launch_units_tiled<Stat, true>(P, sc, tb, cols, units, bounds, valid_elems, nullptr, 0, st)
		              : launch_units_tiled<Stat, false>(P, sc, tb, cols, units, bounds, valid_elems, tileseg, tileseg_cap, st);
	const int threads = 256;
	const uint64_t want = (nunits + 7) / 8;  // one warp per unit, 8 warps per block
	if constexpr (std::is_same<Stat, HetStat>::value) {  // hetWindow: the vectorised byte kernel replaces the generic direct kernel
		const unsigned grid = capped_grid(want);
		{
			ProfScope prof(0, st);
			if (bounds) k_units_het_vec<true><<<grid, 256, 0, st>>>(P, cols.g, units, bounds);
			else k_units_het_vec<false><<<grid, 256, 0, st>>>(P, cols.g, units, bounds);
		}
		g_launches++;
		PGT_CUDA(cudaGetLastError());
		return PGT_OK;
	}
	const uint32_t upl = P.g.u / 32u;
	void (*kern)(DevPlan, Cols, typename Stat::Acc*, const uint64_t*);
	if (bounds) kern = upl == 8 ? k_units<Stat, 8, true> : k_units<Stat, 0, true>;
	else kern = upl == 8 ? k_units<Stat, 8, false> : (upl == 4 ? k_units<Stat, 4, false> : k_units<Stat, 0, false>);
	int per_sm = 0;
	PGT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, 0));
	const uint64_t cap = (uint64_t)num_sms() * (per_sm > 0 ? per_sm : 1);
	const unsigned grid = (unsigned)(want < cap ? want : cap);
	{
		ProfScope prof(0, st);
		kern<<<grid, threads, 0, st>>>(P, cols, units, bounds);
	}
	g_launches++;
	PGT_CUDA(cudaGetLastError());
	return PGT_OK;
}

static int launch_bounds_kernel(const DevPlan& P, const uint32_t* pos, uint64_t ndata, uint64_t* bounds, cudaStream_t st) {
	const uint64_t nb = P.unit_hi - P.unit_lo + 1;
	k_bp_bounds<<<capped_grid((nb + 255) / 256), 256, 0, st>>>(P, pos, ndata, bounds);
	g_launches++;
	PGT_CUDA(cudaGetLastError());
	return PGT_OK;
}

// scan mode (L.hgw): `units` is scanned in place into SUF, `pre` receives PRE; see k_block_scan
template <class Stat>
static int launch_windows(const DevPlan& P, typename Stat::Acc* units, uint64_t units_base, const uint32_t* pos, const typename Stat::Out& out,
                          bool hgw, typename Stat::Acc* pre, uint64_t blk_lo, uint64_t blk_hi, cudaStream_t st) {
	const uint64_t nwin = P.win_hi - P.win_lo;
	if (nwin == 0) return PGT_OK;
	ProfScope prof(1, st);
	if (hgw) {
		k_block_scan<Stat><<<capped_grid(blk_hi - blk_lo), 256, 0, st>>>(P, units, pre, units_base, blk_lo, blk_hi);
		g_launches++;
		k_windows_hgw<Stat><<<capped_grid((nwin + 255) / 256), 256, 0, st>>>(P, units, pre, units_base, pos, out);
	} else if (P.g.wunits <= 32 && g_tune_level2 != 1) {
		// fine windows: a thread per window
		void (*kern)(DevPlan, const typename Stat::Acc*, uint64_t, const uint32_t*, typename Stat::Out);
		const uint32_t wu = P.g.wunits;
		if (wu <= 1) kern = k_windows_small<Stat, 1>;
		else if (wu <= 2) kern = k_windows_small<Stat, 2>;
		else if (wu <= 4) kern = k_windows_small<Stat, 4>;
		else if (wu <= 8) kern = k_windows_small<Stat, 8>;
		else if (wu <= 16) kern = k_windows_small<Stat, 16>;
		else kern = k_windows_small<Stat, 32>;
		kern<<<capped_grid((nwin + 255) / 256), 256, 0, st>>>(P, units, units_base, pos, out);
	} else {
		// few windows: a warp each; many: runs per block, stored 32 rows at a time
		k_windows<Stat><<<capped_grid((nwin + 7) / 8), 256, 0, st>>>(P, units, units_base, pos, out);
	}
	g_launches++;
	PGT_CUDA(cudaGetLastError());
	return PGT_OK;
}

// dxyWindow's global line from the unit partials (two stages); nothing for the statistics without one
template <class Stat>
static int launch_global(const typename Stat::Acc* units, uint64_t n, double* scratch, double* g3, cudaStream_t st) {
	if constexpr (GlobalTerm<Stat>::has) {
		k_global_partial<Stat><<<kGlobalBlocks, 1024, 0, st>>>(units, n, scratch);
		k_global_final<<<1, kGlobalBlocks, 0, st>>>(scratch, kGlobalBlocks, g3);
		g_launches += 2;
		PGT_CUDA(cudaGetLastError());
	}
	return PGT_OK;
}

// Sliding-tile scan of the windows [P.win_lo, P.win_hi) in the shape `sh` (Layout::slide): the columns' element 0 is
// site P.site_origin and they hold `valid_elems` elements.  `pos` may be NULL (host mode gathers positions on the host).
template <class Stat>
static int launch_slide(const pgt_plan* plan, const SlideShape& sh, const DevPlan& P, const Cols& cols, uint64_t valid_elems,
                        const uint32_t* pos, const pgt_windows& out, double* gpart, double* g3, cudaStream_t st) {
	const uint64_t nwin = P.win_hi - P.win_lo;
	if (nwin == 0) return PGT_OK;
	const StatCols scol = tile_columns<Stat>(cols);
	TileCfg tc;
	memset(&tc, 0, sizeof(tc));
	tc.ncol = scol.n + (pos ? 1u : 0u);  // positions ride the ring too: read from HBM once, gathered from shared memory
	tc.nstages = sh.nstages;
	tc.stage_bytes = sh.stage_bytes;
	tc.minind = cols.minind;
	tc.valid_elems = valid_elems;
	for (uint32_t c = 0; c < tc.ncol; ++c) {
		tc.gcol[c] = c < scol.n ? (const char*)scol.ptr[c] : (const char*)pos;
		tc.elem[c] = c < scol.n ? scol.elem[c] : 4u;
		tc.col_off[c] = sh.col_off[c];
		tc.col_cap[c] = sh.col_cap[c];
	}
	SlideCfg sc;
	memset(&sc, 0, sizeof(sc));
	sc.E = sh.E;
	sc.wpb = sh.wpb;
	sc.G = sh.G;
	sc.wp = sh.wp;
	sc.sf_off = sh.sf_off;
	sc.pr_off = sh.pr_off;
	sc.pos_off = sh.pos_off;
	sc.pos_col = pos ? scol.n : 0xffffffffu;
	sc.stage_off = sh.stage_off;
	sc.gpart = gpart;
	void (*kern)(DevPlan, TileCfg, SlideCfg, pgt_windows) = nullptr;
	void (*k2)(DevPlan, TileCfg, SlideCfg, SlideCfg2, pgt_windows) = nullptr;
	SlideCfg2 s2;
	uint64_t slots;  // CTAs resident at once
	if (std::is_same<Stat, FusedStat>::value && sh.G == 1 && g_tune_fused2 != 1) {
		// two crews (fst + het, dxy) share the staged block; their SUF / PRE arrays partition the fused ones
		const uint32_t part[2] = {24u, 16u};  // accumulator bytes per site: FstHetStat, DxyStat
		uint32_t so = sh.sf_off, po = sh.pr_off;
		for (int c = 0; c < 2; ++c) {
			s2.wt_off[c] = kTileCtlBytes + 256u * c;
			s2.sf_off[c] = so;
			s2.pr_off[c] = po;
			so += 2u * sh.wp * part[c];
			po += sh.wp * part[c];
		}
		k2 = sh.E <= 4 ? k_slide_fused2<4> : (sh.E == 5 ? k_slide_fused2<5> : k_slide_fused2<6>);
		PGT_CUDA(cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh.smem));
		slots = (uint64_t)num_sms();
	} else {
		if (sh.G > 1) {
			if (sh.E <= 2) kern = k_slide<Stat, 2, true>;
			else if (sh.E <= 4) kern = k_slide<Stat, 4, true>;
			else kern = k_slide<Stat, 6, true>;
		} else {
			if (sh.E <= 4) kern = k_slide<Stat, 4, false>;
			else if (sh.E == 5) kern = k_slide<Stat, 5, false>;  // W = 1000
			else kern = k_slide<Stat, 6, false>;
		}
		PGT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh.smem));
		int per_sm = 0;
		PGT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSlideThreads, sh.smem));
		slots = (uint64_t)num_sms() * (per_sm < 1 ? 1 : per_sm);
	}
	// chunks: ~4 per resident CTA for balance, but long enough (>= 32 steps of windows) that the W - S sites
	// shared with the next chunk stay a few percent of what a chunk reads
	const uint64_t wps = ((uint64_t)sh.G * plan->g.W + plan->g.S - 1) / plan->g.S;  // windows starting in one step
	sc.chunk_windows = std::max<uint64_t>(32 * wps, (nwin + slots * 4 - 1) / (slots * 4));
	sc.nchunks = (nwin + sc.chunk_windows - 1) / sc.chunk_windows;
	const unsigned grid = (unsigned)std::min<uint64_t>(sc.nchunks, slots);
	{
		ProfScope prof(0, st);
		if (k2) k2<<<grid, kSlide2Threads, sh.smem, st>>>(P, tc, sc, s2, out);
		else kern<<<grid, kSlideThreads, sh.smem, st>>>(P, tc, sc, out);
	}
	g_launches++;
	PGT_CUDA(cudaGetLastError());
	if (gpart) {  // one partial triple per CTA -> the line
		k_global_final<<<1, kGlobalBlocks, 0, st>>>(gpart, grid, g3);
		g_launches++;
		PGT_CUDA(cudaGetLastError());
	}
	return PGT_OK;
}

// Do the sites the sliding-tile kernel counts as owned by its runs -- per segment from the first window's start to the
// start of the first window after the range, or to the end of the segment's last window -- make up exactly the range
// [gsite_lo, gsite_hi) of dxyWindow's global line?  (No when a segment inside the range has sites after its last window
// or no window at all: then the line is taken by a pass over the columns.)
static bool slide_runs_cover_owned_sites(const pgt_plan* plan, const Layout& L) {
	if (L.w_hi <= L.w_lo) return false;
	const uint64_t W = plan->g.W, S = plan->g.S;
	uint32_t si = pgt_plan_seg_of_window(plan, L.w_lo);
	uint64_t w = L.w_lo, cursor = L.gsite_lo;
	while (w < L.w_hi) {
		while (si < plan->segs.size() && w - plan->segs[si].win_base >= plan->segs[si].nwin) ++si;
		if (si >= plan->segs.size()) return false;
		const pgt_seg& sg = plan->segs[si];
		const uint64_t ka = w - sg.win_base, kb = std::min<uint64_t>(L.w_hi - sg.win_base, sg.nwin);
		if (sg.site_base + ka * S != cursor) return false;
		const uint64_t hi = kb == sg.nwin ? std::min<uint64_t>((kb - 1) * S + W, sg.nsites) : kb * S;
		cursor = sg.site_base + hi;
		w = sg.win_base + kb;
	}
	return cursor == L.gsite_hi;
}

// W = S = 1: the vectorised kernel when its preconditions hold (one segment; every used column and output pointer
// 16-byte aligned at the scan's first window -- 4-byte aligned for the genotype column), else the scalar one.  (The
// extreme scan has the scalar kernel only.)
template <class Stat>
static int launch_persite(const pgt_plan* plan, const DevPlan& P, const Cols& C, const typename Stat::Out& out, double* gpart, double* g3,
                          cudaStream_t st) {
	const uint64_t nwin = P.win_hi - P.win_lo;
	if (nwin == 0) return PGT_OK;
	bool vec = false;
	uint64_t site0 = 0;
	if constexpr (!IsXStat<Stat>::value) {
		vec = g_tune_persite != 1 && plan->segs.size() == 1 && nwin >= 4;
		if (vec) {
			site0 = plan->segs[0].site_base + (P.win_lo - plan->segs[0].win_base) - P.site_origin;
			auto ok = [&](const void* p, size_t elem, size_t align) { return !p || (((uintptr_t)p + site0 * elem) & (align - 1)) == 0; };
			ColDesc d[8];
			const int nc = stat_columns(kStatOf<Stat>, PGT_MODE_SITES, d);
			for (int i = 0; i < nc; ++i) vec = vec && col_ptr(C, d[i]) && ok(col_ptr(C, d[i]), d[i].elem, d[i].elem == 1 ? 4 : 16);
			vec = vec && ok(C.pos, 4, 16);
			for_each_field([&](const void* p) { vec = vec && (((uintptr_t)p) & 15) == 0; }, out);
		}
	}
	ProfScope prof(1, st);
	unsigned grid = 0;
	if (vec) {
		if constexpr (!IsXStat<Stat>::value) {
			grid = std::min<unsigned>(one_wave_grid(k_windows_persite4<Stat>, 256, (nwin + 1023) / 1024), kGlobalMaxPartials);
			k_windows_persite4<Stat><<<grid, 256, 0, st>>>(P, C, out, site0, gpart);
		}
	} else {
		grid = std::min<unsigned>(one_wave_grid(k_windows_persite<Stat>, 256, (nwin + 1023) / 1024), kGlobalMaxPartials);  // four windows per thread and turn
		k_windows_persite<Stat><<<grid, 256, 0, st>>>(P, C, out, gpart);
	}
	g_launches++;
	PGT_CUDA(cudaGetLastError());
	if (gpart) {  // the global line over exactly these windows' sites: one partial triple per block
		k_global_final<<<1, kGlobalBlocks, 0, st>>>(gpart, grid, g3);
		g_launches++;
		PGT_CUDA(cudaGetLastError());
	}
	return PGT_OK;
}

// dxyWindow's global line straight from the columns (scans without a unit array)
static int launch_global_sites(const Cols& cols, uint64_t i0, uint64_t i1, double* scratch, double* g3, cudaStream_t st) {
	k_global_sites<<<kGlobalBlocks, 1024, 0, st>>>(cols, i0, i1, scratch);
	k_global_final<<<1, kGlobalBlocks, 0, st>>>(scratch, kGlobalBlocks, g3);
	g_launches += 2;
	PGT_CUDA(cudaGetLastError());
	return PGT_OK;
}

// host-side lower bound of bp entry e on the site axis (bp mode, PGT_MEM_HOST)
static uint64_t host_site_lower_bound(const pgt_plan* plan, const uint64_t* site_off, const uint32_t* pos, uint64_t origin,
                                      uint64_t ndata, uint64_t e) {
	const uint32_t nc = (uint32_t)plan->off.size() - 1;
	uint64_t res;
	if (e >= plan->off[nc]) {
		res = site_off[nc];
	} else {
		const uint32_t c = pgt_plan_contig_of(plan, e);
		const uint32_t p = (uint32_t)(e - plan->off[c]) + 1u;
		uint64_t lo = std::max(site_off[c], origin), hi = std::min(site_off[c + 1], origin + ndata);
		if (hi < lo) hi = lo;
		const uint32_t* b = pos + (lo - origin);
		res = lo + (uint64_t)(std::lower_bound(b, pos + (hi - origin), p) - b);
	}
	return std::min(std::max(res, origin), origin + ndata);
}

// What the checks and set-up shared by both memory spaces establish for a scan.
struct Scan {
	const pgt_plan* plan;
	pgt_stat stat;
	Layout L;
	DevPlan P;
	Cols C;  // the caller's columns (device or host pointers)
	const uint64_t* site_offsets;
	const pgt_windows* out;  // the extreme scan: its geometry rows (all NULL when none are wanted)
	XRows x;                 // the extreme scan's rows (the caller's arrays; site_origin = the scan's)
	char* ws;
	uint64_t* bounds;  // bp mode / unit table: unit bounds in the workspace
	uint64_t ndata;    // bp mode: sites the columns hold
	uint64_t nglobal;  // units the global line sums
	bool bp, want_global;
	cudaStream_t st;
};

// the rows a scan of Stat writes
template <class Stat>
static typename Stat::Out rows_of(const Scan& s) {
	if constexpr (IsXStat<Stat>::value) return s.x;
	else return *s.out;
}

// bp mode: the first and last site this call holds of every chromosome must lie on the chromosome (1 <= pos <= length);
// *bad receives the smallest global index of a site that does not (left as it is when all do)
static void bp_check_positions_host(const pgt_plan* plan, const uint64_t* site_off, const uint32_t* pos, uint64_t origin, uint64_t ndata,
                                    uint64_t* bad) {
	const uint32_t nc = (uint32_t)plan->off.size() - 1;
	for (uint32_t c = 0; c < nc; ++c) {
		const uint64_t lo = std::max(site_off[c], origin), hi = std::min(site_off[c + 1], origin + ndata);
		if (hi <= lo) continue;
		const uint64_t len = plan->off[c + 1] - plan->off[c];
		if (pos[lo - origin] < 1u) *bad = std::min(*bad, lo);
		else if (pos[hi - 1 - origin] > len) *bad = std::min(*bad, hi - 1);
	}
}
static int bp_position_error(uint64_t bad) {
	return pgt_set_error(PGT_ERR_INPUT, "site " + std::to_string(bad) + " lies outside its chromosome (bp positions run from 1 to the chromosome length)");
}

// ---- PGT_MEM_DEVICE: the columns are read in place
template <class Stat>
static int scan_device(const Scan& s) {
	const pgt_plan* plan = s.plan;
	const Layout& L = s.L;
	DevPlan P = s.P;
	const uint64_t nunits = L.u_hi - L.u_lo;
	const uint64_t nwin = L.w_hi - L.w_lo;
	double* gpart = (double*)(s.ws + L.gpart_off);
	if (L.path != PGT_PATH_UNITS) {
		// windows straight from the sites: W = S = 1 (default arguments of fstWindow / hetWindow: an
		// elementwise map) or the sliding tile for fine steps; no unit array, no level 2
		bool global_done = false;
		if (nwin) {
			uint64_t first_site, last_site;
			pgt_plan_window(plan, L.w_lo, &first_site, nullptr, nullptr);
			pgt_plan_window(plan, L.w_hi - 1, nullptr, &last_site, nullptr);
			P.col_elems = last_site + 1 - L.origin;
			if (L.path == PGT_PATH_PERSITE) {
				// the windows ARE the sites: when the owned range of the global line is exactly their span (always, unless the
				// scan owns sites outside any window) the kernel adds its sites up on the way and the dxy columns are read once
				global_done = s.want_global && GlobalTerm<Stat>::has && L.gsite_lo == first_site && L.gsite_hi == last_site + 1;
				PGT_TRY(launch_persite<Stat>(plan, P, s.C, rows_of<Stat>(s), global_done ? gpart : nullptr, s.out->dxy_global, s.st));
			} else if constexpr (!IsXStat<Stat>::value) {
				global_done = s.want_global && GlobalTerm<Stat>::has && g_tune_slideglobal != 1 && slide_runs_cover_owned_sites(plan, L);
				PGT_TRY(launch_slide<Stat>(plan, L.slide, P, s.C, last_site + 1 - L.origin, s.C.pos, *s.out, global_done ? gpart : nullptr,
				                           s.out->dxy_global, s.st));
			}
		}
		if (s.want_global && !global_done) {
			if (L.gsite_lo < L.origin) return pgt_set_error(PGT_ERR_ARGS, "site_origin lies after the first site this scan must read");
			PGT_TRY(launch_global_sites(s.C, L.gsite_lo - L.origin, L.gsite_hi - L.origin, gpart, s.out->dxy_global, s.st));
		}
		return PGT_OK;
	}
	unsigned long long* bad = nullptr;  // the extreme scan of a bp plan checks the positions (read back at the end)
	if (IsXStat<Stat>::value && s.bp) {
		bad = (unsigned long long*)(s.ws + L.flag_off);
		PGT_CUDA(cudaMemsetAsync(bad, 0xff, sizeof(*bad), s.st));
		DevPlan Pc = P;
		Pc.col_elems = s.ndata;
		k_bp_pos_check<<<capped_grid((P.ncontig + 255) / 256), 256, 0, s.st>>>(Pc, s.C.pos, s.ndata, bad);
		g_launches++;
		PGT_CUDA(cudaGetLastError());
	}
	if (s.bp && nunits) PGT_TRY(launch_bounds_kernel(P, s.C.pos, s.ndata, s.bounds, s.st));
	if (L.unit_table) {  // very many segments: unit starts once, then the INDIRECT level-1 kernels
		k_unit_starts<<<capped_grid((nunits + 256) / 256), 256, 0, s.st>>>(P, s.bounds);
		g_launches++;
		PGT_CUDA(cudaGetLastError());
	}
	// elements the caller's columns are known to hold: up to the end of the last unit read
	P.col_elems = s.bp ? s.ndata : pgt_plan_unit_start(plan, L.u_hi) - L.origin;
	typename Stat::Acc* units = (typename Stat::Acc*)(s.ws + L.units_off);
	PGT_TRY(launch_units<Stat>(P, s.C, units, s.bounds, P.col_elems, L.tileseg_cap ? (uint32_t*)(s.ws + L.tileseg_off) : nullptr,
	                           L.tileseg_cap, s.st));
	// the global line reads the raw unit partials: before level 2, which may scan them in place
	if (s.want_global) PGT_TRY(launch_global<Stat>(units, s.nglobal, gpart, s.out->dxy_global, s.st));
	PGT_TRY(launch_windows<Stat>(P, units, L.u_lo, s.C.pos, rows_of<Stat>(s), L.hgw, (typename Stat::Acc*)(s.ws + L.pre_off), L.blk_lo, L.blk_hi, s.st));
	if (bad) {
		unsigned long long h = 0;
		PGT_CUDA(cudaMemcpyAsync(&h, bad, sizeof(h), cudaMemcpyDeviceToHost, s.st));
		PGT_CUDA(cudaStreamSynchronize(s.st));
		if (h != ~0ull) return bp_position_error(h);
	}
	return PGT_OK;
}

// ---- PGT_MEM_HOST: slabs of the axis are staged H2D on a copy stream (double-buffered) while the previous slab is
// reduced; only unit partials stay on the device.  Positions are not copied in site mode: the two edge positions per
// window are gathered on the host.
struct HostStaging {
	cudaStream_t copy = nullptr;
	cudaEvent_t ready[2] = {nullptr, nullptr};  // slot filled (copy stream)
	cudaEvent_t freed[2] = {nullptr, nullptr};  // slot read by its kernels (`st`)
	char* buf[2][8];                            // per slot, per column of `cd`
	ColDesc cd[8];
	int ncol = 0;
	int slot = 0;
	bool used[2] = {false, false};
	~HostStaging() {
		for (int i = 0; i < 2; ++i) {
			if (ready[i]) cudaEventDestroy(ready[i]);
			if (freed[i]) cudaEventDestroy(freed[i]);
		}
		if (copy) cudaStreamDestroy(copy);
	}
	// H2D of sites [s0, s0 + ns) of every column into the current slot, ordered after the kernels that last read it
	int stage(const Scan& s, uint64_t s0, uint64_t ns, Cols* C) {
		if (used[slot]) PGT_CUDA(cudaStreamWaitEvent(copy, freed[slot], 0));
		*C = Cols{};
		C->minind = s.C.minind;
		C->cutoff = s.C.cutoff;
		for (int i = 0; i < ncol; ++i) {
			const char* src = (const char*)col_ptr(s.C, cd[i]) + (s0 - s.L.origin) * cd[i].elem;
			if (ns) PGT_CUDA(cudaMemcpyAsync(buf[slot][i], src, ns * cd[i].elem, cudaMemcpyHostToDevice, copy));
			set_col_ptr(C, cd[i], buf[slot][i]);
		}
		PGT_CUDA(cudaEventRecord(ready[slot], copy));
		PGT_CUDA(cudaStreamWaitEvent(s.st, ready[slot], 0));
		return PGT_OK;
	}
	// the kernels enqueued on `st` since stage() are the last to read the slot; the next slab takes the other one
	int release(cudaStream_t st) {
		PGT_CUDA(cudaEventRecord(freed[slot], st));
		used[slot] = true;
		slot ^= 1;
		return PGT_OK;
	}
};

// Window bookkeeping on the host -- label, nsites, the two edge positions per window -- runs on worker threads next to
// the copy pipeline.  (It cannot simply follow the slab loop: enqueueing ~10 operations per slab blocks once the
// driver's queue is full, so the host would only get to it when most of the transfer is over; 3e7 windows take ~1 s on
// one thread.)
struct Bookkeeper {
	std::vector<std::thread> th;
	void join() {
		for (auto& t : th)
			if (t.joinable()) t.join();
	}
	~Bookkeeper() { join(); }
};
static void start_bookkeeping(const Scan& s, Bookkeeper* book) {
	const pgt_windows* out = s.out;
	const uint64_t nwin = s.L.w_hi - s.L.w_lo;
	if (!nwin || !(out->label || out->nsites || out->start_pos || out->end_pos || out->mid_pos)) return;
	unsigned nt = nwin < (1u << 16) ? 1u : std::min<unsigned>(8u, std::max(1u, std::thread::hardware_concurrency()));
	const uint64_t per = (nwin + nt - 1) / nt;
	for (unsigned t = 0; t < nt; ++t) {
		const uint64_t wa = s.L.w_lo + per * t, wb = std::min<uint64_t>(s.L.w_hi, wa + per);
		if (wa >= wb) break;
		book->th.emplace_back([plan = s.plan, out, pos = s.C.pos, bp = s.bp, wa, wb, origin = s.L.origin, w_lo = s.L.w_lo]() {
			uint32_t si = pgt_plan_seg_of_window(plan, wa);
			for (uint64_t w = wa; w < wb; ++w) {
				while (w >= plan->segs[si].win_base + plan->segs[si].nwin) ++si;
				const pgt_seg& sg = plan->segs[si];
				uint64_t fs;
				const uint32_t n = pgt_window_sites(plan->g, sg, w - sg.win_base, &fs);
				const uint64_t first = sg.site_base + fs, last = first + n - 1;
				const uint32_t label = pgt_plan_contig_of(plan, last);
				const uint64_t o = w - w_lo;
				if (out->label) out->label[o] = label;
				if (out->nsites) out->nsites[o] = n;
				uint32_t sp = 0, ep = 0;
				bool have = false;
				if (bp) {
					sp = (uint32_t)(first - plan->off[pgt_plan_contig_of(plan, first)]) + 1u;
					ep = (uint32_t)(last - plan->off[label]) + 1u;
					have = true;
				} else if (pos) {
					sp = pos[first - origin];
					ep = pos[last - origin];
					have = true;
				}
				if (have) {
					if (out->start_pos) out->start_pos[o] = sp;
					if (out->end_pos) out->end_pos[o] = ep;
					if (out->mid_pos) out->mid_pos[o] = (sp + ep) / 2u;
				}
			}
		});
	}
}

// the values of extreme-score rows the window kernels write on the device (ext_value, ext_pos: gathered on the host from
// ext_site), member by member
template <class F, class... T>
static void for_each_xrow_value(F&& fn, T&... t) {
	fn(t.ext_site...), fn(t.prop...), fn(t.nbig...), fn(t.xnsites...);
}

// Per-window values are produced into device tables, then copied back: one table for the whole scan, or -- when the
// windows come straight from the sites, slab by slab -- two slab-sized tables used in turn.  A table has 12 slots:
// the nine values in slots 0-8 (the extreme scan: for_each_xrow_value), the global triple in slot 11.  `host` are the
// caller's rows the table is copied back to (the extreme scan: ext_site also when only ext_value / ext_pos are wanted).
template <class Out>
static Out device_table(const Scan& s, const Out& host, int which) {
	const uint64_t rows = s.L.path == PGT_PATH_UNITS ? s.L.w_hi - s.L.w_lo : s.L.out_slab_rows;
	const size_t ob = align_up((size_t)rows * 8 + 8, 256);
	char* t = s.ws + s.L.outs_off + (size_t)which * 12 * ob;
	Out d;
	memset(&d, 0, sizeof(d));
	int k = 0;
	auto slot = [&](auto*& dp, auto* want) {
		if (want) dp = (decltype(want))(t + ob * k);
		++k;
	};
	if constexpr (std::is_same<Out, XRows>::value) {
		for_each_xrow_value(slot, d, host);
	} else {
		for_each_value(slot, d, host);
		d.dxy_global = s.want_global ? (double*)(t + ob * 11) : nullptr;
	}
	return d;
}
// rows [row0, row0 + n) of the caller's arrays <- rows [0, n) of a device table, on `st`
template <class Out>
static int copy_back(const Scan& s, const Out& host, const Out& d, uint64_t row0, uint64_t n) {
	cudaError_t e = cudaSuccess;
	auto back = [&](auto* h, auto* dp) {
		if (e == cudaSuccess && h && dp && n) e = cudaMemcpyAsync(h + row0, dp, n * sizeof(*h), cudaMemcpyDeviceToHost, s.st);
	};
	if constexpr (std::is_same<Out, XRows>::value) for_each_xrow_value(back, host, d);
	else for_each_value(back, host, d);
	if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(window table -> host)");
	return PGT_OK;
}

// Windows straight from the sites (sliding tile / W = S = 1): slabs of consecutive WINDOWS; a slab holds the sites of
// its windows, neighbours share the W - S sites of the overlap.  The global line is taken from the same staged sites:
// every slab folds the part of the owned range [gsite_lo, gsite_hi) that no earlier slab has folded, one partial
// triple per slab, added in slab order on the host.
template <class Stat>
static int host_window_slabs(const Scan& s, HostStaging& hs, const typename Stat::Out& host) {
	const pgt_plan* plan = s.plan;
	const Layout& L = s.L;
	const uint64_t slab_target = L.slab_sites - kSlabSlack;
	double* gslab = (double*)(s.ws + L.gslab_off);
	uint64_t ngslab = 0, gcursor = L.gsite_lo;
	auto fold_global = [&](const Cols& C, uint64_t s0, uint64_t s1) -> int {  // owned sites inside the staged [s0, s1)
		const uint64_t a = std::max(gcursor, s0), b = std::min(L.gsite_hi, s1);
		if (!s.want_global || b <= a) return PGT_OK;
		if (ngslab >= L.gslab_cap) return pgt_set_error(PGT_ERR_NOMEM, "internal: global-line slab table too small");
		PGT_TRY(launch_global_sites(C, a - s0, b - s0, (double*)(s.ws + L.gpart_off), gslab + 3 * ngslab, s.st));
		++ngslab;
		gcursor = b;
		return PGT_OK;
	};
	uint64_t w = L.w_lo;
	while (w < L.w_hi) {
		uint64_t fs, last;
		pgt_plan_window(plan, w, &fs, nullptr, nullptr);
		const uint64_t wb = pgt_plan_windows_within(plan, w, std::min<uint64_t>(L.w_hi, w + L.out_slab_rows), fs + slab_target);
		pgt_plan_window(plan, wb - 1, nullptr, &last, nullptr);
		// (in site mode no owned site precedes the scan's first window: only an EOF segment can lack windows)
		const uint64_t s0 = fs;
		const uint64_t ns = last + 1 - s0;
		if (ns > L.slab_sites) return pgt_set_error(PGT_ERR_ARGS, "internal: window slab larger than the staging buffers");
		Cols C;
		PGT_TRY(hs.stage(s, s0, ns, &C));
		DevPlan Ps = s.P;
		Ps.win_lo = w;
		Ps.win_hi = wb;
		Ps.site_origin = s0;
		Ps.col_elems = ns;
		const typename Stat::Out o = device_table(s, host, hs.slot);  // rewritten two slabs later, after this slab's copy-back (order of `st`)
		// (global line: fold_global below)
		if (L.path == PGT_PATH_PERSITE) PGT_TRY(launch_persite<Stat>(plan, Ps, C, o, nullptr, nullptr, s.st));
		else if constexpr (!IsXStat<Stat>::value) PGT_TRY(launch_slide<Stat>(plan, L.slide, Ps, C, ns, nullptr, o, nullptr, nullptr, s.st));
		PGT_TRY(fold_global(C, s0, s0 + ns));
		PGT_TRY(copy_back(s, host, o, w - L.w_lo, wb - w));
		PGT_TRY(hs.release(s.st));
		w = wb;
	}
	// owned sites after the last window (dropped EOF partial) or of a scan without windows
	while (s.want_global && gcursor < L.gsite_hi) {
		const uint64_t ns = std::min<uint64_t>(L.gsite_hi - gcursor, slab_target);
		const uint64_t s0 = gcursor;
		Cols C;
		PGT_TRY(hs.stage(s, s0, ns, &C));
		PGT_TRY(fold_global(C, s0, s0 + ns));
		PGT_TRY(hs.release(s.st));
	}
	if (s.want_global) {
		std::vector<double> part(3 * ngslab + 3, 0.0);
		if (ngslab) PGT_CUDA(cudaMemcpyAsync(part.data(), gslab, 3 * ngslab * sizeof(double), cudaMemcpyDeviceToHost, s.st));
		PGT_CUDA(cudaStreamSynchronize(s.st));
		double g3[3] = {0.0, 0.0, 0.0};
		for (uint64_t i = 0; i < ngslab; ++i)
			for (int q = 0; q < 3; ++q) g3[q] += part[3 * i + q];
		memcpy(s.out->dxy_global, g3, sizeof(g3));
	}
	return PGT_OK;
}

// Level 1 over slabs of consecutive UNITS into the unit array on the device.
template <class Stat>
static int host_unit_slabs(const Scan& s, HostStaging& hs, typename Stat::Acc* units) {
	const pgt_plan* plan = s.plan;
	const Layout& L = s.L;
	const uint64_t slab_target = L.slab_sites - kSlabSlack;
	const uint64_t axis_end = plan->off[0] + plan->nsites;
	uint64_t ua = L.u_lo;
	while (ua < L.u_hi) {
		const uint64_t e0 = pgt_plan_unit_start(plan, ua);
		uint64_t ub;
		if (e0 + slab_target >= axis_end) ub = L.u_hi;
		else ub = std::min<uint64_t>(L.u_hi, pgt_plan_unit_containing(plan, e0 + slab_target));
		if (ub <= ua) ub = ua + 1;
		const uint64_t e1 = pgt_plan_unit_start(plan, ub);
		uint64_t s0 = e0, s1 = e1;  // data-site range of this slab
		if (s.bp) {
			s0 = host_site_lower_bound(plan, s.site_offsets, s.C.pos, L.origin, s.ndata, e0);
			s1 = host_site_lower_bound(plan, s.site_offsets, s.C.pos, L.origin, s.ndata, e1);
		}
		const uint64_t ns = s1 - s0;
		if (ns > L.slab_sites) return pgt_set_error(PGT_ERR_INPUT, "bp mode: more sites than bp in a slab (positions not strictly increasing?)");
		Cols C;
		PGT_TRY(hs.stage(s, s0, ns, &C));
		DevPlan Ps = s.P;
		Ps.unit_lo = ua;
		Ps.unit_hi = ub;
		Ps.site_origin = s0;
		Ps.col_elems = ns;
		uint64_t* sb = s.bounds ? s.bounds + (ua - L.u_lo) : nullptr;
		// bp: bounds are relative to the staged slice.  Slab i writes entries [ua, ub]; the shared
		// entry ub is rewritten by slab i+1 relative to ITS slice, after slab i's unit kernel
		// (stream order on `st`).
		if (s.bp) PGT_TRY(launch_bounds_kernel(Ps, C.pos, ns, sb, s.st));
		PGT_TRY(launch_units<Stat>(Ps, C, units + (ua - L.u_lo), sb, ns, L.tileseg_cap ? (uint32_t*)(s.ws + L.tileseg_off) : nullptr,
		                           L.tileseg_cap, s.st));
		PGT_TRY(hs.release(s.st));
		ua = ub;
	}
	return PGT_OK;
}

template <class Stat>
static int scan_host(const Scan& s) {
	const Layout& L = s.L;
	HostStaging hs;
	PGT_CUDA(cudaStreamCreateWithFlags(&hs.copy, cudaStreamNonBlocking));
	for (int i = 0; i < 2; ++i) {
		PGT_CUDA(cudaEventCreateWithFlags(&hs.ready[i], cudaEventDisableTiming));
		PGT_CUDA(cudaEventCreateWithFlags(&hs.freed[i], cudaEventDisableTiming));
	}
	// the copy stream must not start before the caller's stream reaches this point
	PGT_CUDA(cudaEventRecord(hs.freed[0], s.st));
	PGT_CUDA(cudaStreamWaitEvent(hs.copy, hs.freed[0], 0));
	// the rows copied back; the extreme scan gathers ext_value and ext_pos on the host from ext_site (kept here if not wanted)
	typename Stat::Out host = rows_of<Stat>(s);
	std::vector<uint64_t> site_tmp;
	if constexpr (IsXStat<Stat>::value) {
		if (s.bp) {
			uint64_t bad = ~0ull;
			bp_check_positions_host(s.plan, s.site_offsets, s.C.pos, L.origin, s.ndata, &bad);
			if (bad != ~0ull) return bp_position_error(bad);
		}
		if ((host.ext_value || host.ext_pos) && !host.ext_site) {
			site_tmp.resize(L.w_hi - L.w_lo);
			host.ext_site = site_tmp.data();
		}
	}
	Bookkeeper book;
	start_bookkeeping(s, &book);
	hs.ncol = stat_columns(s.stat, s.plan->mode, hs.cd);
	size_t o = L.stage_off;
	for (int k = 0; k < 2; ++k)
		for (int i = 0; i < hs.ncol; ++i) {
			hs.buf[k][i] = s.ws + o;
			o += L.stage_col_bytes[i];
		}
	if (L.path != PGT_PATH_UNITS) {
		PGT_TRY(host_window_slabs<Stat>(s, hs, host));
	} else {
		typename Stat::Acc* units = (typename Stat::Acc*)(s.ws + L.units_off);
		PGT_TRY(host_unit_slabs<Stat>(s, hs, units));
		const typename Stat::Out dev = device_table(s, host, 0);
		if constexpr (!IsXStat<Stat>::value)
			if (s.want_global) PGT_TRY(launch_global<Stat>(units, s.nglobal, (double*)(s.ws + L.gpart_off), dev.dxy_global, s.st));
		PGT_TRY(launch_windows<Stat>(s.P, units, L.u_lo, nullptr, dev, L.hgw, (typename Stat::Acc*)(s.ws + L.pre_off), L.blk_lo, L.blk_hi, s.st));
		PGT_TRY(copy_back(s, host, dev, 0, L.w_hi - L.w_lo));
		if constexpr (!IsXStat<Stat>::value)
			if (s.want_global) PGT_CUDA(cudaMemcpyAsync(s.out->dxy_global, dev.dxy_global, 3 * sizeof(double), cudaMemcpyDeviceToHost, s.st));
	}
	book.join();
	PGT_CUDA(cudaStreamSynchronize(s.st));
	PGT_CUDA(cudaStreamSynchronize(hs.copy));
	if constexpr (IsXStat<Stat>::value) {
		const uint64_t nan_bits = 0xfff8000000000000ull;  // CUDART_NAN, the empty row's value on the device
		double empty_nan;
		memcpy(&empty_nan, &nan_bits, sizeof(empty_nan));
		// one random read per row and value: split over host threads as the bookkeeping (1e8 rows at W = S = 1)
		const uint64_t nwin = L.w_hi - L.w_lo;
		auto gather = [&host, &s, &L, empty_nan](uint64_t wa, uint64_t wb) {
			for (uint64_t w = wa; w < wb; ++w) {
				const bool empty = host.ext_site[w] == ~0ull;
				if (host.ext_value) host.ext_value[w] = empty ? empty_nan : s.C.score[host.ext_site[w] - L.origin];
				if (host.ext_pos) host.ext_pos[w] = empty ? 0u : s.C.pos[host.ext_site[w] - L.origin];
			}
		};
		if (host.ext_site && (host.ext_value || host.ext_pos)) {
			const unsigned nt = nwin < (1u << 16) ? 1u : std::min<unsigned>(8u, std::max(1u, std::thread::hardware_concurrency()));
			const uint64_t per = (nwin + nt - 1) / nt;
			std::vector<std::thread> th;
			for (unsigned t = 1; t < nt; ++t)
				if (per * t < nwin) th.emplace_back(gather, per * t, std::min<uint64_t>(nwin, per * (t + 1)));
			gather(0, std::min<uint64_t>(nwin, per));
			for (auto& t : th) t.join();
		}
	}
	return PGT_OK;
}

// The device view of a plan whose tables were uploaded to `segs` / `off` of a workspace (or are resident: bound), with
// bp mode's site offsets at `site_off`; the unit, window and site ranges are the caller's to set.
static DevPlan dev_plan(const pgt_plan* plan, const char* segs, const char* off, const char* site_off) {
	DevPlan P;
	memset(&P, 0, sizeof(P));
	const bool resident = plan->d_tables != nullptr;
	P.g = plan->g;
	P.segs = resident ? (const pgt_seg*)plan->d_tables : (const pgt_seg*)segs;
	P.off = resident ? (const uint64_t*)(plan->d_tables + align_up(plan->segs.size() * sizeof(pgt_seg), 256)) : (const uint64_t*)off;
	P.site_off = (const uint64_t*)site_off;
	P.nseg = (uint32_t)plan->segs.size();
	P.ncontig = (uint32_t)plan->off.size() - 1;
	P.nunits_total = plan->nunits;
	P.col_elems = ~0ull;
	P.mode = (int)plan->mode;
	return P;
}

// xrows: the extreme scan's rows (then `out` holds its geometry rows), else NULL
template <class Stat>
static int run_scan(const pgt_plan* plan, const pgt_range* range, pgt_stat stat, const Cols& C, const uint64_t* site_offsets,
                    const pgt_windows* out, const XRows* xrows, void* workspace, size_t workspace_bytes, pgt_mem mem, cudaStream_t st) {
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
		return pgt_set_error(PGT_ERR_CUDA, "no usable CUDA device (libpgtscan has no CPU fallback)");
	Scan s;
	Layout& L = s.L;
	PGT_TRY(make_layout(plan, range, stat, mem, &L));
	if (!workspace) return pgt_set_error(PGT_ERR_ARGS, "workspace is NULL");
	if (workspace_bytes < L.total) return pgt_set_error(PGT_ERR_NOMEM, "workspace too small, see pgt_scan_workspace_bytes");
	const bool bp = plan->mode == PGT_MODE_BP;
	if (bp && (!site_offsets || !C.pos)) return pgt_set_error(PGT_ERR_ARGS, "bp mode needs site_offsets and pos");
	const uint64_t nunits = L.u_hi - L.u_lo;
	if (nunits == 0 && L.w_hi == L.w_lo) return PGT_OK;  // empty input / empty shard: nothing to read or write
	ColDesc cd[8];
	const int ncol = stat_columns(stat, plan->mode, cd);
	for (int i = 0; i < ncol; ++i)
		if (!col_ptr(C, cd[i])) return pgt_set_error(PGT_ERR_ARGS, "a column required by this statistic is NULL");
	if (!bp && nunits > 0 && pgt_plan_unit_start(plan, L.u_lo) < L.origin)
		return pgt_set_error(PGT_ERR_ARGS, "site_origin lies after the first site this scan must read");

	char* ws = (char*)workspace;
	const size_t seg_bytes = plan->segs.size() * sizeof(pgt_seg);
	const size_t off_bytes = plan->off.size() * sizeof(uint64_t);
	const bool resident = plan->d_tables != nullptr;  // pgt_plan_bind_device: nothing to upload (and graph-capturable)
	if (!resident) {
		if (seg_bytes) PGT_CUDA(cudaMemcpyAsync(ws + L.segs_off, plan->segs.data(), seg_bytes, cudaMemcpyHostToDevice, st));
		PGT_CUDA(cudaMemcpyAsync(ws + L.off_off, plan->off.data(), off_bytes, cudaMemcpyHostToDevice, st));
	}
	if (bp) PGT_CUDA(cudaMemcpyAsync(ws + L.siteoff_off, site_offsets, off_bytes, cudaMemcpyHostToDevice, st));

	DevPlan& P = s.P;
	P = dev_plan(plan, ws + L.segs_off, ws + L.off_off, bp ? ws + L.siteoff_off : nullptr);
	P.unit_lo = L.u_lo;
	P.unit_hi = L.u_hi;
	P.win_lo = L.w_lo;
	P.win_hi = L.w_hi;
	P.site_origin = L.origin;

	s.ndata = 0;
	if (bp) {
		if (site_offsets[P.ncontig] < L.origin) return pgt_set_error(PGT_ERR_ARGS, "site_origin beyond the last site");
		s.ndata = (range && range->site_count) ? range->site_count : site_offsets[P.ncontig] - L.origin;
	}
	s.plan = plan;
	s.stat = stat;
	s.C = C;
	s.site_offsets = site_offsets;
	s.out = out;
	memset(&s.x, 0, sizeof(s.x));
	if (xrows) {
		s.x = *xrows;
		s.x.site_origin = L.origin;
	}
	s.ws = ws;
	s.bounds = (bp || L.unit_table) ? (uint64_t*)(ws + L.bounds_off) : nullptr;
	s.nglobal = L.g_hi > L.u_lo ? L.g_hi - L.u_lo : 0;
	s.bp = bp;
	s.want_global = out->dxy_global && (stat == PGT_STAT_DXY || stat == PGT_STAT_FUSED);
	s.st = st;
	return mem == PGT_MEM_DEVICE ? scan_device<Stat>(s) : scan_host<Stat>(s);
}

extern "C" int pgt_scan(const pgt_plan* plan, const pgt_range* range, pgt_stat stat, const pgt_columns* cols, int minind,
                        const uint64_t* site_offsets, const pgt_windows* out, void* workspace, size_t workspace_bytes, pgt_mem mem,
                        void* stream) {
	if (!plan || !cols || !out) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan: plan, cols and out must not be NULL");
	if (mem != PGT_MEM_DEVICE && mem != PGT_MEM_HOST) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan: unknown memory space");
	cudaStream_t st = (cudaStream_t)stream;
	switch (stat) {
		case PGT_STAT_FST: return run_scan<FstStat>(plan, range, stat, cols_from(*cols, minind), site_offsets, out, nullptr, workspace, workspace_bytes, mem, st);
		case PGT_STAT_HET: return run_scan<HetStat>(plan, range, stat, cols_from(*cols, minind), site_offsets, out, nullptr, workspace, workspace_bytes, mem, st);
		case PGT_STAT_DXY:
			if (minind < 1) return pgt_set_error(PGT_ERR_ARGS, "-minind must be at least 1");
			return run_scan<DxyStat>(plan, range, stat, cols_from(*cols, minind), site_offsets, out, nullptr, workspace, workspace_bytes, mem, st);
		case PGT_STAT_FUSED:
			if (minind < 1) return pgt_set_error(PGT_ERR_ARGS, "-minind must be at least 1");
			return run_scan<FusedStat>(plan, range, stat, cols_from(*cols, minind), site_offsets, out, nullptr, workspace, workspace_bytes, mem, st);
	}
	return pgt_set_error(PGT_ERR_ARGS, "pgt_scan: unknown statistic");
}

extern "C" int pgt_scan_fst(const pgt_plan* plan, const pgt_range* range, const pgt_columns* cols, const pgt_windows* out,
                            void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream) {
	return pgt_scan(plan, range, PGT_STAT_FST, cols, 1, nullptr, out, workspace, workspace_bytes, mem, stream);
}
extern "C" int pgt_scan_het(const pgt_plan* plan, const pgt_range* range, const pgt_columns* cols, const pgt_windows* out,
                            void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream) {
	return pgt_scan(plan, range, PGT_STAT_HET, cols, 1, nullptr, out, workspace, workspace_bytes, mem, stream);
}
extern "C" int pgt_scan_dxy(const pgt_plan* plan, const pgt_range* range, const pgt_columns* cols, int minind,
                            const uint64_t* site_offsets, const pgt_windows* out, void* workspace, size_t workspace_bytes, pgt_mem mem,
                            void* stream) {
	return pgt_scan(plan, range, PGT_STAT_DXY, cols, minind, site_offsets, out, workspace, workspace_bytes, mem, stream);
}
extern "C" int pgt_scan_fused(const pgt_plan* plan, const pgt_range* range, const pgt_columns* cols, int minind,
                              const pgt_windows* out, void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream) {
	return pgt_scan(plan, range, PGT_STAT_FUSED, cols, minind, nullptr, out, workspace, workspace_bytes, mem, stream);
}

// ---- sites per bp window (pgt_scan_bp_sites): plan tables and bp site offsets in the workspace, one 8-byte slot for the
// position check, and in host mode the positions of the chromosomes the windows touch plus the staged counts.
struct BpSitesLayout {
	uint64_t w_lo, w_hi, origin, ndata;
	uint64_t s_lo, s_hi;  // host mode: global sites staged
	size_t segs_off, off_off, siteoff_off, flag_off, pos_off, rows_off, total;
};

static int bp_sites_layout(const pgt_plan* plan, const pgt_range* range, const uint64_t* site_offsets, pgt_mem mem, BpSitesLayout* L) {
	if (!plan) return pgt_set_error(PGT_ERR_ARGS, "plan is NULL");
	if (plan->mode != PGT_MODE_BP) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_bp_sites needs a PGT_MODE_BP plan");
	if (mem != PGT_MEM_DEVICE && mem != PGT_MEM_HOST) return pgt_set_error(PGT_ERR_ARGS, "unknown memory space");
	memset(L, 0, sizeof(*L));
	L->w_hi = plan->nwin;
	if (range) {
		if (range->w_hi != 0 || range->w_lo != 0) {
			L->w_lo = range->w_lo;
			L->w_hi = range->w_hi;
		}
		L->origin = range->site_origin;
	}
	if (L->w_lo > L->w_hi || L->w_hi > plan->nwin) return pgt_set_error(PGT_ERR_ARGS, "window range out of bounds");
	const uint32_t nc = (uint32_t)plan->off.size() - 1;
	if (site_offsets) {
		if (site_offsets[nc] < L->origin) return pgt_set_error(PGT_ERR_ARGS, "site_origin beyond the last site");
		L->ndata = (range && range->site_count) ? range->site_count : site_offsets[nc] - L->origin;
	}
	const uint64_t nwin = L->w_hi - L->w_lo;
	if (mem == PGT_MEM_HOST && nwin) {
		if (!site_offsets) return pgt_set_error(PGT_ERR_ARGS, "host-memory pgt_scan_bp_sites needs site_offsets");
		uint64_t e0, e1;
		pgt_plan_window(plan, L->w_lo, &e0, nullptr, nullptr);
		pgt_plan_window(plan, L->w_hi - 1, nullptr, &e1, nullptr);
		L->s_lo = std::max(site_offsets[pgt_plan_contig_of(plan, e0)], L->origin);
		L->s_hi = std::max(L->s_lo, std::min(site_offsets[pgt_plan_contig_of(plan, e1) + 1], L->origin + L->ndata));
	}
	size_t o = 0;
	L->segs_off = o;
	o += align_up(plan->segs.size() * sizeof(pgt_seg) + 8, 256);
	L->off_off = o;
	o += align_up(plan->off.size() * sizeof(uint64_t), 256);
	L->siteoff_off = o;
	o += align_up(plan->off.size() * sizeof(uint64_t), 256);
	L->flag_off = o;
	o += 256;
	L->pos_off = o;
	if (mem == PGT_MEM_HOST) o += align_up((size_t)(L->s_hi - L->s_lo) * sizeof(uint32_t), 256);
	L->rows_off = o;
	if (mem == PGT_MEM_HOST) o += align_up((size_t)nwin * sizeof(uint32_t), 256);
	L->total = o + 256;
	return PGT_OK;
}

extern "C" size_t pgt_scan_bp_sites_workspace_bytes(const pgt_plan* plan, const pgt_range* range, const uint64_t* site_offsets, pgt_mem mem) {
	BpSitesLayout L;
	if (bp_sites_layout(plan, range, site_offsets, mem, &L) != PGT_OK) return 0;
	return L.total;
}

extern "C" int pgt_scan_bp_sites(const pgt_plan* plan, const pgt_range* range, const uint32_t* pos, const uint64_t* site_offsets,
                                 uint32_t* nsites_data, void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream) {
	if (!plan || !pos || !site_offsets || !nsites_data)
		return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_bp_sites: plan, pos, site_offsets and nsites_data must not be NULL");
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
		return pgt_set_error(PGT_ERR_CUDA, "no usable CUDA device (libpgtscan has no CPU fallback)");
	BpSitesLayout L;
	PGT_TRY(bp_sites_layout(plan, range, site_offsets, mem, &L));
	if (!workspace) return pgt_set_error(PGT_ERR_ARGS, "workspace is NULL");
	if (workspace_bytes < L.total) return pgt_set_error(PGT_ERR_NOMEM, "workspace too small, see pgt_scan_bp_sites_workspace_bytes");
	const uint64_t nwin = L.w_hi - L.w_lo;
	if (nwin == 0) return PGT_OK;
	cudaStream_t st = (cudaStream_t)stream;
	char* ws = (char*)workspace;
	const size_t seg_bytes = plan->segs.size() * sizeof(pgt_seg), off_bytes = plan->off.size() * sizeof(uint64_t);
	if (!plan->d_tables) {
		if (seg_bytes) PGT_CUDA(cudaMemcpyAsync(ws + L.segs_off, plan->segs.data(), seg_bytes, cudaMemcpyHostToDevice, st));
		PGT_CUDA(cudaMemcpyAsync(ws + L.off_off, plan->off.data(), off_bytes, cudaMemcpyHostToDevice, st));
	}
	PGT_CUDA(cudaMemcpyAsync(ws + L.siteoff_off, site_offsets, off_bytes, cudaMemcpyHostToDevice, st));
	unsigned long long* d_bad = (unsigned long long*)(ws + L.flag_off);
	PGT_CUDA(cudaMemsetAsync(d_bad, 0xff, sizeof(*d_bad), st));
	DevPlan P = dev_plan(plan, ws + L.segs_off, ws + L.off_off, ws + L.siteoff_off);
	P.win_lo = L.w_lo;
	P.win_hi = L.w_hi;
	const uint32_t* dpos = pos;
	uint32_t* drows = nsites_data;
	uint64_t ndata = L.ndata;
	P.site_origin = L.origin;
	if (mem == PGT_MEM_HOST) {  // the positions of the chromosomes the windows touch, staged once
		ndata = L.s_hi - L.s_lo;
		P.site_origin = L.s_lo;
		dpos = (const uint32_t*)(ws + L.pos_off);
		drows = (uint32_t*)(ws + L.rows_off);
		if (ndata) PGT_CUDA(cudaMemcpyAsync(ws + L.pos_off, pos + (L.s_lo - L.origin), ndata * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
	}
	P.col_elems = ndata;
	k_bp_sites<<<capped_grid((std::max<uint64_t>(nwin, P.ncontig) + 255) / 256), 256, 0, st>>>(P, dpos, ndata, drows, d_bad);
	g_launches++;
	PGT_CUDA(cudaGetLastError());
	if (mem == PGT_MEM_HOST) PGT_CUDA(cudaMemcpyAsync(nsites_data, drows, nwin * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
	unsigned long long bad = 0;
	PGT_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost, st));
	PGT_CUDA(cudaStreamSynchronize(st));
	if (bad != ~0ull)
		return pgt_set_error(PGT_ERR_INPUT, "site " + std::to_string(bad) + " lies outside its chromosome (bp positions run from 1 to the chromosome length)");
	return PGT_OK;
}

// ---- the extreme score over a window plan (pgt_scan_plan_extreme): the scan of pgt_scan with the statistic XStat
extern "C" size_t pgt_scan_plan_extreme_workspace_bytes(const pgt_plan* plan, const pgt_range* range, pgt_mem mem) {
	Layout L;
	if (make_layout(plan, range, kStatExtreme, mem, &L) != PGT_OK) return 0;
	return L.total;
}

extern "C" int pgt_scan_plan_extreme(const pgt_plan* plan, const pgt_range* range, pgt_xstat stat, double cutoff, const uint32_t* pos,
                                     const double* score, const uint64_t* site_offsets, const pgt_windows* rows, const pgt_xwindows* out,
                                     void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream) {
	if (!plan || !out) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme: plan and out must not be NULL");
	if (stat != PGT_XSTAT_IHS && stat != PGT_XSTAT_XPEHH) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme: unknown statistic");
	if (mem != PGT_MEM_DEVICE && mem != PGT_MEM_HOST) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme: unknown memory space");
	if (!score) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme: score column is NULL");
	pgt_windows geo;
	memset(&geo, 0, sizeof(geo));
	if (rows) {
		bool other = rows->dxy_global != nullptr;
		for_each_value([&](const void* p) { other = other || p; }, *rows);
		if (other) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme: rows may only ask for label, start_pos, end_pos, mid_pos and nsites");
		geo = *rows;
	}
	if (!pos && (plan->mode == PGT_MODE_BP || out->ext_pos || geo.start_pos || geo.end_pos || geo.mid_pos))
		return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme: pos is required in bp mode and for ext_pos, start_pos, end_pos and mid_pos");
	Cols C;
	memset(&C, 0, sizeof(C));
	C.pos = pos;
	C.score = score;
	C.minind = 1;
	C.cutoff = cutoff;
	XRows x{geo.label, geo.start_pos, geo.end_pos, geo.mid_pos, geo.nsites, out->ext_value, out->ext_pos, out->ext_site, out->nbig, out->nsites,
	        out->prop, score, pos, 0};
	cudaStream_t st = (cudaStream_t)stream;
	if (stat == PGT_XSTAT_IHS) return run_scan<XStat<XMODE_ABS>>(plan, range, kStatExtreme, C, site_offsets, &geo, &x, workspace, workspace_bytes, mem, st);
	if (cutoff < 0) return run_scan<XStat<XMODE_MIN>>(plan, range, kStatExtreme, C, site_offsets, &geo, &x, workspace, workspace_bytes, mem, st);
	return run_scan<XStat<XMODE_MAX>>(plan, range, kStatExtreme, C, site_offsets, &geo, &x, workspace, workspace_bytes, mem, st);
}
