// pgt_internal.h -- shared between the host planner (pgt_plan.cpp) and the CUDA side (pgt_scan.cu).
#ifndef PGT_INTERNAL_H
#define PGT_INTERNAL_H

#include <string>
#include <vector>

#include "../../include/pgt_extreme.h"
#include "../../include/pgt_scan.h"
#include "pgt_geom.h"

struct pgt_plan {
	pgt_mode mode;
	pgt_geom g;
	std::vector<uint64_t> off;  // contig offsets, ncontig+1
	std::vector<pgt_seg> segs;
	uint64_t nwin;
	uint64_t nunits;
	uint64_t nsites;
	uint64_t nblocks;  // scan blocks of g.wunits units over all segments
	uint64_t window_units_total;  // unit partials a direct level 2 reads over all windows (short segments have short windows)
	uint64_t scan_units_total;    // units the block scans of scan mode touch (whole blocks, at least one per segment)
	// optional caller-owned device copy of segs | off (pgt_plan_bind_device); nullptr = upload per scan
	unsigned char* d_tables = nullptr;
};

int pgt_set_error(int code, const std::string& msg);

// shared by the .cu files: launch counter and the optional per-kernel event timing (pgt_scan.cu)
void pgt_count_launch();
bool pgt_profile_enabled();
void pgt_profile_push(int kind, void* ev_a, void* ev_b);  // cudaEvent_t pair, recorded by the caller

// segment index containing global window w / global unit j / global site x
uint32_t pgt_plan_seg_of_window(const pgt_plan* p, uint64_t w);
uint32_t pgt_plan_seg_of_unit(const pgt_plan* p, uint64_t j);
// global index of the unit containing global site/entry x (x inside the axis)
uint64_t pgt_plan_unit_containing(const pgt_plan* p, uint64_t x);
// global site/entry index where global unit j starts; j == nunits gives the end of the axis
uint64_t pgt_plan_unit_start(const pgt_plan* p, uint64_t j);
// largest wb in (w, w_hi] such that all windows [w, wb) end at or before global site `limit` (>= w + 1)
uint64_t pgt_plan_windows_within(const pgt_plan* p, uint64_t w, uint64_t w_hi, uint64_t limit);
// contig c with off[c] <= x < off[c+1]
uint32_t pgt_plan_contig_of(const pgt_plan* p, uint64_t x);

// The per-window arrays of one or more result tables, member by member: fn(a.sum_a, b.sum_a), fn(a.sum_b, b.sum_b), ...
// for_each_value visits the nine values the window kernels write, in the order of the slots of a host-mode output
// table; for_each_field visits all fourteen arrays.  (dxy_global is one triple per scan, not a per-window array.)
template <class F, class... T>
void for_each_value(F&& fn, T&... t) {
	fn(t.sum_a...), fn(t.sum_b...), fn(t.fst...), fn(t.nhet...), fn(t.nonmissing...), fn(t.het...), fn(t.dxy...), fn(t.neffective...),
	    fn(t.nskip...);
}
template <class F, class... T>
void for_each_field(F&& fn, T&... t) {
	fn(t.label...), fn(t.start_pos...), fn(t.end_pos...), fn(t.mid_pos...), fn(t.nsites...);
	for_each_value(fn, t...);
}
// the same for extreme-score tables, in the order of the host-mode staging blocks; ext_pos last (host-memory scans
// gather it on the host)
template <class F, class... T>
void for_each_xfield(F&& fn, T&... t) {
	fn(t.ext_value...), fn(t.ext_site...), fn(t.prop...), fn(t.nbig...), fn(t.nsites...), fn(t.ext_pos...);
}

#endif
