/*
 * pgt_extreme.h -- C ABI of libpgtscan.so, part 2: bp-window "most extreme score" scans.
 *
 * Drop-in boundary for the hot path of tplinderoth/PopGenomicsTools' ihsWindow and xpehhWindow
 * (SURVEY.md §8f rank 3).  The reference has no library API; its line loops
 *
 *     calciHSWindows     /root/reference/ihsWindow.cpp:93-187    (+ updateMax :69-73, printWindow :75-84)
 *     calcXpehhWindows   /root/reference/xpehhWindow.cpp:87-193  (+ updateOutlier :59-63)
 *
 * interleave two things that this ABI separates:
 *
 *   pgt_xplan_*        "which windows get a row, and which sites does each hold": the flush /
 *                      empty-window / -chrlen padding bookkeeping of ihsWindow.cpp:130-157,179-186.
 *                      Host, one integer pass over the positions, bit-exact incl. the quirks
 *                      listed in oracle/pgt_oracle_extreme.c.  Windows are contiguous site ranges
 *                      in file order, non-overlapping, possibly empty.
 *   pgt_scan_extreme   the per-site statistic (|iHS|, or +-XPEHH, and the cutoff test) fused with
 *                      the segmented window reduction (first arg-extreme, count above cutoff):
 *                      CUDA, every site's score is read from HBM once (8 B/site).
 *
 * Same conventions as pgt_scan.h: plain C types, 0 / negative pgt_status + pgt_last_error(),
 * caller-owned buffers, no CPU fallback, `stream` = cudaStream_t as void*.
 */
#ifndef PGT_EXTREME_H
#define PGT_EXTREME_H

#include "pgt_scan.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pgt_xplan pgt_xplan; /* opaque: window table (CSR over sites) + reduction units */

typedef enum {
	/* ihsWindow: most extreme |score| (the signed score is reported), count |score| > cutoff
	 * (ihsWindow.cpp:160-173) */
	PGT_XSTAT_IHS = 0,
	/* xpehhWindow: cutoff < 0: minimum score, count score < cutoff; else maximum score, count
	 * score > cutoff (xpehhWindow.cpp:171-177) */
	PGT_XSTAT_XPEHH = 1
} pgt_xstat;

/* Window bookkeeping of one file (HOST memory, any thread count inside):
 *   pos[nsites]               physical position column (2nd field, ihsWindow.cpp:119), file order
 *   contig_offsets[ncontig+1] cumulative site counts of the runs of equal chromosome name
 *                             (the text before '_' in the locus id, extractChr ihsWindow.cpp:56-67)
 *   contig_len[ncontig]       -chrlen length of each run's name, 0 = not listed / no file
 *                             (lenmap lookups ihsWindow.cpp:125,139-141); NULL = all 0
 *   winsize                   -winsize in bp, >= 1
 *   unit_sites                cap on the reduction unit in sites (0 = default 2048); results do
 *                             not depend on it (max / argmax / counts are order-free)
 * Errors: PGT_ERR_INPUT when a site lies beyond its chromosome's -chrlen length (the reference
 * then prints empty windows forever, ihsWindow.cpp:151-156 with winend pinned at chrlen). */
int pgt_xplan_create(pgt_xplan** plan, const uint32_t* pos, const uint64_t* contig_offsets, const uint32_t* contig_len,
                     uint32_t ncontig, uint32_t winsize, uint32_t unit_sites);
void pgt_xplan_destroy(pgt_xplan* plan);

uint64_t pgt_xplan_num_windows(const pgt_xplan* plan); /* rows the reference prints */
uint64_t pgt_xplan_num_units(const pgt_xplan* plan);
uint64_t pgt_xplan_num_sites(const pgt_xplan* plan);

/* Window table, host arrays of pgt_xplan_num_windows elements (any pointer may be NULL):
 * label = contig run whose name is printed; start/end = printed window bounds (end < start for
 * the degenerate window a SNP on the last base opens); first_site/nsites = the sites it holds. */
int pgt_xplan_windows(const pgt_xplan* plan, uint32_t* label, uint32_t* start, uint32_t* end, uint64_t* first_site,
                      uint32_t* nsites);

/* Contiguous window ranges balanced by sites; shards are independent (windows do not overlap, so
 * there is no halo).  Returns [w_lo, w_hi) and the site range [site_lo, site_hi) they hold. */
int pgt_xplan_shard(const pgt_xplan* plan, uint32_t shard, uint32_t nshards, uint64_t* w_lo, uint64_t* w_hi,
                    uint64_t* site_lo, uint64_t* site_hi);

/* Optional: keep the window tables (16 B per window) resident on the device so that repeated
 * scans do not re-upload them.  `buffer` is caller-owned device memory of at least
 * pgt_xplan_device_bytes(); it must outlive the binding.  buffer = NULL unbinds.  A bound plan
 * may only be scanned on the device that owns the buffer. */
size_t pgt_xplan_device_bytes(const pgt_xplan* plan);
int pgt_xplan_bind_device(pgt_xplan* plan, void* buffer, size_t bytes, void* stream);

/* Per-window results, w_hi - w_lo elements each, any pointer may be NULL.  Empty windows (the
 * reference's "NA NA NA 0" rows, ihsWindow.cpp:82) get ext_value = prop = NaN, ext_pos = 0,
 * ext_site = UINT64_MAX, nbig = nsites = 0. */
typedef struct {
	double* ext_value;  /* printed score: maxihs[1] (ihsWindow.cpp:80) / outlierstat[0] (xpehhWindow.cpp:70) */
	uint32_t* ext_pos;  /* position of that site */
	uint64_t* ext_site; /* its global site index (first one on ties: strict comparisons, :166) */
	uint32_t* nbig;     /* sites beyond the cutoff */
	uint32_t* nsites;   /* sites in the window */
	double* prop;       /* (double)nbig / nsites (ihsWindow.cpp:79) */
} pgt_xwindows;

/* Device scratch for a scan over `range` (NULL = everything) with columns in `mem`. */
size_t pgt_scan_extreme_workspace_bytes(const pgt_xplan* plan, const pgt_range* range, pgt_mem mem);

/* The scan.  `score` is the normalised statistic column (field 7 of a selscan iHS .norm row,
 * sitevec[4] ihsWindow.cpp:160; field 9 of an XP-EHH .norm row, sitevec[6] xpehhWindow.cpp:165);
 * `pos` may be NULL when ext_pos is not requested.  Column pointers address element
 * range->site_origin of the global columns, as in pgt_scan(). */
int pgt_scan_extreme(const pgt_xplan* plan, const pgt_range* range, pgt_xstat stat, double cutoff, const uint32_t* pos,
                     const double* score, const pgt_xwindows* out, void* workspace, size_t workspace_bytes, pgt_mem mem,
                     void* stream);

/* One host column set, several GPUs of one process (see pgt_scan_sharded in pgt_scan.h): the window list is cut by
 * pgt_xplan_shard, shard i runs on devices[i] from its own host thread and writes its rows into `out` (host arrays of
 * pgt_xplan_num_windows elements) at its window offset.  `pos` / `score` are host columns over ALL sites.  Scratch is
 * allocated and freed by the call.  Results are bit-identical for any device list (the reduction is exact). */
int pgt_scan_extreme_sharded(const pgt_xplan* plan, pgt_xstat stat, double cutoff, const uint32_t* pos, const double* score,
                             const pgt_xwindows* out, const int* devices, uint32_t ndev);

/* ---- the same statistics over the windows of a pgt_plan (pgt_scan.h): sliding site or bp windows whose rows line up
 * row for row with pgt_scan's fst / het / dxy / fused rows of the same plan and range.
 *
 * Window w reduces the sites pgt_scan reduces for it: sites first..last in site mode; in bp mode the sites whose
 * positions fall on the window's bp (`site_offsets` = cumulative sites per chromosome, as for pgt_scan).  Per row:
 *   key       PGT_XSTAT_IHS |v|; PGT_XSTAT_XPEHH v (cutoff >= 0) or -v (cutoff < 0); a NaN key counts as -inf
 *   big       IHS |v| > cutoff; XPEHH v > cutoff, or v < cutoff when cutoff < 0 (strict; NaN is never big)
 *   ext_site  the smallest global site index among the window's sites of largest key (a non-empty window always
 *             has one, even when every score is NaN); ext_value = score[ext_site], ext_pos = pos[ext_site]
 *   nbig      big sites; nsites = the window's sites (in bp mode = pgt_scan_bp_sites); prop = nbig / nsites
 *   empty     (bp windows without sites) ext_value = prop = NaN, ext_pos = 0, ext_site = UINT64_MAX, nbig = nsites = 0
 * `rows` (may be NULL) receives the geometry pgt_scan writes for the same plan: only label, start_pos, end_pos,
 * mid_pos and nsites (bp: counts bp) may be set, anything else is PGT_ERR_ARGS.  These rows do not reproduce
 * ihsWindow's own window layout or its NaN-first-site quirk (that is pgt_scan_extreme).
 *
 * `range`, its site_origin / site_count, `site_offsets` and `mem` mean what they mean for pgt_scan; column pointers
 * address element range->site_origin.  `pos` is required in bp mode and for ext_pos, start_pos, end_pos and mid_pos.
 * Errors: those of pgt_scan, PGT_ERR_ARGS for an unknown `stat` or a NULL `score`, PGT_ERR_INPUT in bp mode when a
 * site lies outside its chromosome (a device-memory bp scan waits for its stream to report that).
 *
 * Kernel path (results do not depend on it): W = S = 1 in site mode maps every site to its row (one kernel); all
 * other plans take pgt_scan's units path -- level 1 per-unit extremes (direct or TMA-tiled, unit-start table, bp
 * unit bounds), level 2 warp / thread per window, or scan mode (block prefix / suffix, exact for a maximum) for
 * fine steps -- under the same pgt_tune knobs.  The sliding tile (PGT_PATH_SLIDE) is not used.  The level 1 / 2
 * timings appear under pgt_profile_read. */
size_t pgt_scan_plan_extreme_workspace_bytes(const pgt_plan* plan, const pgt_range* range, pgt_mem mem);
int pgt_scan_plan_extreme(const pgt_plan* plan, const pgt_range* range, pgt_xstat stat, double cutoff, const uint32_t* pos,
                          const double* score, const uint64_t* site_offsets, const pgt_windows* rows, const pgt_xwindows* out,
                          void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream);
/* Host columns over ALL sites, several GPUs of one process: windows cut by pgt_plan_shard, shard i on devices[i]
 * (see pgt_scan_sharded); scratch is allocated by the call; `rows` / `out` are host arrays of pgt_plan_num_windows
 * elements.  Bit-identical for any device list, a device listed more than once included. */
int pgt_scan_plan_extreme_sharded(const pgt_plan* plan, pgt_xstat stat, double cutoff, const uint32_t* pos, const double* score,
                                  const uint64_t* site_offsets, const pgt_windows* rows, const pgt_xwindows* out, const int* devices,
                                  uint32_t ndev);

/* Synthetic score column of global sites [site0, site0+n): ~N(0,1) with heavy ties removed
 * (counter-based, bit-identical to the CPU twin in pgt_synth.h).  Device pointer. */
int pgt_synth_score(uint64_t seed, uint64_t site0, uint64_t n, double* score, void* stream);

/* Per-kernel device timing of the extreme scan while pgt_profile(1) is on: level 1 = per-unit
 * reduction (reads the score column), level 2 = per-window combine.  Clears what it returns. */
int pgt_profile_read_extreme(double* units_ms, uint64_t* units_launches, double* windows_ms, uint64_t* windows_launches);

#ifdef __cplusplus
}
#endif
#endif /* PGT_EXTREME_H */
