/*
 * pgt_scan.h -- C ABI of libpgtscan.so: the B200 (sm_100a) windowed site-statistic scan.
 *
 * Drop-in boundary for the hot path of tplinderoth/PopGenomicsTools' fstWindow, hetWindow
 * and dxyWindow.  The reference has no library API; its only internal seam is
 *
 *     calcWindow(buffer*, chr*, winsize, step, nsites*[, skip_missing]) -> iterator
 *         /root/reference/fstWindow.cpp:69   (FST   = sum a / sum b over the buffered sites)
 *         /root/reference/hetWindow.cpp:66   (het   = #g==1 / #g>=0)
 *         /root/reference/dxyWindow.cpp:172  (dxy   = sum of per-site dxy, + neffective, nskip)
 *
 * driven by the flush triggers of calcFst / calcHeterozygosity / maf2dxy
 * (fstWindow.cpp:125-152, hetWindow.cpp:123-150, dxyWindow.cpp:334-426).  This ABI replaces
 * that pair -- "when does a window flush, over which sites, with which label" (pgt_plan_*,
 * closed form, host) and "reduce the window" (pgt_scan_*, CUDA) -- with one columnar call:
 *
 *     columns + contig offsets + (W, S, mode)  ->  per-window SoA result arrays
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success or a negative pgt_status,
 *     pgt_last_error() gives the message (thread-local).  The library never exits, never
 *     prints, and has no CPU fallback: without a usable CUDA device every pgt_scan_* /
 *     pgt_synth_* call fails with PGT_ERR_CUDA.
 *   - the caller owns all column, output and workspace buffers.  `mem` says where columns and
 *     outputs live: PGT_MEM_DEVICE (device pointers, work is enqueued on `stream` and not
 *     synchronised) or PGT_MEM_HOST (host pointers, pinned preferred; the call stages
 *     host->device->host through the workspace and returns after the results are on the host).
 *     The workspace is always device memory of at least pgt_scan_workspace_bytes().
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - 1 <= S <= W is required (the reference has undefined behaviour otherwise:
 *     heap corruption for S=0, segfault for S>W); violations return PGT_ERR_ARGS.
 */
#ifndef PGT_SCAN_H
#define PGT_SCAN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGT_ABI_VERSION 1

typedef enum {
	PGT_OK = 0,
	PGT_ERR_ARGS = -1,      /* invalid argument (message says which) */
	PGT_ERR_CUDA = -2,      /* CUDA runtime/driver error or no device */
	PGT_ERR_NOMEM = -3,     /* host allocation failed / workspace too small */
	PGT_ERR_INPUT = -4      /* input violates the format contract (e.g. unsorted positions in bp mode) */
} pgt_status;

typedef enum {
	PGT_MEM_DEVICE = 0,
	PGT_MEM_HOST = 1
} pgt_mem;

typedef enum {
	/* windows of W sites stepping S sites: fstWindow, hetWindow, dxyWindow -fixedsite 1
	 * (fstWindow.cpp:6-7, hetWindow.cpp:6-7, dxyWindow.cpp:357-359,376-378) */
	PGT_MODE_SITES = 0,
	/* windows of W bp stepping S bp over the dense per-bp entry stream of every chromosome:
	 * dxyWindow -fixedsite 0 (dxyWindow.cpp:336-355,363-373,407-426).  `contig_offsets` then
	 * holds cumulative chromosome LENGTHS IN BP (from -sizefile), not site counts.  Every
	 * statistic can be scanned over such a plan: the windows are the ones dxyWindow -fixedsite 0
	 * prints (its quirks included), so the tables of all statistics over one plan line up row for
	 * row, and a window reduces the sites whose positions fall on its bp (site i of chromosome c
	 * sits on entry contig_offsets[c] + pos[i] - 1; bp without a site contribute nothing).
	 * nsites then counts bp; pgt_scan_bp_sites gives the sites per window. */
	PGT_MODE_BP = 1
} pgt_mode;

typedef struct pgt_plan pgt_plan; /* opaque: closed-form window enumeration + reduction geometry */

/* ---- error / device ------------------------------------------------------------------ */
const char* pgt_last_error(void);
int pgt_abi_version(void);
int pgt_device_count(void);            /* >= 0, or PGT_ERR_CUDA */
int pgt_set_device(int device);

/* pinned host memory for PGT_MEM_HOST callers (cudaHostAlloc / cudaFreeHost) */
int pgt_host_alloc(void** p, size_t bytes);
int pgt_host_free(void* p);
/* page-lock / unlock an existing host allocation (cudaHostRegister) */
int pgt_host_register(void* p, size_t bytes);
int pgt_host_unregister(void* p);
/* device memory for the workspace of callers that do not link the CUDA runtime (the CLIs) */
int pgt_device_alloc(void** p, size_t bytes);
int pgt_device_free(void* p);

/* One process per GPU (SURVEY.md §8e): result tables shared inside a box.  The owner (rank 0) exports memory it got
 * from pgt_device_alloc as a 64-byte handle, the other processes map it (peer access over NVLink is enabled on
 * first use) and pass pointers into it as their pgt_windows arrays: every shard's window kernel then writes its
 * rows straight into the owner's table, and no gather step exists.  Close before the owner frees. */
#define PGT_IPC_HANDLE_BYTES 64
int pgt_ipc_export(const void* devptr, void* handle, size_t handle_bytes);
int pgt_ipc_open(const void* handle, void** devptr);
int pgt_ipc_close(void* devptr);

/* ---- plan: which windows exist (replaces the flush triggers of calcFst & co.) ----------
 *
 * contig_offsets[ncontig+1]: cumulative sizes, contig c spans [off[c], off[c+1]) in site
 * indices (PGT_MODE_SITES) or in entries = bp (PGT_MODE_BP).  Contigs are in file order;
 * adjacent lines with equal names form one contig, as in the reference (chr != oldchr).
 * unit_sites: cap on the reduction unit in sites (0 = default 256; a multiple of 32, <= 4096); part
 * of the summation order, see DESIGN.md "Summation order".  In PGT_MODE_BP the unit is a bp range: for
 * sparse data choose about 341 x (bp per site), capped at 4096 (what the dxyWindow CLI does).
 *
 * The enumeration reproduces, in closed form, the reference's behaviour incl. its quirks
 * (SURVEY.md Appendix A): trailing partial window at every contig change but at EOF only if
 * it holds > W-S sites; cross-contig carry when the buffer is exactly full at a contig
 * change; in bp mode the stale carry of chromosomes no longer than W-S.
 */
int pgt_plan_create(pgt_plan** plan, pgt_mode mode, const uint64_t* contig_offsets, uint32_t ncontig,
                    uint32_t W, uint32_t S, uint32_t unit_sites);
void pgt_plan_destroy(pgt_plan* plan);

uint64_t pgt_plan_num_windows(const pgt_plan* plan);
uint64_t pgt_plan_num_units(const pgt_plan* plan);
uint32_t pgt_plan_num_segments(const pgt_plan* plan);
uint64_t pgt_plan_num_sites(const pgt_plan* plan); /* off[ncontig] */

/* Host-side description of window w (tests, CLIs, sharding).  first/last are indices into the
 * site (or entry) axis, inclusive; label = contig index of the last site (the printed name). */
int pgt_plan_window(const pgt_plan* plan, uint64_t w, uint64_t* first, uint64_t* last, uint32_t* label);
/* Bulk variant: fills arrays of length pgt_plan_num_windows (any pointer may be NULL). */
int pgt_plan_windows(const pgt_plan* plan, uint64_t* first, uint64_t* last, uint32_t* label);
/* Reduction unit j: [start, start+len) on the site/entry axis (tests, DESIGN.md geometry). */
int pgt_plan_unit(const pgt_plan* plan, uint64_t j, uint64_t* start, uint32_t* len);
/* Units summed for window w: [first_unit, first_unit + count). */
int pgt_plan_window_units(const pgt_plan* plan, uint64_t w, uint64_t* first_unit, uint64_t* count);

/* Sharding (SURVEY.md §8e): split the window list into `nshards` contiguous ranges balanced by
 * sites read; shard cuts fall on window starts, neighbours overlap by the W-S halo.
 * Returns the window range [w_lo, w_hi) and the site/entry range [site_lo, site_hi) that shard
 * `shard` must hold.  Results are bit-identical for any nshards. */
int pgt_plan_shard(const pgt_plan* plan, uint32_t shard, uint32_t nshards, uint64_t* w_lo, uint64_t* w_hi,
                   uint64_t* site_lo, uint64_t* site_hi);

/* Optional: keep the plan's device tables (segments and contig offsets, a few KB) resident in
 * caller-owned device memory of at least pgt_plan_device_bytes(), so that scans upload nothing
 * (lower per-call latency for small inputs; a device-mode site scan then consists of kernel
 * launches only and can be captured into a CUDA graph).  The buffer must outlive the binding;
 * buffer = NULL unbinds.  A bound plan may only be scanned on the device that owns the buffer. */
size_t pgt_plan_device_bytes(const pgt_plan* plan);
int pgt_plan_bind_device(pgt_plan* plan, void* buffer, size_t bytes, void* stream);

/* ---- scan: the hot path ----------------------------------------------------------------
 *
 * A scan processes windows [w_lo, w_hi) of the plan.  Column pointers address element
 * `site_origin` of the global column (site_origin = 0 and the full window range for a
 * single-GPU whole-genome call; the shard's site_lo otherwise).  Output arrays have
 * w_hi - w_lo elements; any output pointer may be NULL.
 */
typedef struct {
	uint64_t w_lo, w_hi;   /* window range; w_lo = w_hi = 0 means "all windows" */
	uint64_t site_origin;  /* global SITE index of element 0 of the column pointers */
	uint64_t site_count;   /* elements the columns hold; 0 = up to the end of the genome.
	                          Only consulted in PGT_MODE_BP (bounds the position searches). */
} pgt_range;

typedef enum {
	PGT_STAT_FST = 0,   /* fstWindow (PGT_MODE_BP plan: fixed-bp windows, as ANGSD's realSFS fst stats2 -win/-step) */
	PGT_STAT_HET = 1,   /* hetWindow (PGT_MODE_BP plan: fixed-bp windows) */
	PGT_STAT_DXY = 2,   /* dxyWindow (-fixedsite 1: PGT_MODE_SITES plan; -fixedsite 0: PGT_MODE_BP plan) */
	PGT_STAT_FUSED = 3  /* fst + dxy + het over one site axis in one pass (BASELINE config 5), either mode; each
	                       statistic equals its single scan bit for bit */
} pgt_stat;

/* Input columns, one element per site; only the columns of the requested statistic are read.
 *   pos        uint32  fstWindow.cpp:18 / hetWindow.cpp:18 / dxyWindow.cpp:26.  Gathered only at
 *              window edges; may be NULL in PGT_MODE_SITES (positions are then not written).
 *              Required in PGT_MODE_BP (it places sites on the bp axis; must be strictly
 *              increasing within a chromosome and <= the chromosome length).
 *   a, b       double  per-site FST numerator / denominator (fstWindow.cpp:19-20)
 *   geno       int8    genotype 0/1/2, negative = missing (hetWindow.cpp:78-80; the parser
 *              clamps wider ints: <0 -> -1, >127 -> 127)
 *   f1,f2,n1,n2  allele frequency (double) and nInd (int32) of pop 1 / pop 2 at the synced
 *              sites (dxyWindow.cpp:24-32,381) */
typedef struct {
	const uint32_t* pos;
	const double* a;
	const double* b;
	const int8_t* geno;
	const double* f1;
	const double* f2;
	const int32_t* n1;
	const int32_t* n2;
} pgt_columns;

/* Per-window results (SoA, w_hi - w_lo elements each; any pointer may be NULL).
 *   fstWindow.cpp:88   chr start end mid fst nsites
 *   hetWindow.cpp:87   chr start last mid h nonmissing
 *   dxyWindow.cpp:190  chr start end dxy neffective nskip   (+ global line, :429-433)
 * -skip_missing 1 (dxyWindow.cpp:189) is a row filter `neffective > 0` for the caller. */
typedef struct {
	uint32_t* label;       /* contig index whose name is printed (contig of the last site) */
	uint32_t* start_pos;   /* pos of first site (bp mode: first bp of the window) */
	uint32_t* end_pos;     /* pos of last site  (bp mode: last bp of the window) */
	uint32_t* mid_pos;     /* (start+end)/2 in uint32 arithmetic (fstWindow.cpp:73) */
	uint32_t* nsites;      /* sites in the window (PGT_MODE_BP: bp; see pgt_scan_bp_sites) */
	double* sum_a;         /* fst */
	double* sum_b;
	double* fst;           /* sum_b != 0 ? sum_a/sum_b : 0 (fstWindow.cpp:85) */
	uint32_t* nhet;        /* het */
	uint32_t* nonmissing;
	double* het;           /* nonmissing ? nhet/nonmissing : 0 (hetWindow.cpp:84) */
	double* dxy;           /* dxy: window SUM of per-site dxy (dxyWindow.cpp:179-186) */
	uint32_t* neffective;
	uint32_t* nskip;
	double* dxy_global;    /* [3] = dxy_global, neffective_global, nskip_global over the units this
	                          scan owns (all sites for an unsharded scan; dxyWindow.cpp:382-385) */
} pgt_windows;

/* Which kernels a scan of `stat` over this plan runs -- a function of (W, S, unit_sites, stat) only, never of
 * the input size or the shard, because it fixes the summation order (DESIGN.md "Summation order"):
 *   PGT_PATH_UNITS    level 1 (unit partials) + level 2 (window combine): every geometry with steps of >= 32 sites
 *   PGT_PATH_SLIDE    fine steps under long windows (e.g. W = 1000, S = 1; what the reference does at
 *                     fstWindow.cpp:80-99 per window): windows formed straight from the sites in shared memory
 *   PGT_PATH_PERSITE  W = S = 1, the tools' default arguments: an elementwise map
 * Returns the path (>= 0) or a negative pgt_status. */
enum { PGT_PATH_UNITS = 0, PGT_PATH_SLIDE = 1, PGT_PATH_PERSITE = 2 };
int pgt_plan_scan_path(const pgt_plan* plan, pgt_stat stat);

/* Device scratch needed by a scan of `stat` over `range` with columns in `mem`. */
size_t pgt_scan_workspace_bytes(const pgt_plan* plan, const pgt_range* range, pgt_stat stat, pgt_mem mem);

/* The scan.  minind: dxyWindow -minind (ignored for fst/het).  site_offsets: PGT_MODE_BP only,
 * host array [ncontig+1] of cumulative SITE counts per chromosome of the plan (global site
 * indices, same origin convention as the columns); NULL in PGT_MODE_SITES. */
int pgt_scan(const pgt_plan* plan, const pgt_range* range, pgt_stat stat, const pgt_columns* cols, int minind,
             const uint64_t* site_offsets, const pgt_windows* out, void* workspace, size_t workspace_bytes,
             pgt_mem mem, void* stream);

/* Sites per window of a PGT_MODE_BP plan: nsites_data[w - w_lo] = number of sites whose positions fall on the bp of
 * window w, for the windows of `range` (the rows of a pgt_scan over the same plan and range; its `nsites` counts bp).
 * pos and site_offsets as for pgt_scan: pos addresses element range->site_origin of the position column and holds
 * range->site_count elements (0 = up to the end of the genome).  The call
 * also checks that every chromosome's first and last site it reads lie on the chromosome (1 <= pos <= length) and
 * returns PGT_ERR_INPUT otherwise; to report that it waits for `stream` in both memory spaces.  PGT_MEM_HOST stages
 * the positions of the chromosomes the windows touch through the workspace (4 bytes per site).  The workspace is
 * device memory of at least pgt_scan_bp_sites_workspace_bytes() (site_offsets may be NULL for PGT_MEM_DEVICE). */
size_t pgt_scan_bp_sites_workspace_bytes(const pgt_plan* plan, const pgt_range* range, const uint64_t* site_offsets, pgt_mem mem);
int pgt_scan_bp_sites(const pgt_plan* plan, const pgt_range* range, const uint32_t* pos, const uint64_t* site_offsets,
                      uint32_t* nsites_data, void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream);

/* One host column set, several GPUs of ONE process (the reference is a single process, fstWindow.cpp:158-177: a
 * user of the drop-in tools on an 8-GPU box should not have to split the input).  The window list is cut by
 * pgt_plan_shard into `ndev` contiguous ranges; shard i runs the PGT_MEM_HOST scan on devices[i] from its own
 * host thread and stream, reads only the slabs of `cols` its windows cover (columns address the WHOLE axis, as
 * for an unsharded scan with site_origin 0) and copies its rows device -> host straight into `out` at its window
 * offset; `out` arrays hold pgt_plan_num_windows elements.  No gather, no collective.  Per-window results are
 * bit-identical for any ndev; dxy_global is the sum of the shards' disjoint partial lines in shard order.
 * workspaces[i] is device memory on devices[i] of at least pgt_scan_sharded_workspace_bytes(plan, stat, i, ndev);
 * workspaces = workspace_bytes = NULL lets the call allocate and free its scratch itself.
 * The plan must not be bound to a device (pgt_plan_bind_device). */
size_t pgt_scan_sharded_workspace_bytes(const pgt_plan* plan, pgt_stat stat, uint32_t shard, uint32_t nshards);
int pgt_scan_sharded(const pgt_plan* plan, pgt_stat stat, const pgt_columns* cols, int minind,
                     const uint64_t* site_offsets, const pgt_windows* out, const int* devices, uint32_t ndev,
                     void* const* workspaces, const size_t* workspace_bytes);

/* ---- streaming upload -----------------------------------------------------------------------------------------
 * The reference streams its input (fstWindow.cpp:123-146).  A producer that is still running -- the tools' parser
 * threads, a reader of a binary column cache -- hands finished ranges to an uploader, which moves them to device
 * memory through a persistent ring of `nslots` page-locked slots of `slot_bytes` each: `nthreads` copy threads fill
 * free slots (memcpy from ordinary pageable memory, or pread from a file so that a cache never goes through a
 * page-cache mapping) and send them on with cudaMemcpyAsync, the filling of one slot overlapping the DMA of the
 * others (pageable cudaMemcpy: ~11 GB/s on these hosts; pinned: ~54 GB/s).  The scan then runs on the resident
 * columns (PGT_MEM_DEVICE).  `pinned` is caller-owned page-locked memory (pgt_host_alloc) of at least
 * pgt_uploader_pinned_bytes() that outlives the uploader, or NULL to let the uploader own its ring.  The uploader
 * belongs to the device current at creation.  put / put_file only enqueue and return; drain waits until every
 * queued byte is on the device (and reports how many went).  Errors of the copy threads surface at the next call. */
typedef struct pgt_uploader pgt_uploader;
size_t pgt_uploader_pinned_bytes(uint32_t nslots, size_t slot_bytes);
int pgt_uploader_create(pgt_uploader** up, void* pinned, size_t pinned_bytes, uint32_t nslots, size_t slot_bytes,
                        uint32_t nthreads);
int pgt_uploader_put(pgt_uploader* up, void* dev_dst, const void* host_src, size_t bytes);
int pgt_uploader_put_file(pgt_uploader* up, void* dev_dst, int fd, uint64_t file_offset, size_t bytes);
int pgt_uploader_drain(pgt_uploader* up, uint64_t* bytes_sent);
void pgt_uploader_destroy(pgt_uploader* up);
/* for callers that do not link the CUDA runtime (the CLIs): synchronous device -> host copy, free / total HBM */
int pgt_memcpy_to_host(void* host, const void* dev, size_t bytes);
int pgt_device_mem_info(size_t* free_bytes, size_t* total_bytes);

/* Convenience entry points named after the tools they replace.  pgt_scan_fst, _het and _fused pass no site_offsets,
 * so they scan PGT_MODE_SITES plans only; a PGT_MODE_BP scan of those statistics goes through pgt_scan. */
int pgt_scan_fst(const pgt_plan* plan, const pgt_range* range, const pgt_columns* cols, const pgt_windows* out,
                 void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream);
int pgt_scan_het(const pgt_plan* plan, const pgt_range* range, const pgt_columns* cols, const pgt_windows* out,
                 void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream);
int pgt_scan_dxy(const pgt_plan* plan, const pgt_range* range, const pgt_columns* cols, int minind,
                 const uint64_t* site_offsets, const pgt_windows* out, void* workspace, size_t workspace_bytes,
                 pgt_mem mem, void* stream);
int pgt_scan_fused(const pgt_plan* plan, const pgt_range* range, const pgt_columns* cols, int minind,
                   const pgt_windows* out, void* workspace, size_t workspace_bytes, pgt_mem mem, void* stream);

/* ---- synthetic inputs (SURVEY.md §8d): on-device counter-based generator --------------- */
/* Fills a[0..n), b[0..n) with the fst columns of global sites [site0, site0+n). Device pointers. */
int pgt_synth_fst(uint64_t seed, uint64_t site0, uint64_t n, double* a, double* b, void* stream);
int pgt_synth_het(uint64_t seed, uint64_t site0, uint64_t n, int8_t* geno, void* stream);
int pgt_synth_dxy(uint64_t seed, uint64_t site0, uint64_t n, double* f1, double* f2, int32_t* n1, int32_t* n2,
                  void* stream);
/* pos[i] for global sites [site0, site0+n) given the genome's contig offsets (host array). */
int pgt_synth_pos(uint64_t seed, uint64_t site0, uint64_t n, const uint64_t* contig_offsets, uint32_t ncontig,
                  uint32_t density, uint32_t* pos, void* stream);

/* Optional per-kernel device timing (bench.py's roofline): while enabled, every level-1 (unit
 * reduction) and level-2 (window combine) launch is bracketed by CUDA events on its stream.
 * pgt_profile_read synchronises those events, returns summed milliseconds / launch counts since
 * the last read, and clears them. */
int pgt_profile(int enable);
int pgt_profile_read(double* units_ms, uint64_t* units_launches, double* windows_ms, uint64_t* windows_launches);

/* Tuning knobs for tests and experiments (never needed for correct results):
 *   "level1": 0 auto | 1 direct warp-per-unit kernel (long units only) | 2 tiled TMA-staged kernel
 *   "level2": 0 auto | 1 always warp-per-window | 2 always scan mode (block prefix/suffix scans)
 *   "fused2": 0 auto (fused sliding tile, W > 512: two crews of warps -- fst + het, dxy -- over one staged block) | 1 one crew with the fused accumulator
 *   "slideglobal": 0 auto (the sliding tile adds up dxyWindow's global line on the way when its runs own exactly the line's sites) | 1 always a separate pass over the dxy columns
 *   "persite": 0 auto | 1 always the scalar per-site kernel (W = S = 1)
 *   "unittable": 0 auto (plans of more than 32 segments in device mode: level 1 reads unit starts from a table) | 1 never | 2 always
 *   "slide": 0 auto | 1 never use the sliding-tile kernel for fine steps | 2 use it for every site-mode geometry whose block fits shared memory (W <= 1048)
 *   "stages", "stage_kb": shared-memory ring of the tiled kernel
 *   "xsmall": extreme scan, 0 auto (short windows: a thread per window over a shared-memory tile) | 1 never | 2 whenever the longest window is <= 2048 sites
 *   "xgroup": lanes per unit of the extreme scan's level 1 (pgt_extreme.h), 0 auto | 4 | 8 | 16 | 32 */
int pgt_tune(const char* key, int value);

/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t pgt_kernel_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PGT_SCAN_H */
