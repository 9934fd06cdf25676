// pgt_slide.cuh -- fine steps under long windows: windows formed straight from the sites in shared memory (k_slide), and dxyWindow's global line kernels
// Part of the one translation unit pgt_scan.cu (device code only; included from there, in this order:
// pgt_kernels_common.cuh, pgt_level1.cuh, pgt_level2.cuh, pgt_slide.cuh).
#ifndef PGT_SLIDE_CUH
#define PGT_SLIDE_CUH

// ----------------------------------------------------------------------------- fine steps: sliding tile
//
// W = 1000, S = 1 and its kin: steps so short that a "unit" would be a handful of sites (pgt_geom.h:
// units never span a step), so the two-level scheme degenerates into copying every site into the unit
// array and scanning that array twice in global memory (~3x the compulsory traffic).  Here the windows
// are formed straight from the sites, in shared memory, and no unit array exists:
//
//   * the site axis of a segment is cut into BLOCKS of W sites from the segment origin; window k
//     (first site f = k*S, last site l) touches block m = f div W and at most block m + 1, so
//         window = SUF_m[f mod W] (+ PRE_{m+1}[l mod W] when l is in block m + 1)
//     with PRE / SUF the inclusive prefix / suffix sums inside a block (van Herk / Gil-Werman): only
//     additions of true partial sums, no differences, no cancellation;
//   * persistent CTAs take CHUNKS of consecutive windows; a chunk walks its blocks in order, G blocks per
//     step: the producer warp stages the step's slice of every column (positions included) with bulk
//     async copies (the ring of k_units_tiled); every block is scanned by its own team of WPB warps
//     (thread q of a team owns elements [q*E, (q+1)*E) of its block: forward total, two warp shuffle scans,
//     the team's warp totals through shared memory, then PRE running forward from the thread's base and
//     SUF running backward from it); the windows that start in the blocks of the step -- all but its last
//     block, plus the last block of the step before -- are emitted from SUF and PRE in shared memory with
//     coalesced row stores.  SUF and the positions are double-buffered by step parity, so a step has two
//     CTA-wide barriers.  Every site is read once per chunk; neighbouring chunks share W - S sites.
//     (E, WPB, G) are chosen per W so that a step covers as many sites as the 7 consumer warps can own:
//     W = 1000: E = 5, one block of 7 warps; W = 256: E = 4, three blocks of 2 warps.
//
// Summation order: a pure function of (W, S) and the position of a site inside its block -- not of
// chunks, CTAs, stages or shards (a chunk that starts or ends inside a block simply has the sites
// outside its windows absent, and those only ever enter prefix / suffix values no window of the chunk
// reads), so results are bit-identical for any GPU count.  Reference semantics: fstWindow.cpp:80-99.

static constexpr int kSlideWarps = 7;                          // consumer warps (+ the producer warp = 256 threads: 128 registers each at two CTAs per SM)
static constexpr int kSlideConsumers = kSlideWarps * 32;
static constexpr int kSlideThreads = kSlideConsumers + 32;     // + the producer warp (the last one)
static constexpr uint32_t kSlideMaxE = 6;                      // W <= 1344 (and the fused step must fit shared memory: W <= 1048)
static constexpr uint32_t kSlideWtBytes = 512;                 // warp totals: 7 x Acc (<= 40 B)

// The team shape for a window size: E elements per thread, WPB warps per block, G = 7 / WPB blocks per step --
// the (E, WPB) with the most sites per step, the smaller E on ties.  Part of the summation order.
struct SlideTeam {
	uint32_t E, wpb, G;
};
// (a step holds at most 1024 sites -- G * (W rounded up to 32) -- so that the fused statistic's step fits shared memory)
__host__ __device__ inline SlideTeam slide_team(uint32_t W) {
	SlideTeam best{1, kSlideWarps, 0};
	const uint32_t wp = (W + 31u) / 32u * 32u;
	for (uint32_t E = 1; E <= kSlideMaxE; ++E) {
		const uint32_t tpb = (W + E - 1) / E;
		const uint32_t wpb = (tpb + 31) / 32;
		if (wpb > (uint32_t)kSlideWarps) continue;
		uint32_t G = (uint32_t)kSlideWarps / wpb;
		if (G > 1024u / wp) G = 1024u / wp;
		if (G < 1) G = 1;
		if (G > best.G) best = SlideTeam{E, wpb, G};
	}
	return best;
}

struct SlideCfg {
	uint32_t E, wpb, G;      // slide_team(W)
	uint32_t wp;             // stride of one block's arrays in shared memory (W rounded up to 32)
	uint32_t sf_off, pr_off, pos_off, stage_off;  // byte offsets inside the dynamic shared memory
	uint32_t pos_col;        // staging index of the position column, 0xffffffff = positions not wanted
	uint64_t chunk_windows;  // windows per chunk
	uint64_t nchunks;
	double* gpart;           // dxyWindow's global line taken on the way: one partial triple per CTA (NULL: not wanted)
};

template <class Acc>
__device__ __forceinline__ Acc shfl_down_acc(const Acc& v, unsigned delta) {
	static_assert(sizeof(Acc) % 4 == 0, "Acc is made of 32-bit words");
	uint32_t w[sizeof(Acc) / 4];
	memcpy(w, &v, sizeof(Acc));
#pragma unroll
	for (unsigned i = 0; i < sizeof(Acc) / 4; ++i) w[i] = __shfl_down_sync(0xffffffffu, w[i], delta);
	Acc r;
	memcpy(&r, w, sizeof(Acc));
	return r;
}

// the part of a chunk that lies in one segment: windows [ka, kb) of segment `sg` (segment-local), reading
// the segment-local sites [lo, hi)
struct SlideRun {
	pgt_seg sg;
	uint32_t si;
	uint64_t ka, kb, lo, hi;
};
// first run of the chunk [wa, wb) / the run after `r`; false when the chunk is exhausted
__device__ __forceinline__ bool slide_run_at(const DevPlan& P, uint64_t w, uint64_t wb, SlideRun& r, bool first) {
	if (w >= wb) return false;
	if (first) {
		r.si = find_seg<false>(P, w);
		r.sg = P.segs[r.si];
	}
	while (w - r.sg.win_base >= r.sg.nwin) {  // also skips segments without windows
		++r.si;
		r.sg = P.segs[r.si];
	}
	r.ka = w - r.sg.win_base;
	r.kb = wb - r.sg.win_base < r.sg.nwin ? wb - r.sg.win_base : r.sg.nwin;
	r.lo = r.ka * P.g.S;
	const uint64_t e = (r.kb - 1) * P.g.S + P.g.W;
	r.hi = e < r.sg.nsites ? e : r.sg.nsites;
	return true;
}

// (register budget: two CTAs per SM for the narrow statistics -- 128 registers -- and one for the fused
// scan, whose step fills the shared memory of an SM anyway)
template <class Stat>
struct SlideMinBlocks {
	static constexpr int value = 2;
};
template <>
struct SlideMinBlocks<FusedStat> {
	static constexpr int value = 1;
};
// A crew of 7 consumer warps: scans the staged blocks and emits the windows of ONE statistic (the whole job of
// k_slide's consumers).  The fused scan with one block per step runs TWO crews per CTA over the same staged block
// (k_slide_fused2: fst + het, and dxy), each with its own shared-memory arrays and named barrier.
struct SlideCrew {
	uint32_t t;          // thread inside the crew (0..223)
	uint32_t warp;       // warp inside the crew (0..6)
	uint32_t bar_id;     // named barrier of the crew
	uint32_t col_shift;  // first staged column of the crew's statistic
	bool common;         // the crew writes what all statistics share: label, positions, nsites
	void* wt;            // shared memory: warp totals, SUF [2][G * wp], PRE [G * wp], positions [2][G * wp]
	void* sf;
	void* pr;
	uint32_t* pos;
	double* gpart;       // this crew adds up the global line of the sites its windows own (NULL: no)
};

__device__ __forceinline__ void slide_bar(uint32_t id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(kSlideConsumers) : "memory"); }

template <class Stat, int EMAX, bool MULTI>
__device__ __forceinline__ void slide_consume(const DevPlan& P, const TileCfg& tc, const SlideCfg& sc, const pgt_windows& out, TileCtl* ctl,
                                              const SlideCrew& crew) {
	typedef typename Stat::Acc Acc;
	Acc* wt = reinterpret_cast<Acc*>(crew.wt);
	Acc* SfBase = reinterpret_cast<Acc*>(crew.sf);
	Acc* Pr = reinterpret_cast<Acc*>(crew.pr);
	uint32_t* PosBase = crew.pos;
	const uint64_t W = P.g.W, S = P.g.S;
	const uint32_t Wu = P.g.W, Su = P.g.S, G = MULTI ? sc.G : 1u, gw = G * sc.wp;
	const uint32_t wpb = MULTI ? sc.wpb : (uint32_t)kSlideWarps;
	const bool has_pos = crew.common && sc.pos_col != 0xffffffffu;
	const uint32_t t = crew.t, warp = crew.warp, lane = crew.t & 31u;
	const uint32_t team = MULTI ? warp / wpb : 0u;  // which block of a step this thread works on (>= G: none)
	const uint32_t tw = warp - team * wpb;          // warp inside its team
	const uint32_t e0 = (tw * 32u + lane) * sc.E;   // first element of the block this thread owns
	const bool member = MULTI ? team < G : true;
	uint32_t it = 0, step = 0;  // `step` selects the halves of the double buffers
	// dxyWindow's global line: a run of windows [ka, kb) OWNS the sites from its first window's start up to the start of
	// window kb (the next run's first site), or to the end of what it stages when kb is the segment's last window; the runs
	// of all chunks tile the windows, so every staged site is owned exactly once (the overlap W - S belongs to the later run)
	const bool take_global = GlobalTerm<Stat>::has && crew.gpart != nullptr;
	double gd = 0.0;
	unsigned long long gne = 0, gnk = 0;
	for (uint64_t c = blockIdx.x; c < sc.nchunks; c += gridDim.x) {
		const uint64_t wa = P.win_lo + c * sc.chunk_windows;
		const uint64_t wb = P.win_hi - wa < sc.chunk_windows ? P.win_hi : wa + sc.chunk_windows;
		SlideRun r;
		for (bool ok = slide_run_at(P, wa, wb, r, true); ok; ok = slide_run_at(P, r.sg.win_base + r.kb, wb, r, false)) {
			const uint64_t m_first = r.lo / W, m_last = (r.hi - 1) / W;
			const uint64_t own_hi = r.kb == r.sg.nwin ? r.hi : r.kb * S;  // relative to the segment, like r.lo / r.hi
			// label = contig of the window's last site: the windows a thread emits go up the axis, so a cursor
			// that only walks forward replaces a binary search per window
			uint32_t lc = r.sg.first_contig;
			uint64_t lc_end = r.sg.ncontig > 1 ? P.off[lc + 1] : ~0ull;  // global site where contig lc ends
			// kc = ceil(b*W / S): first window that starts at or after block b; kept incrementally
			uint64_t kq = m_first * W / S;
			uint32_t krem = (uint32_t)(m_first * W - kq * S);
			uint64_t kc_from = kq + (krem != 0u);  // first window not yet emitted (by block start)
			for (uint64_t b = m_first; b <= m_last; b += G, ++step) {
				// blocks [b, b + gi) arrive; the windows starting in blocks [b - 1, b + gi - 2] leave -- and those of
				// block b + gi - 1 too when it is the run's last block (they end inside it)
				const uint32_t gi = (uint32_t)(m_last + 1 - b < G ? m_last + 1 - b : G);
				Acc* Sf = SfBase + (step & 1u) * gw;
				const Acc* SfPrev = SfBase + ((step & 1u) ^ 1u) * gw + (G - 1u) * sc.wp;  // SUF of block b - 1
				uint32_t* Pos = PosBase + (step & 1u) * gw;
				const uint32_t* PosPrev = PosBase + ((step & 1u) ^ 1u) * gw + (G - 1u) * sc.wp;
				const uint32_t stg = it % tc.nstages;
				mbar_wait(&ctl->full[stg], (it / tc.nstages) & 1u);
				++it;
				Acc leaf[EMAX];
				uint32_t pv[EMAX];
				Acc up = Stat::zero(), dn = Stat::zero();
				{
					const char* cp[kMaxTileCols];
#pragma unroll
					for (int cc = 0; cc < kMaxTileCols; ++cc) cp[cc] = cc + (int)crew.col_shift < kMaxStageCols ? ctl->cp[stg][cc + crew.col_shift] : nullptr;
					const uint32_t* pstage = has_pos ? reinterpret_cast<const uint32_t*>(ctl->cp[stg][sc.pos_col]) : nullptr;
					const uint64_t x0 = b * W > r.lo ? b * W : r.lo;            // first staged site
					const uint64_t x1 = (b + gi) * W < r.hi ? (b + gi) * W : r.hi;
					// sites of a block outside [x0, x1) are absent (other chunk / beyond the segment): +0 leaves
					const uint32_t s_lo = (uint32_t)(x0 - b * W), s_hi = (uint32_t)(x1 - b * W);  // relative to block b
					const uint32_t base = team * Wu + e0;                                          // this thread's first element, same frame
					const uint32_t g_hi = !take_global || own_hi <= b * W ? 0u : (own_hi - b * W < (uint64_t)s_hi ? (uint32_t)(own_hi - b * W) : s_hi);
					Acc tot = Stat::zero();
#pragma unroll
					for (int e = 0; e < EMAX; ++e) {
						leaf[e] = Stat::zero();
						pv[e] = 0u;
						const uint32_t i = base + (uint32_t)e;
						if (member && (uint32_t)e < sc.E && e0 + (uint32_t)e < Wu && i >= s_lo && i < s_hi) {
							PGT_CHECK(i - s_lo < ctl->ns[stg]);
							Stat::fold(leaf[e], Stat::load_tile(cp, i - s_lo), tc.minind, 0.0, 0);  // (no statistic of this path reads the site index)
							if (has_pos) pv[e] = pstage[i - s_lo];
							if (GlobalTerm<Stat>::has && i < g_hi) GlobalTerm<Stat>::add(leaf[e], gd, gne, gnk);
						}
						Stat::add(tot, leaf[e]);
					}
					__syncwarp();
					if (lane == 0) mbar_arrive(&ctl->empty[stg]);  // the step's sites now live in registers
					up = tot;
					dn = tot;
#pragma unroll
					for (unsigned d = 1; d < 32; d <<= 1) {
						Acc o = shfl_up_acc(up, d);
						if (lane >= d) {  // earlier threads first
							Stat::add(o, up);
							up = o;
						}
						Acc q = shfl_down_acc(dn, d);
						if (lane + d < 32u) {  // later threads first
							Stat::add(q, dn);
							dn = q;
						}
					}
					if (lane == 31u) wt[warp] = up;  // the warp's total, forward order
				}
				slide_bar(crew.bar_id);  // warp totals visible; every thread has left the emit phase of the step before
				{
					Acc bpre = Stat::zero(), bsuf = Stat::zero();
#pragma unroll
					for (int w2 = 0; w2 < kSlideWarps - 1; ++w2)  // the team's warps before this one, in order
						if ((uint32_t)w2 < tw && member) Stat::add(bpre, wt[team * wpb + w2]);
#pragma unroll
					for (int w2 = kSlideWarps - 1; w2 > 0; --w2)  // the team's warps after it, last first
						if ((uint32_t)w2 > tw && (uint32_t)w2 < wpb && member) Stat::add(bsuf, wt[team * wpb + w2]);
					Acc xu = shfl_up_acc(up, 1), xd = shfl_down_acc(dn, 1);
					if (lane == 0) xu = Stat::zero();
					if (lane == 31u) xd = Stat::zero();
					Stat::add(bpre, xu);
					Stat::add(bsuf, xd);
					const uint32_t o0 = team * sc.wp + e0;
#pragma unroll
					for (int e = 0; e < EMAX; ++e) {  // PRE: running forward from everything before this thread
						if (member && (uint32_t)e < sc.E && e0 + (uint32_t)e < Wu) {
							Stat::add(bpre, leaf[e]);
							Pr[o0 + e] = bpre;
							if (has_pos) Pos[o0 + e] = pv[e];
						}
					}
#pragma unroll
					for (int e = EMAX - 1; e >= 0; --e) {  // SUF: running backward from everything after it
						if (member && (uint32_t)e < sc.E && e0 + (uint32_t)e < Wu) {
							Stat::add(bsuf, leaf[e]);
							Sf[o0 + e] = bsuf;
						}
					}
				}
				slide_bar(crew.bar_id);  // PRE, SUF and the positions of the step's blocks complete
				{
					// windows that start in blocks [eb_lo, eb_hi]; everything below is relative to the start of block b - 1
					const uint64_t eb_lo = b > m_first ? b - 1 : b;
					const uint64_t eb_hi = (b + gi - 1 == m_last) ? m_last : b + gi - 2;  // may be eb_lo - 1: nothing to emit yet
					// ceil((eb_hi + 1) * W / S): the quotient / remainder of (blocks emitted so far) * W / S stepped forward
					uint64_t kc_to = kc_from;
					if (eb_hi + 1 > eb_lo) {
						const uint32_t nb = (uint32_t)(eb_hi + 1 - eb_lo);
						kq += (uint64_t)nb * P.g.q;
						krem += nb * P.g.r;
						while (krem >= Su) {
							krem -= Su;
							++kq;
						}
						kc_to = kq + (krem != 0u);
					}
					const uint64_t k_lo = kc_from > r.ka ? kc_from : r.ka, k_hi = kc_to < r.kb ? kc_to : r.kb;
					if (eb_hi + 1 > eb_lo && k_hi > k_lo) {
						const uint32_t cnt = (uint32_t)(k_hi - k_lo);
						const uint32_t rel0 = (uint32_t)(k_lo * S + W - b * W);  // first window's start, relative to block b - 1
						const uint64_t left = r.sg.nsites + W - b * W;            // sites of the segment from block b - 1 on
						const uint32_t last_rel = (uint32_t)(left < (uint64_t)(G + 2u) * Wu ? left : (uint64_t)(G + 2u) * Wu) - 1u;
						const uint64_t obase = r.sg.win_base + k_lo - P.win_lo;
						const uint64_t gbase = r.sg.site_base + b * W - W;  // global site of relative position 0
						for (uint32_t i = t; i < cnt; i += kSlideConsumers) {
							const uint32_t rel = rel0 + i * Su;
							uint32_t blk = 0, brel = 0;  // blk = rel / W; brel = blk * W
							if (MULTI) {
								while (rel >= brel + Wu) {  // <= G <= 7 steps
									brel += Wu;
									++blk;
								}
							} else if (rel >= Wu) {
								brel = Wu;
								blk = 1u;
							}
							const uint32_t j = rel - brel;  // blk = 0: block b - 1; blk = 1 + g: block g of this step
							uint32_t lr = rel + Wu - 1u;
							if (lr > last_rel) lr = last_rel;
							const bool two = lr >= brel + Wu;  // the window ends in the next block
							const uint32_t jl = two ? lr - brel - Wu : lr - brel;
							PGT_CHECK(j < Wu && jl < Wu && blk <= gi && (!two || blk < gi) && obase + i < P.win_hi - P.win_lo);
							const uint32_t boff = (blk - 1u) * sc.wp;  // (unused when blk == 0)
							Acc acc = blk == 0u ? SfPrev[j] : Sf[boff + j];
							if (two) Stat::add(acc, Pr[blk * sc.wp + jl]);
							const uint64_t o = obase + i;
							const uint64_t glast = gbase + lr;
							while (glast >= lc_end) {
								++lc;
								lc_end = P.off[lc + 1];
							}
							if (crew.common && out.label) out.label[o] = lc;
							if (crew.common && out.nsites) out.nsites[o] = lr - rel + 1u;
							if (has_pos) {
								const uint32_t* ps = blk == 0u ? PosPrev : Pos + boff;  // positions of the window's first block
								const uint32_t sp = ps[j];
								const uint32_t ep = two ? Pos[blk * sc.wp + jl] : ps[jl];
								if (out.start_pos) out.start_pos[o] = sp;
								if (out.end_pos) out.end_pos[o] = ep;
								if (out.mid_pos) out.mid_pos[o] = (sp + ep) / 2u;  // uint32 arithmetic, fstWindow.cpp:73
							}
							Stat::emit(out, o, acc);
						}
					}
					if (eb_hi + 1 > eb_lo) kc_from = kc_to;
				}
			}
		}
	}
	if (GlobalTerm<Stat>::has && crew.gpart != nullptr) {  // crew-uniform: warps, then the crew's seven warps in order
#pragma unroll
		for (int m = 16; m >= 1; m >>= 1) {
			gd = __dadd_rn(gd, shfl_xor_f64(gd, m));
			gne += __shfl_xor_sync(0xffffffffu, gne, m);
			gnk += __shfl_xor_sync(0xffffffffu, gnk, m);
		}
		slide_bar(crew.bar_id);  // everybody has left the last emit phase: PRE is free
		double* g3 = reinterpret_cast<double*>(Pr);
		if (lane == 0) {
			g3[3 * warp] = gd;
			g3[3 * warp + 1] = (double)gne;
			g3[3 * warp + 2] = (double)gnk;
		}
		slide_bar(crew.bar_id);
		if (t == 0) {
			double d = 0.0, ne = 0.0, nk = 0.0;  // counts: exact in double below 2^53
			for (int w2 = 0; w2 < kSlideWarps; ++w2) {
				d = __dadd_rn(d, g3[3 * w2]);
				ne += g3[3 * w2 + 1];
				nk += g3[3 * w2 + 2];
			}
			crew.gpart[3 * blockIdx.x] = d;
			crew.gpart[3 * blockIdx.x + 1] = ne;
			crew.gpart[3 * blockIdx.x + 2] = nk;
		}
	}
}

// The producer warp of a sliding-tile CTA: one stage per step (G blocks) of every chunk this CTA walks.
__device__ __forceinline__ void slide_produce(const DevPlan& P, const TileCfg& tc, const SlideCfg& sc, TileCtl* ctl, unsigned char* stages,
                                              uint32_t G, uint32_t lane) {
	const uint64_t W = P.g.W;
	uint32_t it = 0;
	for (uint64_t c = blockIdx.x; c < sc.nchunks; c += gridDim.x) {
		const uint64_t wa = P.win_lo + c * sc.chunk_windows;
		const uint64_t wb = P.win_hi - wa < sc.chunk_windows ? P.win_hi : wa + sc.chunk_windows;
		SlideRun r;
		for (bool ok = slide_run_at(P, wa, wb, r, true); ok; ok = slide_run_at(P, r.sg.win_base + r.kb, wb, r, false)) {
			for (uint64_t b = r.lo / W; b * W < r.hi; b += G, ++it) {
				const uint64_t x0 = b * W > r.lo ? b * W : r.lo;
				const uint64_t x1 = (b + G) * W < r.hi ? (b + G) * W : r.hi;
				const uint32_t stg = it % tc.nstages;
				if (it >= tc.nstages) mbar_wait(&ctl->empty[stg], ((it / tc.nstages) - 1u) & 1u);
				producer_fill_stage(tc, ctl, stages, stg, r.sg.site_base + x0 - P.site_origin, r.sg.site_base + x1 - P.site_origin, lane);
			}
		}
	}
}

// MULTI = several blocks per step (G > 1, W <= 512); with one block per step the team arithmetic folds away
template <class Stat, int EMAX, bool MULTI>
__global__ void __launch_bounds__(kSlideThreads, SlideMinBlocks<Stat>::value) k_slide(DevPlan P, TileCfg tc, SlideCfg sc, pgt_windows out) {
	extern __shared__ __align__(128) unsigned char smem[];
	TileCtl* ctl = reinterpret_cast<TileCtl*>(smem);
	const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
	if (threadIdx.x == 0) {
		for (uint32_t s = 0; s < tc.nstages; ++s) {
			mbar_init(&ctl->full[s], 2);
			mbar_init(&ctl->empty[s], kSlideWarps);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncthreads();
	if (warp == kSlideWarps) {
		slide_produce(P, tc, sc, ctl, smem + sc.stage_off, MULTI ? sc.G : 1u, lane);
		return;
	}
	SlideCrew crew;
	crew.t = threadIdx.x;
	crew.warp = warp;
	crew.bar_id = 1;
	crew.col_shift = 0;
	crew.common = true;
	crew.wt = smem + kTileCtlBytes;
	crew.sf = smem + sc.sf_off;    // SUF of the step's blocks: [2][G * wp], by step parity
	crew.pr = smem + sc.pr_off;    // PRE of the step's blocks: [G * wp]
	crew.pos = reinterpret_cast<uint32_t*>(smem + sc.pos_off);  // positions of the step's blocks: [2][G * wp]
	crew.gpart = sc.gpart;
	slide_consume<Stat, EMAX, MULTI>(P, tc, sc, out, ctl, crew);
}

// The fused statistic with one block per step (W > 512) as two crews of 7 warps: crew 0 scans fst + het (staged columns
// a, b, geno: 24-byte accumulators); crew 1 scans dxy (f1, f2, n1, n2: 16 bytes) and also writes label, positions and
// nsites (with those on crew 0 the dxy crew spent 40 % of its time waiting for the next block, ncu r03g: 3.34 -> 3.23 ms
// per 1e8 sites).  They read the same staged block and keep their own SUF / PRE arrays (24 + 16 = the 40 bytes per site
// of the fused accumulator), named barriers 1 and 2.  16 warps per SM instead of 8 at 128 registers per thread instead of 190,
// and every column of the table holds exactly the bits of its single-statistic scan.  A stage drains when all 14
// consumer warps have taken their sites into registers.  (Three crews -- fst, dxy, het: 22 warps, 80 registers -- spilled
// ~420 bytes per thread and gained nothing: DESIGN.md section 12.)
struct SlideCfg2 {
	uint32_t wt_off[2], sf_off[2], pr_off[2];
};
static constexpr int kSlide2Threads = 2 * kSlideConsumers + 32;
template <int EMAX>
__global__ void __launch_bounds__(kSlide2Threads, 1) k_slide_fused2(DevPlan P, TileCfg tc, SlideCfg sc, SlideCfg2 s2, pgt_windows out) {
	extern __shared__ __align__(128) unsigned char smem[];
	TileCtl* ctl = reinterpret_cast<TileCtl*>(smem);
	const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
	if (threadIdx.x == 0) {
		for (uint32_t s = 0; s < tc.nstages; ++s) {
			mbar_init(&ctl->full[s], 2);
			mbar_init(&ctl->empty[s], 2 * kSlideWarps);
		}
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncthreads();
	if (warp == 2 * kSlideWarps) {
		slide_produce(P, tc, sc, ctl, smem + sc.stage_off, 1u, lane);
		return;
	}
	const uint32_t ci = warp / kSlideWarps;  // 0: fst + het, 1: dxy
	SlideCrew crew;
	crew.t = threadIdx.x - ci * kSlideConsumers;
	crew.warp = warp - ci * kSlideWarps;
	crew.col_shift = ci == 0 ? 0u : 2u;
	crew.common = ci == 1;  // dxy has the lighter rows (16 of the 56 statistic bytes): it also writes the 20 shared ones
	crew.wt = smem + s2.wt_off[ci];
	crew.sf = smem + s2.sf_off[ci];
	crew.pr = smem + s2.pr_off[ci];
	crew.pos = reinterpret_cast<uint32_t*>(smem + sc.pos_off);
	crew.gpart = ci == 1 ? sc.gpart : nullptr;
	if (ci == 0) {
		crew.bar_id = 1;
		slide_consume<FstHetStat, EMAX, false>(P, tc, sc, out, ctl, crew);
	} else {
		crew.bar_id = 2;
		slide_consume<DxyStat, EMAX, false>(P, tc, sc, out, ctl, crew);
	}
}

// dxyWindow's global line (dxyWindow.cpp:382-385,429-433) over the unit partials [0, n): one
// block; thread t adds partials t, t+1024, ...; warp butterflies; counts in 64 bit.
template <class Stat>
struct GlobalOf;
template <>
struct GlobalOf<DxyStat> {
	static __device__ __forceinline__ const DxyStat::Acc& get(const DxyStat::Acc& a) { return a; }
};
template <>
struct GlobalOf<FusedStat> {
	static __device__ __forceinline__ const DxyStat::Acc& get(const FusedStat::Acc& a) { return a.dxy; }
};

// stage 1: block b adds partials b*1024 + t + k*(256*1024) per thread t, then reduces the block
template <class Stat>
__global__ void __launch_bounds__(1024) k_global_partial(const typename Stat::Acc* __restrict__ units, uint64_t n, double* __restrict__ partial3) {
	double d = 0.0;
	unsigned long long ne = 0, nk = 0;
	for (uint64_t i = (uint64_t)blockIdx.x * 1024u + threadIdx.x; i < n; i += (uint64_t)kGlobalBlocks * 1024u) {
		const DxyStat::Acc& a = GlobalOf<Stat>::get(units[i]);
		d = __dadd_rn(d, a.dxy);
		ne += a.neff;
		nk += a.nskip;
	}
	block_reduce_global(d, ne, nk, partial3 + 3 * blockIdx.x);
}
// stage 2: one block over the n block partials (thread t adds partials t, t + 256, ... in that order; n = 256: one each)
__global__ void __launch_bounds__(kGlobalBlocks) k_global_final(const double* __restrict__ partial3, uint32_t n, double* __restrict__ global3) {
	double d = 0.0;
	unsigned long long ne = 0, nk = 0;
	for (uint32_t i = threadIdx.x; i < n; i += kGlobalBlocks) {
		d = __dadd_rn(d, partial3[3 * i]);
		ne += (unsigned long long)partial3[3 * i + 1];
		nk += (unsigned long long)partial3[3 * i + 2];
	}
	block_reduce_global(d, ne, nk, global3);
}

// dxyWindow's global line when no unit array exists (sliding-tile and per-site scans): thread t of
// block b folds sites i0 + b*1024 + t + k*(256*1024) of the owned range [i0, i1) (column element
// indices) in that order, then the block reductions of k_global_partial.  Classification as
// DxyStat::fold (dxyWindow.cpp:179-186).
__global__ void __launch_bounds__(1024) k_global_sites(Cols cols, uint64_t i0, uint64_t i1, double* __restrict__ partial3) {
	double d = 0.0;
	unsigned long long ne = 0, nk = 0;
	constexpr int U = 4;  // four sites' column loads in flight per thread; folded in index order
	const uint64_t stride = (uint64_t)kGlobalBlocks * 1024u;
	for (uint64_t i = i0 + (uint64_t)blockIdx.x * 1024u + threadIdx.x; i < i1; i += U * stride) {
		DxyStat::Site v[U];
#pragma unroll
		for (int q = 0; q < U; ++q)
			if (i + q * stride < i1) v[q] = DxyStat::load(cols, i + q * stride);
#pragma unroll
		for (int q = 0; q < U; ++q) {
			if (i + q * stride >= i1) break;
			DxyStat::Acc a = DxyStat::zero();
			DxyStat::fold(a, v[q], cols.minind, 0.0, 0);
			d = __dadd_rn(d, a.dxy);
			ne += a.neff;
			nk += a.nskip;
		}
	}
	block_reduce_global(d, ne, nk, partial3 + 3 * blockIdx.x);
}

#endif  // PGT_SLIDE_CUH
