// sitewindow_main.cpp -- drop-in `fstWindow` (-DPGT_TOOL_FST) and `hetWindow` (-DPGT_TOOL_HET).
//
// Same argv grammar, defaults, usage text, messages, stdout columns and exit codes as
//   /root/reference/fstWindow.cpp:23-67,158-177   and   /root/reference/hetWindow.cpp:20-64,156-175
// The line loop + calcWindow of the reference (fstWindow.cpp:109-155, 69-107) is replaced by:
// parse the text into columns (multi-threaded), ask libpgtscan for the closed-form window plan
// and run the CUDA scan (pgt_scan, PGT_MEM_HOST), print the rows.
//
// Documented deviations (the reference has undefined behaviour there, SURVEY.md §5):
//   * step size <= 0: the reference prints the message and carries on into heap corruption;
//     we print the same message and exit 255.
//   * step size > window size: the reference segfaults; we print an error and exit 255.
//   * a line that does not parse: the reference silently reuses stale values; we report it.
//   * the input file is opened read-only (the reference needs write permission, fstWindow.cpp:45).
// Binary columnar cache (pgt_colfile.h): PGT_PACK=<out.pgtc> parses the text, writes the cache and
// exits without touching the GPU; a `.pgtc` file given as the input (magic sniff) skips the parsing.
// Set PGT_TIMING=1 for a JSON timing line on stderr (parse / scan / format, opt-in so stderr
// stays byte-identical by default); PGT_DEVICE selects the GPU, PGT_THREADS the parser threads.
#include "pgt_cli.h"
#include "pgt_colfile.h"

using namespace pgtcli;

#if defined(PGT_TOOL_FST)
static const char* kTool = "fstWindow";
static const char* kUsageLine = "fstWindow [ANGSD fst variance component file] [window size (number sites)] [step size (number sites)]\n";
static const char* kStatName = "(5) Fst\n";
static const char* kOpenErr = "Unable to open Fst variance components file ";
#elif defined(PGT_TOOL_HET)
static const char* kTool = "hetWindow";
static const char* kUsageLine = "hetWindow [genotypes file] [window size (number sites)] [step size (number sites)]\n";
static const char* kStatName = "(5) heterozygosity\n";
static const char* kOpenErr = "Unable to open genotypes file ";
#else
#error "define PGT_TOOL_FST or PGT_TOOL_HET"
#endif

// fstWindow.cpp:23-35 / hetWindow.cpp:20-32
static void info(unsigned winsize, unsigned stepsize) {
	printf("\nUsage:\n%sdefault window size: %u\ndefault step size: %u\n\nOutput:\n(1) chromosome\n(2) window start\n(3) window end\n"
	       "(4) window midpoint position\n%s(6) Number sites in window\n\n",
	       kUsageLine, winsize, stepsize, kStatName);
}

int main(int argc, char** argv) {
	unsigned winsize = 1, stepsize = 1;  // fstWindow.cpp:161-162
	if (argc < 2) {
		info(winsize, stepsize);
		return 0;
	}
	const double t_start = now_ms();
	Input in;
	if (read_input(argv[1], &in, false) != 0) {
		fprintf(stderr, "%s%s\n", kOpenErr, argv[1]);
		return -1;
	}
	if (argc > 2) {
		int w = atoi(argv[2]);
		if (w <= 0) {
			fprintf(stderr, "Window size must be a positive integer\n");
			return -1;
		}
		winsize = (unsigned)w;
	}
	if (argc > 3) {
		int s = atoi(argv[3]);
		if (s <= 0) {
			fprintf(stderr, "Step size must be a positive integer\n");
			return -1;
		}
		stepsize = (unsigned)s;
	}
	if (stepsize > winsize) {
		fprintf(stderr, "Step size must not exceed window size\n");
		return -1;
	}

	// ---- parse (timed separately from compute) --------------------------------------------
	Timing tm;
	DeviceWarmup warm;
	const char* pack_path = getenv("PGT_PACK");
	if (!pack_path) warm.start();
#if defined(PGT_TOOL_FST)
	const uint32_t want_kind = pgtcol::KIND_FST;
#else
	const uint32_t want_kind = pgtcol::KIND_HET;
#endif
	pgtcol::View view;
	const bool columnar = pgtcol::is_colfile(in.data, in.size);
	if (columnar && pgtcol::open_view_of(in.data, in.size, want_kind, &view, kTool, argv[1]) != 0) return -1;
	const size_t n_eff = columnar ? 0 : effective_size(in.data, in.size);
	const unsigned nt = n_eff < parallel_min_bytes() ? 1 : parse_threads();
	tm.threads = nt;
	// Many more chunks than threads, handed out in file order: rows reach the uploader below chunk by chunk
	// while the rest is still being parsed.
	const unsigned nchunk_want = (nt > 1 && n_eff >= ((size_t)64 << 20)) ? nt * 8 : nt;
	uint64_t n = 0;
	std::vector<TextChunk> chunks = split_lines(in.data, 0, n_eff, nchunk_want, nt, &n);
	if (columnar) n = view.nsites;
	// columnar input: the columns are the file mapping itself (read-only from here on)
	uint32_t* pos = columnar ? (uint32_t*)view.col[0] : (uint32_t*)malloc(std::max<uint64_t>(n, 1) * sizeof(uint32_t));
#if defined(PGT_TOOL_FST)
	double* col_a = columnar ? (double*)view.col[1] : (double*)malloc(std::max<uint64_t>(n, 1) * sizeof(double));
	double* col_b = columnar ? (double*)view.col[2] : (double*)malloc(std::max<uint64_t>(n, 1) * sizeof(double));
	if (!pos || !col_a || !col_b) {
#else
	int8_t* geno = columnar ? (int8_t*)view.col[1] : (int8_t*)malloc(std::max<uint64_t>(n, 1));
	if (!pos || !geno) {
#endif
		fprintf(stderr, "%s: out of memory for %llu sites\n", kTool, (unsigned long long)n);
		return -1;
	}
#if defined(PGT_TOOL_FST)
	StreamColumn scol[3] = {{pos, 4, columnar ? (uint64_t)((const char*)view.col[0] - in.data) : 0, 0},
	                        {col_a, 8, columnar ? (uint64_t)((const char*)view.col[1] - in.data) : 0, 1},
	                        {col_b, 8, columnar ? (uint64_t)((const char*)view.col[2] - in.data) : 0, 2}};
	const int nscol = 3;
#else
	StreamColumn scol[2] = {{pos, 4, columnar ? (uint64_t)((const char*)view.col[0] - in.data) : 0, 0},
	                        {geno, 1, columnar ? (uint64_t)((const char*)view.col[1] - in.data) : 0, 3}};
	const int nscol = 2;
#endif
	// Streaming upload (pgt_cli.h ColumnStreamer): device-resident columns filled while the parser runs (text) or
	// straight from the cache file (pread into the pinned ring); the scan then reads HBM, not host memory.
	ColumnStreamer streamer;
	if (!pack_path && n > 0) streamer.start(&warm, scol, nscol, n, (uint64_t)n / stepsize + 65536, 28, columnar ? argv[1] : nullptr);
	for_chunks(chunks, nt, [&](TextChunk& c, size_t) {
		const char* p = in.data + c.begin;
		const char* e = in.data + c.end;
		uint64_t row = c.row0;
		long li = 0;
		while (p < e) {
			const char* s;
			const char* t;
			const char* q;
			// common line shape in one pass (pgt_cli.h fast_line); anything unusual takes the general path below
			const char* next = nullptr;
#if defined(PGT_TOOL_FST)
			double ab[2];
			const bool fast = fast_line<2, false>(p, e, &s, &t, &pos[row], ab, nullptr, &next);
			if (fast) {
				col_a[row] = ab[0];
				col_b[row] = ab[1];
			}
#else
			int32_t g = 0;
			const bool fast = fast_line<1, true>(p, e, &s, &t, &pos[row], nullptr, &g, &next);
#endif
			if (fast) {
				q = next < e || (next == e && e[-1] == '\n') ? next - 1 : nullptr;  // position of this line's '\n', if any
			} else {
				q = (const char*)memchr(p, '\n', (size_t)(e - p));
				const char* le = q ? q : e;
				s = skip_ws(p, le);
				t = token_end(s, le);
				bool ok = t > s;
				const char* cur = t;
				if (ok) ok = parse_u32(cur, le, &pos[row]);
#if defined(PGT_TOOL_FST)
				if (ok) ok = parse_f64(cur, le, &col_a[row]);
				if (ok) ok = parse_f64(cur, le, &col_b[row]);
#else
				g = 0;
				if (ok) ok = parse_i32(cur, le, &g);
#endif
				if (!ok && c.bad_line < 0) c.bad_line = li;
			}
#if defined(PGT_TOOL_HET)
			// hetWindow.cpp:78-80 only distinguishes g < 0, g == 1, other
			geno[row] = (int8_t)(g < 0 ? -1 : (g > 127 ? 127 : g));
#endif
			c.add_row(s, t);
			++row;
			++li;
			if (!q) break;
			p = q + 1;
		}
		if (!columnar) streamer.rows_ready(c.row0, c.row0 + c.nlines);
	});
	std::vector<ContigRun> runs;
	if (columnar) runs = view.runs;
	const int64_t bad = merge_chunks(chunks, &runs);
	if (bad >= 0) {
		fprintf(stderr, "%s: cannot parse line %llu of %s\n", kTool, (unsigned long long)(bad + 1), argv[1]);
		return -1;
	}
	tm.sites = n;
	tm.parse_ms = now_ms() - t_start;
	if (pack_path) {  // write the binary columnar cache and stop: no GPU involved
#if defined(PGT_TOOL_FST)
		const void* cols[3] = {pos, col_a, col_b};
#else
		const void* cols[2] = {pos, geno};
#endif
		if (pgtcol::write_file(pack_path, want_kind, runs, n, cols) != 0) {
			fprintf(stderr, "%s: cannot write %s\n", kTool, pack_path);
			return -1;
		}
		tm.total_ms = now_ms() - t_start;
		tm.report(kTool);
		return 0;
	}
	if (n == 0) {
		tm.total_ms = now_ms() - t_start;
		tm.report(kTool);
		return 0;
	}

	// ---- plan + scan (libpgtscan, CUDA) ------------------------------------------------------
	const double t_scan = now_ms();
	std::vector<uint64_t> off(runs.size() + 1, 0);
	for (size_t i = 0; i < runs.size(); ++i) off[i + 1] = off[i] + runs[i].count;
	pgt_plan* plan = nullptr;
#if defined(PGT_TOOL_HET)
	const uint32_t unit_sites = 4096;  // integer counts: unit size does not change results, larger is faster
#else
	const uint32_t unit_sites = 512;  // 13 units per 110 KB tile = one round of the 15 consumer warps (measured +2 % over 256)
#endif
	if (pgt_plan_create(&plan, PGT_MODE_SITES, off.data(), (uint32_t)runs.size(), winsize, stepsize, unit_sites) != PGT_OK) {
		fprintf(stderr, "%s\n", pgt_last_error());
		return -1;
	}
	const uint64_t nwin = pgt_plan_num_windows(plan);
	std::vector<uint32_t> label(nwin), startp(nwin), endp(nwin), midp(nwin), cnt(nwin);
	std::vector<double> stat(nwin);
	if (nwin) {
		if (warm.finish() != 0) return -1;
		tm.cuda_init_ms = warm.ms;
		pgt_columns cols;
		memset(&cols, 0, sizeof(cols));
		cols.pos = pos;
		pgt_windows out;
		memset(&out, 0, sizeof(out));
		out.label = label.data();
		out.start_pos = startp.data();
		out.end_pos = endp.data();
		out.mid_pos = midp.data();
#if defined(PGT_TOOL_FST)
		cols.a = col_a;
		cols.b = col_b;
		out.fst = stat.data();
		out.nsites = cnt.data();  // fstWindow.cpp:88 prints *nsites
		const pgt_stat which = PGT_STAT_FST;
#else
		cols.geno = geno;
		out.het = stat.data();
		out.nonmissing = cnt.data();  // hetWindow.cpp:87 prints nonmissing
		const pgt_stat which = PGT_STAT_HET;
#endif
		int rc;
		if (streamer.finish(&tm) == 0) {  // columns are resident in HBM: scan there, copy the rows back
			rc = streamer.scan(plan, which, &out, nwin);
		} else {
			rc = scan_on_devices(plan, nullptr, which, &cols, 1, nullptr, &out);
		}
		if (rc != PGT_OK) {
			fprintf(stderr, "%s: %s\n", kTool, pgt_last_error());
			return -1;
		}
	}
	tm.windows = nwin;
	tm.scan_ms = now_ms() - t_scan;

	// ---- print -----------------------------------------------------------------------------
	const double t_fmt = now_ms();
	size_t maxname = 0;
	for (const ContigRun& r : runs) maxname = std::max(maxname, r.name.size());
	static char obuf[1 << 20];
	setvbuf(stdout, obuf, _IOFBF, sizeof(obuf));
	write_rows(stdout, nwin, maxname + 96, [&](char* p, uint64_t w) {
		const std::string& nm = runs[label[w]].name;
		memcpy(p, nm.data(), nm.size());
		p += nm.size();
		*p++ = '\t';
		p = put_u32(p, startp[w]);
		*p++ = '\t';
		p = put_u32(p, endp[w]);
		*p++ = '\t';
		p = put_u32(p, midp[w]);
		*p++ = '\t';
		p = put_g(p, stat[w]);
		*p++ = '\t';
		p = put_u32(p, cnt[w]);
		*p++ = '\n';
		return p;
	});
	fflush(stdout);
	tm.format_ms = now_ms() - t_fmt;
	tm.total_ms = now_ms() - t_start;
	tm.report(kTool);
	pgt_plan_destroy(plan);
	return 0;
}
