// dxywindow_main.cpp -- drop-in `dxyWindow`.
//
// Same options, defaults, help text, messages, stdout/stderr split and exit codes as
// /root/reference/dxyWindow.cpp:34-139,518-550.  maf2dxy (dxyWindow.cpp:253-436) is replaced by:
//   1. read both MAFs (plain or gzip, magic sniff as dxyWindow.cpp:82-83), parse them into
//      columns on several threads, skipping the header line (dxyWindow.cpp:284,290);
//   2. the two-file position sync state machine of dxyWindow.cpp:315-331, restated over the
//      parsed arrays (SURVEY.md Appendix A.4: position-only catch-up, silent stop);
//   3. closed-form window plan + CUDA scan in libpgtscan (site windows for -fixedsite 1, sparse
//      bp windows for -fixedsite 0: no per-bp filler entries are ever materialised);
//   4. rows to stdout (-skip_missing filters neffective == 0, dxyWindow.cpp:189), the global
//      line to stderr, or to stdout for -winsize 0 (dxyWindow.cpp:429-433).
//
// Documented deviations (reference behaviour is undefined or a crash there):
//   * -winsize 0 with -fixedsite 0 segfaults in the reference; here: error, exit 255.
//   * -stepsize > -winsize: error, exit 255.
//   * bp mode needs positions strictly increasing within a chromosome and <= its sizefile
//     length (the reference silently produces misplaced entries otherwise): error, exit 255.
//   * MAF files without data lines: error instead of reading an empty record.
// Binary columnar cache (pgt_colfile.h): PGT_PACK=<pop1.pgtc> PGT_PACK2=<pop2.pgtc> parse the two MAFs,
// write one cache per population and exit without touching the GPU; a `.pgtc` file given in place of
// a MAF (magic sniff, next to the gzip sniff of dxyWindow.cpp:82-83) skips the parsing of that file.
// PGT_PACK_SYNCED=<out.pgtc> writes the SYNCED site list of the two files (kind 5) and exits: the result of the
// two-file sync state machine of dxyWindow.cpp:315-331, for inspection and for the CPU fuzz of that logic.
#include <map>
#include <memory>

#include "pgt_cli.h"
#include "pgt_colfile.h"

using namespace pgtcli;

static void help_info(unsigned winsize, unsigned stepsize, int minind, int fixedsite, int skip_missing) {
	// dxyWindow.cpp:34-61 (setw(14) / setw(8), left aligned)
	printf("\ndxyWindow [options] <pop1 maf file> <pop2 maf file>\n\nOptions:\n");
	printf("%-14s%-8sWindow size in base pairs (0 for global calculation) [%u]\n", "-winsize", "INT", winsize);
	printf("%-14s%-8sNumber of base pairs to progress window [%u]\n", "-stepsize", "INT", stepsize);
	printf("%-14s%-8sMinimum number of individuals in each population with data [%d]\n", "-minind", "INT", minind);
	printf("%-14s%-8s(1) Use fixed number of sites from MAF input for each window (window sizes may vary) or (0) constant window size [%d]\n",
	       "-fixedsite", "INT", fixedsite);
	printf("%-14s%-8sTwo-column TSV file with each row having (1) chromsome name (2) chromosome size in base pairs\n", "-sizefile", "FILE");
	printf("%-14s%-8sDo not print windows with zero effective sites if INT=1 [%d]\n", "-skip_missing", "INT", skip_missing);
	printf("\nNotes:\n"
	       "* -winsize 1 -stepsize 1 calculates per site dxy\n"
	       "* -sizefile is REQUIRED(!) with -fixedsite 0 (the default)\n"
	       "* Both input MAF files need to have the same chromosomes in the same order\n"
	       "* Assumes SNPs are biallelic across populations\n"
	       "* For global Dxy calculations only columns 4, 5, and 6 below are printed\n"
	       "* Input MAF files can contain all sites (including monomorphic sites) or just variable sites\n"
	       "* -fixedsite 1 -winsize 500 would for example ensure that all windows contain 500 SNPs\n"
	       "\nOutput:\n"
	       "(1) chromosome\n"
	       "(2) Window start\n"
	       "(3) Window end\n"
	       "(4) dxy\n"
	       "(5) number sites in MAF input that were analyzed\n"
	       "(6) number of sites in MAF input that were skipped due to too few individuals\n\n");
}

// One population's MAF as columns: n sites in file order; runs = maximal runs of equal chromosome name
// (a name may come back later as another run).  The columns are malloc'ed by parse_maf, or point into the
// mapping of a .pgtc cache.
struct Maf {
	uint64_t n = 0;
	const uint32_t* pos = nullptr;
	const double* freq = nullptr;
	const int32_t* nind = nullptr;
	std::vector<ContigRun> runs;
	void* owned[3] = {nullptr, nullptr, nullptr};
	~Maf() {
		for (void* p : owned) free(p);
	}
};

// tokenizeStr, dxyWindow.cpp:141-153: chr, unsigned pos, three single chars, double, int
static bool parse_maf_line(const char* p, const char* le, const char** name_b, const char** name_e, uint32_t* pos, double* f, int32_t* n) {
	const char* s = skip_ws(p, le);
	const char* t = token_end(s, le);
	if (t == s) return false;
	*name_b = s;
	*name_e = t;
	const char* cur = t;
	if (!parse_u32(cur, le, pos)) return false;
	for (int k = 0; k < 3; ++k) {  // `ss >> char` takes ONE non-blank character
		cur = skip_ws(cur, le);
		if (cur >= le) return false;
		++cur;
	}
	if (!parse_f64(cur, le, f)) return false;
	if (!parse_i32(cur, le, n)) return false;
	return true;
}

// The common MAF line `chr <b> pos <b> X <b> Y <b> Z <b> freq <b> nInd` with plain decimals, in one pass
// (pgt_cli.h fast_decimal: exact by Clinger's fast path); anything else returns false without side
// effects and goes through parse_maf_line.
static bool fast_maf_line(const char* p, const char* le, const char** name_b, const char** name_e, uint32_t* pos, double* f, int32_t* n) {
	const char* t = p;
	while (t < le && *t != ' ' && *t != '\t' && *t != '\r' && *t != '\v' && *t != '\f') ++t;
	if (t == p || t >= le) return false;
	const char* q = skip_blanks(t, le);
	uint64_t x = 0;
	int nd = 0;
	while (q < le && (unsigned)(*q - '0') <= 9u) {
		x = x * 10u + (unsigned)(*q - '0');
		++q;
		++nd;
	}
	if (nd == 0 || nd > 9) return false;
	for (int k = 0; k < 3; ++k) {  // three single-character columns
		if (q >= le || (*q != ' ' && *q != '\t')) return false;
		q = skip_blanks(q, le);
		if (q >= le || *q == '\r') return false;
		++q;
	}
	if (q >= le || (*q != ' ' && *q != '\t')) return false;
	q = skip_blanks(q, le);
	double fv;
	if (!fast_decimal(q, le, &fv)) return false;
	if (q >= le || (*q != ' ' && *q != '\t')) return false;
	q = skip_blanks(q, le);
	bool neg = false;
	if (q < le && *q == '-') {
		neg = true;
		++q;
	}
	uint32_t g = 0;
	int gd = 0;
	while (q < le && (unsigned)(*q - '0') <= 9u) {
		g = g * 10u + (unsigned)(*q - '0');
		++q;
		++gd;
	}
	if (gd == 0 || gd > 9) return false;
	if (q < le && *q != ' ' && *q != '\t' && *q != '\r') return false;
	*name_b = p;
	*name_e = t;
	*pos = (uint32_t)x;
	*f = fv;
	*n = neg ? -(int32_t)g : (int32_t)g;
	return true;
}

// read_input's verdict on one MAF file, worded as the reference words it
static int report_maf(int rc, const char* path, const char* which) {
	if (rc == -2) {  // the reference dies here with boost's gzip_error (dxyWindow.cpp:256-278): never print partial rows
		fprintf(stderr, "Corrupt or truncated gzip stream in %s MAF file: %s\n", which, path);
		return -1;
	}
	if (rc != 0) {
		fprintf(stderr, "Unable to open %s MAF file: %s\n", which, path);
		return -1;
	}
	return 0;
}

static int parse_maf(const Input& in, Maf* m, const char* path) {
	if (pgtcol::is_colfile(in.data, in.size)) {  // cached columns of one population
		pgtcol::View v;
		if (pgtcol::open_view_of(in.data, in.size, pgtcol::KIND_MAF, &v, "dxyWindow", path) != 0) return -1;
		m->n = v.nsites;  // the columns are the file mapping itself (`in` outlives the Maf)
		m->pos = (const uint32_t*)v.col[0];
		m->freq = (const double*)v.col[1];
		m->nind = (const int32_t*)v.col[2];
		m->runs = v.runs;
		return 0;
	}
	// skip the header line (dxyWindow.cpp:284), stop at the first empty line (:313)
	const char* nl = (const char*)memchr(in.data, '\n', in.size);
	size_t begin = nl ? (size_t)(nl + 1 - in.data) : in.size;
	size_t n_eff = begin + effective_size(in.data + begin, in.size - begin);
	const unsigned nt = (n_eff - begin) < parallel_min_bytes() ? 1 : parse_threads();
	uint64_t n = 0;
	std::vector<TextChunk> chunks = split_lines(in.data, begin, n_eff, nt, nt, &n);
	uint32_t* pos = (uint32_t*)malloc(std::max<uint64_t>(n, 1) * sizeof(uint32_t));
	double* freq = (double*)malloc(std::max<uint64_t>(n, 1) * sizeof(double));
	int32_t* nind = (int32_t*)malloc(std::max<uint64_t>(n, 1) * sizeof(int32_t));
	m->owned[0] = pos;
	m->owned[1] = freq;
	m->owned[2] = nind;
	if (!pos || !freq || !nind) {
		fprintf(stderr, "dxyWindow: out of memory for %llu sites of %s\n", (unsigned long long)n, path);
		return -1;
	}
	for_chunks(chunks, nt, [&](TextChunk& c, size_t) {
		const char* p = in.data + c.begin;
		const char* e = in.data + c.end;
		uint64_t row = c.row0;
		long li = 0;
		while (p < e) {
			const char* q = (const char*)memchr(p, '\n', (size_t)(e - p));
			const char* le = q ? q : e;
			const char *nb = nullptr, *ne = nullptr;
			uint32_t ps = 0;
			double f = 0;
			int32_t ni = 0;
			if (!fast_maf_line(p, le, &nb, &ne, &ps, &f, &ni) && !parse_maf_line(p, le, &nb, &ne, &ps, &f, &ni)) {
				if (c.bad_line < 0) c.bad_line = li;
				nb = ne = p;
			}
			c.add_row(nb, ne);
			pos[row] = ps;
			freq[row] = f;
			nind[row] = ni;
			++row;
			++li;
			if (!q) break;
			p = q + 1;
		}
	});
	const int64_t bad = merge_chunks(chunks, &m->runs);
	if (bad >= 0) {
		fprintf(stderr, "dxyWindow: cannot parse line %llu of %s\n", (unsigned long long)(2 + bad), path);
		return -1;
	}
	m->n = n;
	m->pos = pos;
	m->freq = freq;
	m->nind = nind;
	return 0;
}

int main(int argc, char** argv) {
	unsigned winsize = 0, stepsize = 0;  // dxyWindow.cpp:529-534
	int minind = 1, fixedsite = 0, skip_missing = 0;
	if (argc < 3) {
		help_info(winsize, stepsize, minind, fixedsite, skip_missing);
		return 0;  // parseArgs returns 1, main maps it to 0 (dxyWindow.cpp:537-538)
	}
	const double t_start = now_ms();
	Timing tm;
	tm.threads = parse_threads();
	// files are opened before the options are looked at (dxyWindow.cpp:73-95)
	Input in1, in2;
	Maf m1, m2;
	{
		// both files are read (and inflated) at the same time; Pop1's verdict is reported first, as the reference
		// opens Pop1 first (dxyWindow.cpp:73-95)
		int rc2 = 0;
		std::thread second([&]() { rc2 = read_input(argv[argc - 1], &in2, true); });
		const int rc1 = read_input(argv[argc - 2], &in1, true);
		second.join();
		if (report_maf(rc1, argv[argc - 2], "Pop1") != 0) return -1;
		if (report_maf(rc2, argv[argc - 1], "Pop2") != 0) return -1;
	}
	const char* sizefname = nullptr;
	bool have_sizefile = false;
	Input sizein;
	for (int argpos = 1; argpos < argc - 2; argpos += 2) {  // dxyWindow.cpp:97-126
		const char* o = argv[argpos];
		const char* v = argv[argpos + 1];
		if (strcmp(o, "-winsize") == 0) {
			int x = atoi(v);
			if (x < 0) {
				fprintf(stderr, "-winsize must not be negative\n");
				return -1;
			}
			winsize = (unsigned)x;
		} else if (strcmp(o, "-stepsize") == 0) {
			int x = atoi(v);
			stepsize = x < 0 ? 0u : (unsigned)x;
		} else if (strcmp(o, "-minind") == 0) {
			minind = atoi(v);
			if (minind <= 0) {
				fprintf(stderr, "-minind must be at least 1\n");
				return -1;
			}
		} else if (strcmp(o, "-sizefile") == 0) {
			sizefname = v;
			if (read_input(sizefname, &sizein, false) != 0) {
				fprintf(stderr, "Unable to open sizefile: %s\n", sizefname);
				return -1;
			}
			have_sizefile = true;
		} else if (strcmp(o, "-fixedsite") == 0) {
			fixedsite = atoi(v);
		} else if (strcmp(o, "-skip_missing") == 0) {
			skip_missing = atoi(v);
		} else {
			fprintf(stderr, "Unknown command: %s\n", o);
			return -1;
		}
	}
	if (winsize > 0 && stepsize < 1) {
		fprintf(stderr, "Must specify a -stepsize > 0 when -winsize is > 0\n");
		return -1;
	}
	// dxyWindow.cpp:133-136 tests `!sizefile` on a never-opened ifstream, which is false: the
	// "Must supply size file unless -fixedsite 1" branch is unreachable in the reference.  Without
	// -sizefile the size map is simply empty and the run ends with "Unable to determine size for X"
	// at the first chromosome end, which is what happens here too.
	(void)have_sizefile;
	if (winsize > 0 && stepsize > winsize) {
		fprintf(stderr, "-stepsize must not exceed -winsize\n");
		return -1;
	}
	if (winsize == 0 && !fixedsite) {
		fprintf(stderr, "-winsize 0 (global calculation) requires -fixedsite 1\n");
		return -1;
	}

	// parseSizes, dxyWindow.cpp:155-170 (first entry of a name wins: std::map::insert)
	std::map<std::string, unsigned> chrsize;
	if (!fixedsite) {
		const char* p = sizein.data;
		const char* e = sizein.data + sizein.size;
		while (p < e) {
			const char* q = (const char*)memchr(p, '\n', (size_t)(e - p));
			const char* le = q ? q : e;
			const char* s = skip_ws(p, le);
			const char* t = token_end(s, le);
			const char* cur = t;
			uint32_t len = 0;
			bool ok = t > s && parse_u32(cur, le, &len) && len > 0;
			if (!ok) {
				fprintf(stderr, "Unable to correctly parse chromosome size file\n");
				return -1;
			}
			chrsize.insert(std::make_pair(std::string(s, t), len));
			if (!q) break;
			p = q + 1;
		}
	}

	DeviceWarmup warm;
	const char* pack1 = getenv("PGT_PACK");
	const char* pack2 = getenv("PGT_PACK2");
	if (!pack1 && !pack2 && !getenv("PGT_PACK_SYNCED")) warm.start();
	if (parse_maf(in1, &m1, argv[argc - 2]) != 0) return -1;
	if (parse_maf(in2, &m2, argv[argc - 1]) != 0) return -1;
	if (pack1 || pack2) {  // write the binary columnar caches and stop: no GPU involved
		auto pack = [&](const char* path, const Maf& m) -> int {
			const void* cols[3] = {m.pos, m.freq, m.nind};
			if (pgtcol::write_file(path, pgtcol::KIND_MAF, m.runs, m.n, cols) != 0) {
				fprintf(stderr, "dxyWindow: cannot write %s\n", path);
				return -1;
			}
			return 0;
		};
		if (pack1 && pack(pack1, m1) != 0) return -1;
		if (pack2 && pack(pack2, m2) != 0) return -1;
		return 0;
	}
	const uint64_t n1 = m1.n, n2 = m2.n;
	if (n1 == 0 || n2 == 0) {
		fprintf(stderr, "dxyWindow: MAF file without data lines\n");
		return -1;
	}
	if (m1.runs[0].name != m2.runs[0].name) {  // dxyWindow.cpp:294-298
		fprintf(stderr, "Chromosomes in MAF files differ\n");
		return -1;
	}

	// ---- two-file sync, dxyWindow.cpp:313-331,399-403 ------------------------------------------
	// Chromosome names are compared as small integers (one id per distinct name over both files); each
	// file's cursor carries the run it is in, so there is no per-site chromosome column.
	const uint64_t ncap = std::min(n1, n2);
	std::unique_ptr<uint32_t[]> pos(new uint32_t[ncap]);
	std::unique_ptr<double[]> f1(new double[ncap]), f2(new double[ncap]);
	std::unique_ptr<int32_t[]> ni1(new int32_t[ncap]), ni2(new int32_t[ncap]);
	std::vector<ContigRun> runs;
	uint64_t n = 0;
	{
		std::map<std::string, uint32_t> ids;
		auto uids = [&](const std::vector<ContigRun>& rs) {
			std::vector<uint32_t> u;
			u.reserve(rs.size());
			for (const ContigRun& r : rs) u.push_back(ids.emplace(r.name, (uint32_t)ids.size()).first->second);
			return u;
		};
		const std::vector<uint32_t> u1 = uids(m1.runs), u2 = uids(m2.runs);
		uint64_t i1 = 0, i2 = 0;
		size_t r1 = 0, r2 = 0;                                  // run of site i1 / i2
		uint64_t e1 = m1.runs[0].count, e2 = m2.runs[0].count;  // end of that run
		auto fix1 = [&]() {
			while (i1 >= e1) e1 += m1.runs[++r1].count;
		};
		auto fix2 = [&]() {
			while (i2 >= e2) e2 += m2.runs[++r2].count;
		};
		uint32_t chr = u1[0];
		uint32_t last_uid = 0xffffffffu;
		const uint32_t *p1 = m1.pos, *p2 = m2.pos;
		for (;;) {
			fix1();
			fix2();
			if (p1[i1] != p2[i2] || u1[r1] != u2[r2]) {
				const bool samechr = u1[r1] == u2[r2];
				if ((samechr && p1[i1] < p2[i2]) || (!samechr && u2[r2] != chr)) {
					while (p1[i1] != p2[i2]) {  // catch maf1 up to maf2 (position-only compare)
						if (i1 + 1 >= n1) break;
						++i1;
					}
					if (p1[i1] != p2[i2]) break;
					fix1();
				} else {
					while (p2[i2] < p1[i1]) {
						if (i2 + 1 >= n2) break;
						++i2;
					}
					if (p1[i1] != p2[i2]) break;
					fix2();
				}
			}
			chr = u1[r1];
			if (chr != last_uid) {
				runs.push_back(ContigRun{m1.runs[r1].name, 0});
				last_uid = chr;
			}
			runs.back().count++;
			pos[n] = p1[i1];
			f1[n] = m1.freq[i1];
			f2[n] = m2.freq[i2];
			ni1[n] = m1.nind[i1];
			ni2[n] = m2.nind[i2];
			++n;
			if (++i1 >= n1) break;
			if (++i2 >= n2) break;
		}
	}
	tm.sites = n;
	tm.parse_ms = now_ms() - t_start;
	if (const char* synced = getenv("PGT_PACK_SYNCED")) {  // the synced site list as a kind-5 .pgtc, then stop (no GPU)
		const void* cols[5] = {pos.get(), f1.get(), f2.get(), ni1.get(), ni2.get()};
		if (pgtcol::write_file(synced, pgtcol::KIND_DXY, runs, n, cols) != 0) {
			fprintf(stderr, "dxyWindow: cannot write %s\n", synced);
			return -1;
		}
		return 0;
	}

	// ---- plan ---------------------------------------------------------------------------------
	const double t_scan = now_ms();
	std::vector<uint64_t> soff(runs.size() + 1, 0);
	for (size_t i = 0; i < runs.size(); ++i) soff[i + 1] = soff[i] + runs[i].count;
	uint32_t nchr = (uint32_t)runs.size();
	std::vector<uint64_t> axis = soff;  // plan axis: sites (-fixedsite 1) or bp (-fixedsite 0)
	const char* nosize = nullptr;       // first chromosome (data order) without a sizefile entry
	uint64_t print_limit = UINT64_MAX;  // bp mode with a missing size: windows whose last entry < limit
	uint64_t n_used = n;
	if (!fixedsite) {
		axis.assign(1, 0);
		for (uint32_t c = 0; c < nchr; ++c) {
			auto it = chrsize.find(runs[c].name);
			uint64_t L;
			if (it == chrsize.end()) {
				// dxyWindow.cpp:338-343,408-413: the reference has printed every window that flushed
				// before this chromosome ended, then fails.  Those are the windows completed by the
				// arrival of a later entry: last entry index <= (#entries so far) - 2.
				nosize = runs[c].name.c_str();
				L = pos[soff[c + 1] - 1];
				axis.push_back(axis.back() + L);
				print_limit = axis.back() - 1;
				nchr = c + 1;
				n_used = soff[c + 1];
				break;
			}
			L = it->second;
			axis.push_back(axis.back() + L);
		}
		for (uint32_t c = 0; c < nchr; ++c) {
			const uint64_t L = axis[c + 1] - axis[c];
			for (uint64_t i = soff[c]; i < soff[c + 1]; ++i) {
				if (pos[i] < 1 || pos[i] > L || (i > soff[c] && pos[i] <= pos[i - 1])) {
					fprintf(stderr, "dxyWindow: %s position %u (site %llu) is not strictly increasing within 1..%llu; bp windows need sorted positions inside the sizefile length\n",
					        runs[c].name.c_str(), pos[i], (unsigned long long)(i + 1), (unsigned long long)L);
					return -1;
				}
			}
		}
	}
	const unsigned W = winsize ? winsize : 1, S = winsize ? stepsize : 1;  // -winsize 0: only the global line is used
	pgt_plan* plan = nullptr;
	// bp mode: a reduction unit is a bp range; on sparse data (SNP-only MAFs) 256-bp units hold a handful
	// of sites each and the per-unit cost dominates, so the unit grows with the bp-per-site ratio
	// (measured on B200, 1e8 sites over 3e9 bp: 6.3 ms at 256 bp, 0.65 ms at 4096 bp).  The unit size
	// only changes the summation order (DESIGN.md section 4).
	uint32_t unit_sites = 0;
	if (!fixedsite && n_used > 0) {
		const double bp_per_site = (double)axis[nchr] / (double)n_used;
		if (bp_per_site >= 1.5) {
			const double u = 341.0 * bp_per_site;
			unit_sites = u >= 4096.0 ? 4096u : ((uint32_t)u + 31u) / 32u * 32u;
		}
	}
	if (pgt_plan_create(&plan, fixedsite ? PGT_MODE_SITES : PGT_MODE_BP, axis.data(), nchr, W, S, unit_sites) != PGT_OK) {
		fprintf(stderr, "%s\n", pgt_last_error());
		return -1;
	}
	const uint64_t nwin = pgt_plan_num_windows(plan);
	std::vector<uint32_t> label(nwin), startp(nwin), endp(nwin), neff(nwin), nskip(nwin);
	std::vector<double> dxy(nwin);
	double global[3] = {0, 0, 0};
	{
		if (warm.finish() != 0) return -1;
		tm.cuda_init_ms = warm.ms;
		pgt_columns cols;
		memset(&cols, 0, sizeof(cols));
		cols.pos = pos.get();
		cols.f1 = f1.get();
		cols.f2 = f2.get();
		cols.n1 = ni1.get();
		cols.n2 = ni2.get();
		pgt_windows out;
		memset(&out, 0, sizeof(out));
		out.label = label.data();
		out.start_pos = startp.data();
		out.end_pos = endp.data();
		out.dxy = dxy.data();
		out.neffective = neff.data();
		out.nskip = nskip.data();
		out.dxy_global = global;
		pgt_range range;
		memset(&range, 0, sizeof(range));
		range.w_hi = nwin;
		range.site_count = n_used;
		std::vector<uint64_t> soff_used(soff.begin(), soff.begin() + nchr + 1);
		// the synced columns go to the device through the pinned ring (pageable cudaMemcpy would run at a fifth of
		// the rate); two-file parsing and the sync are sequential in the site order, so there is nothing to overlap
		StreamColumn scol[5] = {{pos.get(), 4, 0, 0}, {f1.get(), 8, 0, 4}, {f2.get(), 8, 0, 5}, {ni1.get(), 4, 0, 6}, {ni2.get(), 4, 0, 7}};
		ColumnStreamer streamer;
		if (n_used > 0) streamer.start(&warm, scol, 5, n_used, nwin + 65536, 32, nullptr);
		streamer.rows_ready(0, n_used);
		int rc;
		if (streamer.finish(&tm) == 0) rc = streamer.scan(plan, PGT_STAT_DXY, &out, nwin, minind, &range, fixedsite ? nullptr : soff_used.data());
		// (n_used == soff_used[nchr]: the sharded call's "up to the end of the genome" is the same range)
		else rc = scan_on_devices(plan, &range, PGT_STAT_DXY, &cols, minind, fixedsite ? nullptr : soff_used.data(), &out);
		if (rc != PGT_OK) {
			fprintf(stderr, "dxyWindow: %s\n", pgt_last_error());
			return -1;
		}
	}
	tm.windows = nwin;
	tm.scan_ms = now_ms() - t_scan;

	// ---- print --------------------------------------------------------------------------------
	const double t_fmt = now_ms();
	static char obuf[1 << 20];
	setvbuf(stdout, obuf, _IOFBF, sizeof(obuf));
	if (winsize > 0) {
		std::vector<uint64_t> last_entry;
		if (nosize) {
			last_entry.resize(nwin);
			pgt_plan_windows(plan, nullptr, last_entry.data(), nullptr);
		}
		size_t maxname = 0;
		for (const ContigRun& r : runs) maxname = std::max(maxname, r.name.size());
		write_rows(stdout, nwin, maxname + 96, [&](char* p, uint64_t w) {
			if (skip_missing && neff[w] == 0) return p;        // dxyWindow.cpp:189
			if (nosize && last_entry[w] >= print_limit) return p;  // never flushed before the failure
			const std::string& nm = runs[label[w]].name;
			memcpy(p, nm.data(), nm.size());
			p += nm.size();
			*p++ = '\t';
			p = put_i32(p, (int32_t)startp[w]);
			*p++ = '\t';
			p = put_i32(p, (int32_t)endp[w]);
			*p++ = '\t';
			p = put_g(p, dxy[w]);
			*p++ = '\t';
			p = put_u32(p, neff[w]);
			*p++ = '\t';
			p = put_u32(p, nskip[w]);
			*p++ = '\n';
			return p;
		});
	}
	fflush(stdout);
	int rv = 0;
	if (nosize) {
		fprintf(stderr, "Unable to determine size for %s\n", nosize);
		rv = -1;
	} else {
		// dxyWindow.cpp:429-433
		char line[128];
		char* p = put_g(line, global[0]);
		*p++ = '\t';
		p = put_u32(p, (uint32_t)global[1]);
		*p++ = '\t';
		p = put_u32(p, (uint32_t)global[2]);
		*p++ = '\n';
		fwrite(line, 1, (size_t)(p - line), winsize == 0 ? stdout : stderr);
		fflush(stdout);
	}
	tm.format_ms = now_ms() - t_fmt;
	tm.total_ms = now_ms() - t_start;
	tm.report("dxyWindow");
	pgt_plan_destroy(plan);
	return rv;
}
