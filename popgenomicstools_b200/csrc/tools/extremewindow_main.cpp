// extremewindow_main.cpp -- drop-in `ihsWindow` (-DPGT_TOOL_IHS) and `xpehhWindow` (-DPGT_TOOL_XPEHH).
//
// Same argv grammar, defaults, usage text, messages, stdout/stderr split and exit codes as
//   /root/reference/ihsWindow.cpp:16-82,189-204   and   /root/reference/xpehhWindow.cpp:16-85,195-210
// The line loops (calciHSWindows ihsWindow.cpp:93-187, calcXpehhWindows xpehhWindow.cpp:87-193) are
// replaced by: parse the selscan .norm text into a position and a score column (multi-threaded),
// pgt_xplan_create for the window bookkeeping, pgt_scan_extreme (CUDA, PGT_MEM_HOST) for the
// per-window extreme / proportion, print the rows.
//
// Stream semantics kept from the reference's `ss >> ...` parsing:
//   * chromosome = locus id up to the first '_' (extractChr, ihsWindow.cpp:56-67); the position is the
//     2nd field, not the id's suffix (:119);
//   * a blank line re-counts the previous site (failed extractions leave locus, pos and scores unchanged);
//   * a line with too few numeric fields keeps the previous line's score (sitevec is reused, :101,120-123);
//     a non-numeric token in the score field reads as 0 (C++11 num_get stores 0 on failure);
//   * the first line of an XP-EHH file is a header and is skipped (xpehhWindow.cpp:110-115).
// Documented deviations (the reference has undefined behaviour or never terminates there):
//   * a site beyond its -chrlen length: the reference prints empty windows forever; here error, exit 255;
//   * a flag without a value (`-winsize` as last argument): the reference dereferences argv[argc]; here error;
//   * more than 6 (iHS) / 8 (XP-EHH) numeric fields after the position overflow the reference's vector;
//     extra fields are ignored here.
// Binary columnar cache (pgt_colfile.h): PGT_PACK=<out.pgtc> parses, writes the cache and exits
// without touching the GPU; a `.pgtc` file given as the input (magic sniff) skips the parsing.
// PGT_TIMING=1 prints parse / scan / format milliseconds to stderr; PGT_DEVICE, PGT_THREADS as in the other tools.
#include <map>

#include "../../../include/pgt_extreme.h"
#include "pgt_cli.h"
#include "pgt_colfile.h"

using namespace pgtcli;

#if defined(PGT_TOOL_IHS)
static const char* kTool = "ihsWindow";
static const int kScoreField = 4;  // sitevec[4], ihsWindow.cpp:160
#elif defined(PGT_TOOL_XPEHH)
static const char* kTool = "xpehhWindow";
static const int kScoreField = 6;  // sitevec[6], xpehhWindow.cpp:165
#else
#error "define PGT_TOOL_IHS or PGT_TOOL_XPEHH"
#endif

#if defined(PGT_TOOL_IHS)
// ihsWindow.cpp:16-33
static void info(unsigned winsize, double cutoff) {
	printf("\nUsage:\nihsWindow [selscan normalized iHS *.norm file] [options]\n"
	       "\nAssumes iHS locus ID in format chr*_position\n"
	       "\nOptions:\n"
	       "-winsize INT Window size (bp) [%u]\n"
	       "-cutoff FLOAT Determine fraction of sites with |iHS| > cutoff [%g]\n"
	       "-chrlen FILE TSV-file with columns (1) chr (2) chromosome length (bp), and each row is a different chromosome\n"
	       "\nOutput:\n"
	       "(1) chromosome\n"
	       "(2) window start\n"
	       "(3) window stop\n"
	       "(4) most extreme iHS score\n"
	       "(5) extreme iHS position\n"
	       "(6) proportion |iHS| > cutoff\n"
	       "(7) Number SNPs in window\n\n",
	       winsize, cutoff);
}
#else
// xpehhWindow.cpp:16-37
static void info(unsigned winsize) {
	printf("\nUsage:\nxpehhWindow <selscan normalized XPEHH *.norm file> <cutoff> [options]\n"
	       "\nInput file must have locus ID in format chr*_position\n"
	       "cutoff (FLOAT): Calculate proportion of sites with EXPEHH less (if negative) or greater (if positive) than cutoff\n"
	       "\nOptions:\n"
	       "-winsize INT Window size (bp) [%u]\n"
	       "-chrlen FILE TSV-file with columns (1) chr (2) chromosome length (bp), and each row is a different chromosome\n"
	       "\nOutput:\n"
	       "(1) chromosome\n"
	       "(2) window start\n"
	       "(3) window stop\n"
	       "(4) minimum (negative cutoff) or maximum (postive cutoff) XPEHH score\n"
	       "(5) extreme XPEHH position\n"
	       "(6) proportion XPEHH scores > or < cutoff\n"
	       "(7) Number SNPs in window\n\n",
	       winsize);
}
#endif

// `ss >> double` of libstdc++: digits / sign / '.' / exponent only -- "nan" and "inf" do not parse
static bool stream_f64(const char*& p, const char* e, double* v) {
	const char* s = skip_ws(p, e);
	const char* d = s;
	if (d < e && (*d == '+' || *d == '-')) ++d;
	if (d >= e || !((*d >= '0' && *d <= '9') || *d == '.')) return false;
	p = s;
	return parse_f64(p, e, v);
}

enum : uint8_t { ROW_OK = 0, ROW_STALE_SCORE = 1, ROW_BLANK = 2 };

static const char* kSame = "\x01";  // name of a chunk's first run when it continues the previous chunk's last run

int main(int argc, char** argv) {
	unsigned winsize = 100000;  // ihsWindow.cpp:194, xpehhWindow.cpp:199
	double cutoff = 2;          // ihsWindow.cpp:195
	const double t_start = now_ms();
#if defined(PGT_TOOL_IHS)
	if (argc < 2) {
		fprintf(stderr, "Must supply iHS input file\n");
		info(winsize, cutoff);
		return 1;
	}
	int argpos = 2;
#else
	if (argc < 3) {
		fprintf(stderr, "Must supply XPEHH file and cutoff value\n");
		info(winsize);
		return 1;
	}
	int argpos = 3;
#endif
	Input in;
	if (read_input(argv[1], &in, false) != 0) {
#if defined(PGT_TOOL_IHS)
		fprintf(stderr, "Unable to open iHS file %s\n", argv[1]);
#else
		fprintf(stderr, "Unable to open XPEHH inpt file %s\n", argv[1]);
#endif
		return -1;
	}
#if defined(PGT_TOOL_XPEHH)
	cutoff = atof(argv[2]);
	if (cutoff == 0) fprintf(stderr, "WARNING: cutoff value of zero will calculate proportion of non-negative XPEHH scores\n");
#endif
	Input lenfile;
	bool have_lenfile = false;
	while (argpos < argc) {
		const char* flag = argv[argpos];
		const bool known = strcmp(flag, "-winsize") == 0 || strcmp(flag, "-chrlen") == 0
#if defined(PGT_TOOL_IHS)
		                   || strcmp(flag, "-cutoff") == 0
#endif
		    ;
		if (!known) {
			fprintf(stderr, "Unknown argument %s\n", flag);
			return -1;
		}
		if (argpos + 1 >= argc) {
			fprintf(stderr, "Missing value for %s\n", flag);
			return -1;
		}
		const char* val = argv[argpos + 1];
		if (strcmp(flag, "-winsize") == 0) {
			winsize = (unsigned)atoi(val);  // unsigned in the reference: only 0 is rejected (ihsWindow.cpp:47-52)
			if (winsize == 0) {
				fprintf(stderr, "Window size must be a positive integer\n");
				return -1;
			}
		} else if (strcmp(flag, "-cutoff") == 0) {
			cutoff = atof(val);
			if (cutoff < 0) {
				fprintf(stderr, "|iHS| cutoff must be >= zero\n");
				return -1;
			}
		} else {
			if (read_input(val, &lenfile, false) != 0) {
				fprintf(stderr, "Unable to open chromosome length file %s\n", val);
				return -1;
			}
			have_lenfile = true;
		}
		argpos += 2;
	}

	// -chrlen table (setLengthMap, ihsWindow.cpp:86-95): `ss >> chr >> pos`, first entry of a name wins
	std::map<std::string, uint32_t> lenmap;
	if (have_lenfile) {
		const char* p = lenfile.data;
		const char* e = lenfile.data + lenfile.size;
		std::string chr;
		uint32_t len = 0;
		while (p < e) {
			const char* q = (const char*)memchr(p, '\n', (size_t)(e - p));
			const char* le = q ? q : e;
			const char* s = skip_ws(p, le);
			const char* t = token_end(s, le);
			if (t > s) {
				chr.assign(s, t);
				const char* cur = t;
				uint32_t v = 0;
				if (skip_ws(cur, le) < le) len = parse_u32(cur, le, &v) ? v : 0u;  // failed extraction stores 0
			}
			lenmap.insert(std::make_pair(chr, len));
			if (!q) break;
			p = q + 1;
		}
	}

	// ---- parse (timed separately from compute) --------------------------------------------
	Timing tm;
	DeviceWarmup warm;
	const char* pack_path = getenv("PGT_PACK");
	if (!pack_path) warm.start();
	pgtcol::View view;
	const bool columnar = pgtcol::is_colfile(in.data, in.size);
	if (columnar && pgtcol::open_view_of(in.data, in.size, pgtcol::KIND_SCORE, &view, kTool, argv[1]) != 0) return -1;
	size_t begin = 0;
#if defined(PGT_TOOL_XPEHH)
	if (!columnar) {  // skip header (xpehhWindow.cpp:110-115)
		const char* nl = in.size ? (const char*)memchr(in.data, '\n', in.size) : nullptr;
		if (!nl) {
			fprintf(stderr, "Input XPEHH file had zero sites\n");
			return 0;
		}
		begin = (size_t)(nl + 1 - in.data);
	}
#endif
	const size_t text_end = columnar ? begin : in.size;  // columnar input: nothing to parse
	const unsigned nt = (text_end - begin) < parallel_min_bytes() ? 1 : parse_threads();
	tm.threads = nt;
	uint64_t n = 0;
	std::vector<TextChunk> chunks = split_lines(in.data, begin, text_end, nt, nt, &n);
	if (columnar) n = view.nsites;
	uint32_t* pos = columnar ? (uint32_t*)view.col[0] : (uint32_t*)malloc(std::max<uint64_t>(n, 1) * sizeof(uint32_t));
	double* score = columnar ? (double*)view.col[1] : (double*)malloc(std::max<uint64_t>(n, 1) * sizeof(double));
	if (!pos || !score) {
		fprintf(stderr, "%s: out of memory for %llu sites\n", kTool, (unsigned long long)n);
		return -1;
	}
	// Values a row inherits from the row before it (stream semantics above) are copied on the spot, unless that
	// row is itself still waiting for the previous CHUNK's last row: the dependency is then recorded in the
	// chunk's head_fix and resolved in row order after all chunks are parsed.
	std::vector<std::vector<std::pair<uint64_t, uint8_t>>> head_fix(chunks.size());
	for_chunks(chunks, nt, [&](TextChunk& c, size_t ci) {
		const char* p = in.data + c.begin;
		const char* e = in.data + c.end;
		uint64_t row = c.row0;
		bool pend_pos = true, pend_score = true;  // "row - 1 is unresolved": true at the chunk head
		while (p < e) {
			const char* q = (const char*)memchr(p, '\n', (size_t)(e - p));
			const char* le = q ? q : e;
			const char* s = skip_ws(p, le);
			const char* t = token_end(s, le);
			const bool have_prev = row > c.row0;
			if (t == s) {  // blank line: every extraction fails, the previous site is counted again
				if (!pend_pos && !pend_score) {
					pos[row] = pos[row - 1];
					score[row] = score[row - 1];
				} else {
					head_fix[ci].emplace_back(row, ROW_BLANK);
					pend_pos = pend_score = true;
				}
				if (have_prev) c.runs.back().count++;
				else c.runs.push_back(ContigRun{kSame, 1});
			} else {
				const char* us = (const char*)memchr(s, '_', (size_t)(t - s));
				const char* ne = us ? us : t;  // extractChr
				const char* cur = t;
				uint32_t pv = 0;
				bool ok = true;
				bool deferred = false;
				if (skip_ws(cur, le) >= le) {  // no position field: pos and scores stay
					ok = false;
					if (!pend_pos && !pend_score) {
						pos[row] = pos[row - 1];
					} else {
						pos[row] = 0;
						head_fix[ci].emplace_back(row, ROW_BLANK);  // takes pos and score of the previous row
						deferred = true;
						pend_pos = pend_score = true;
					}
				} else if (!parse_u32(cur, le, &pv)) {
					pos[row] = 0;  // failed numeric extraction stores 0 and fails the stream
					ok = false;
					pend_pos = false;
				} else {
					pos[row] = pv;
					pend_pos = false;
				}
				uint8_t st = ROW_STALE_SCORE;
				double v = 0;
				if (ok) {
					for (int k = 0; k <= kScoreField; ++k) {
						if (skip_ws(cur, le) >= le) break;  // out of tokens: later fields stay
						if (!stream_f64(cur, le, &v)) {
							if (k == kScoreField) {  // the score token itself does not parse: 0 is stored
								v = 0;
								st = ROW_OK;
							}
							break;
						}
						if (k == kScoreField) st = ROW_OK;
					}
				}
				if (st == ROW_OK) {
					score[row] = v;
					pend_score = false;
				} else if (!deferred) {
					if (!pend_score) {
						score[row] = score[row - 1];
					} else {
						head_fix[ci].emplace_back(row, ROW_STALE_SCORE);
						pend_score = true;
					}
				}
				c.add_row(s, ne);
			}
			++row;
			if (!q) break;
			p = q + 1;
		}
	});
	// rows at a chunk head that repeat the previous chunk's last row (sequential, rare)
	std::vector<ContigRun> runs;
	if (columnar) runs = view.runs;
	for (size_t ci = 0; ci < chunks.size(); ++ci) {
		for (auto& fx : head_fix[ci]) {
			const uint64_t r = fx.first;
			if (fx.second == ROW_BLANK) pos[r] = r ? pos[r - 1] : 0u;
			score[r] = r ? score[r - 1] : 0.0;
		}
		for (const ContigRun& r : chunks[ci].runs) {
			if (r.name == kSame) {
				if (runs.empty()) runs.push_back(ContigRun{std::string(), r.count});
				else runs.back().count += r.count;
			} else if (!runs.empty() && runs.back().name == r.name) {
				runs.back().count += r.count;
			} else {
				runs.push_back(r);
			}
		}
	}
	tm.sites = n;
	tm.parse_ms = now_ms() - t_start;
	if (pack_path) {  // write the binary columnar cache and stop: no GPU involved
		const void* cols[2] = {pos, score};
		if (pgtcol::write_file(pack_path, pgtcol::KIND_SCORE, runs, n, cols) != 0) {
			fprintf(stderr, "%s: cannot write %s\n", kTool, pack_path);
			return -1;
		}
		tm.total_ms = now_ms() - t_start;
		tm.report(kTool);
		return 0;
	}
	static char obuf[1 << 20];
	setvbuf(stdout, obuf, _IOFBF, sizeof(obuf));
	if (n == 0) {
		// the reference still prints its open window, with an empty name (ihsWindow.cpp:180)
		printf("\t1\t%u\tNA\tNA\tNA\t0\n", 1u + (winsize - 1u));
		fflush(stdout);
		tm.total_ms = now_ms() - t_start;
		tm.report(kTool);
		return 0;
	}

	// ---- window bookkeeping + scan (libpgtscan) ------------------------------------------------
	const double t_scan = now_ms();
	std::vector<uint64_t> off(runs.size() + 1, 0);
	std::vector<uint32_t> clen(runs.size(), 0);
	for (size_t i = 0; i < runs.size(); ++i) {
		off[i + 1] = off[i] + runs[i].count;
		auto it = lenmap.find(runs[i].name);
		if (it != lenmap.end()) clen[i] = it->second;
	}
	pgt_xplan* plan = nullptr;
	if (pgt_xplan_create(&plan, pos, off.data(), lenmap.empty() ? nullptr : clen.data(), (uint32_t)runs.size(), winsize, 0) != PGT_OK) {
		fprintf(stderr, "%s: %s\n", kTool, pgt_last_error());
		return -1;
	}
	const uint64_t nwin = pgt_xplan_num_windows(plan);
	std::vector<uint32_t> label(nwin), startp(nwin), endp(nwin), cnt(nwin), extpos(nwin);
	std::vector<double> ext(nwin), prop(nwin);
	pgt_xplan_windows(plan, label.data(), startp.data(), endp.data(), nullptr, nullptr);
	{
		if (warm.finish() != 0) return -1;
		tm.cuda_init_ms = warm.ms;
		pgt_xwindows out;
		memset(&out, 0, sizeof(out));
		out.ext_value = ext.data();
		out.ext_pos = extpos.data();
		out.prop = prop.data();
		out.nsites = cnt.data();
#if defined(PGT_TOOL_IHS)
		const pgt_xstat which = PGT_XSTAT_IHS;
#else
		const pgt_xstat which = PGT_XSTAT_XPEHH;
#endif
		const std::vector<int>& devs = device_list();
		DeviceWorkspace ws;
		int rc;
		if (devs.size() > 1) {  // PGT_DEVICES: one shard of windows per GPU, same table
			rc = pgt_scan_extreme_sharded(plan, which, cutoff, pos, score, &out, devs.data(), (uint32_t)devs.size());
		} else {
			ws.bytes = pgt_scan_extreme_workspace_bytes(plan, nullptr, PGT_MEM_HOST);
			rc = pgt_device_alloc(&ws.p, ws.bytes);
			if (rc == PGT_OK) rc = pgt_scan_extreme(plan, nullptr, which, cutoff, pos, score, &out, ws.p, ws.bytes, PGT_MEM_HOST, nullptr);
		}
		if (rc != PGT_OK) {
			fprintf(stderr, "%s: %s\n", kTool, pgt_last_error());
			return -1;
		}
	}
	tm.windows = nwin;
	tm.scan_ms = now_ms() - t_scan;

	// ---- print (printWindow, ihsWindow.cpp:75-84) ------------------------------------------------
	const double t_fmt = now_ms();
	size_t maxname = 0;
	for (const ContigRun& r : runs) maxname = std::max(maxname, r.name.size());
	write_rows(stdout, nwin, maxname + 128, [&](char* p, uint64_t w) {
		const std::string& nm = runs[label[w]].name;
		memcpy(p, nm.data(), nm.size());
		p += nm.size();
		*p++ = '\t';
		p = put_u32(p, startp[w]);
		*p++ = '\t';
		p = put_u32(p, endp[w]);
		*p++ = '\t';
		if (cnt[w] > 0) {
			p = put_g(p, ext[w]);
			*p++ = '\t';
			p = put_u32(p, extpos[w]);
			*p++ = '\t';
			p = put_g(p, prop[w]);
			*p++ = '\t';
			p = put_u32(p, cnt[w]);
			*p++ = '\n';
		} else {
			memcpy(p, "NA\tNA\tNA\t0\n", 11);
			p += 11;
		}
		return p;
	});
	fflush(stdout);
	tm.format_ms = now_ms() - t_fmt;
	tm.total_ms = now_ms() - t_start;
	tm.report(kTool);
	pgt_xplan_destroy(plan);
	return 0;
}
