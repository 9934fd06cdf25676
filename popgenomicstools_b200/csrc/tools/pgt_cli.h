// pgt_cli.h -- host plumbing shared by the drop-in CLIs (fstWindow, hetWindow, dxyWindow):
// whole-file input (mmap, or zlib inflate for .gz), multi-threaded line parsing with
// std::from_chars (correctly rounded like libstdc++'s num_get -> strtod that the reference
// uses, /root/reference/fstWindow.cpp:141), contig run-length bookkeeping, %g output
// formatting (the reference prints doubles with default ostream settings == printf("%g"),
// fstWindow.cpp:88) and the timing report.  No arithmetic of the hot path happens here: the
// columns go to libpgtscan.so (pgt_scan, PGT_MEM_HOST).
#ifndef PGT_CLI_H
#define PGT_CLI_H

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <charconv>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/pgt_scan.h"

namespace pgtcli {

inline double now_ms() {
	using namespace std::chrono;
	return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// ---- input -----------------------------------------------------------------------------

struct Input {
	const char* data = nullptr;
	size_t size = 0;
	void* map = nullptr;
	size_t map_size = 0;
	std::vector<char> owned;
	char* heap = nullptr;  // inflated BGZF input (malloc: a vector would zero gigabytes on one thread first)
	~Input() {
		if (map) munmap(map, map_size);
		free(heap);
	}
};

inline unsigned parse_threads() {
	const char* env = getenv("PGT_THREADS");
	unsigned n = env ? (unsigned)atoi(env) : std::thread::hardware_concurrency();
	if (n < 1) n = 1;
	if (n > 64) n = 64;
	return n;
}

// BGZF (bgzip / htslib -- what ANGSD writes its .mafs.gz with): a series of independent gzip members of at most
// 64 KB, each carrying its own compressed size in a 'BC' extra subfield (SAM spec 4.1) and its uncompressed size in
// the trailer.  That makes the output offset of every member known up front, so members inflate in parallel.
struct BgzfBlock {
	size_t in_off;     // first byte of the raw deflate data
	uint32_t in_len;   // bytes of deflate data
	uint32_t out_len;  // ISIZE
	uint32_t crc;      // CRC32 of the uncompressed bytes
	size_t out_off;
};
// true when [d, d + n) is nothing but well-formed BGZF members
inline bool bgzf_index(const unsigned char* d, size_t n, std::vector<BgzfBlock>* blocks, size_t* total) {
	auto u16 = [&](size_t o) { return (uint32_t)d[o] | ((uint32_t)d[o + 1] << 8); };
	auto u32 = [&](size_t o) { return u16(o) | (u16(o + 2) << 16); };
	size_t o = 0, out = 0;
	while (o < n) {
		if (n - o < 18 + 8 || d[o] != 0x1f || d[o + 1] != 0x8b || d[o + 2] != 8 || d[o + 3] != 4) return false;  // FEXTRA only
		const size_t xlen = u16(o + 10);
		if (n - o < 12 + xlen + 8) return false;
		size_t bsize = 0;
		for (size_t x = o + 12; x + 4 <= o + 12 + xlen;) {
			const size_t slen = u16(x + 2);
			if (d[x] == 'B' && d[x + 1] == 'C' && slen == 2 && x + 6 <= o + 12 + xlen) bsize = (size_t)u16(x + 4) + 1;
			x += 4 + slen;
		}
		if (bsize < 12 + xlen + 8 || bsize > n - o) return false;
		BgzfBlock b;
		b.in_off = o + 12 + xlen;
		b.in_len = (uint32_t)(bsize - 12 - xlen - 8);
		b.crc = u32(o + bsize - 8);
		b.out_len = u32(o + bsize - 4);
		if (b.out_len > (1u << 16)) return false;
		b.out_off = out;
		out += b.out_len;
		blocks->push_back(b);
		o += bsize;
	}
	*total = out;
	return true;
}
// 0 ok, -2 a member does not inflate to its declared size / checksum, -1 out of memory
inline int bgzf_inflate_parallel(const unsigned char* d, const std::vector<BgzfBlock>& blocks, char* out, unsigned nt) {
	std::atomic<size_t> next{0};
	std::atomic<int> status{0};
	auto work = [&]() {
		z_stream zs;
		memset(&zs, 0, sizeof(zs));
		if (inflateInit2(&zs, -15) != Z_OK) {
			status = -1;
			return;
		}
		for (;;) {
			const size_t b0 = next.fetch_add(64);  // 64 members (<= 4 MB of text) per grab
			if (b0 >= blocks.size() || status.load() != 0) break;
			const size_t b1 = std::min(blocks.size(), b0 + 64);
			for (size_t i = b0; i < b1; ++i) {
				const BgzfBlock& b = blocks[i];
				inflateReset(&zs);
				zs.next_in = (Bytef*)(d + b.in_off);
				zs.avail_in = b.in_len;
				zs.next_out = (Bytef*)(out + b.out_off);
				zs.avail_out = b.out_len;
				const int rc = inflate(&zs, Z_FINISH);
				if (rc != Z_STREAM_END || zs.avail_out != 0 || zs.avail_in != 0 ||
				    (uint32_t)crc32(crc32(0L, Z_NULL, 0), (const Bytef*)(out + b.out_off), b.out_len) != b.crc) {
					status = -2;
					break;
				}
			}
		}
		inflateEnd(&zs);
	};
	std::vector<std::thread> th;
	for (unsigned t = 1; t < nt; ++t) th.emplace_back(work);
	work();
	for (auto& t : th) t.join();
	return status.load();
}

// 0 ok, -1 cannot open, -2 corrupt or truncated gzip stream (the reference aborts there with boost's
// gzip_error, dxyWindow.cpp:256-278; partial rows must never be presented as a complete result)
inline int read_input(const char* path, Input* in, bool allow_gzip) {
	int fd = open(path, O_RDONLY);
	if (fd < 0) return -1;
	struct stat st;
	if (fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) {
		// pipes / process substitution: slurp
		std::vector<char> buf;
		char tmp[1 << 16];
		ssize_t k;
		while ((k = read(fd, tmp, sizeof(tmp))) > 0) buf.insert(buf.end(), tmp, tmp + k);
		close(fd);
		in->owned.swap(buf);
		in->data = in->owned.data();
		in->size = in->owned.size();
	} else {
		in->size = (size_t)st.st_size;
		if (in->size) {
			in->map = mmap(nullptr, in->size, PROT_READ, MAP_PRIVATE, fd, 0);
			if (in->map == MAP_FAILED) {
				in->map = nullptr;
				close(fd);
				return -1;
			}
			in->map_size = in->size;
			madvise(in->map, in->size, MADV_SEQUENTIAL);  // advice values are an enumeration, not flags: one call each
			madvise(in->map, in->size, MADV_WILLNEED);
			in->data = (const char*)in->map;
		}
		close(fd);
	}
	// gzip magic sniff as the reference does (dxyWindow.cpp:82-83)
	if (allow_gzip && in->size >= 2 && (unsigned char)in->data[0] == 0x1f && (unsigned char)in->data[1] == 0x8b) {
		{
			std::vector<BgzfBlock> blocks;
			size_t total = 0;
			const unsigned nt = parse_threads();
			const char* off = getenv("PGT_BGZF_PARALLEL");  // "0": always the serial zlib stream
			if (!(off && off[0] == '0') && bgzf_index((const unsigned char*)in->data, in->size, &blocks, &total) && blocks.size() >= 2) {
				char* out = (char*)malloc(std::max<size_t>(total, 1));
				if (!out) return -1;
				const int rc = bgzf_inflate_parallel((const unsigned char*)in->data, blocks, out, std::min<size_t>(nt, (blocks.size() + 63) / 64));
				if (rc != 0) {
					free(out);
					return rc;
				}
				if (in->map) munmap(in->map, in->map_size);
				in->map = nullptr;
				std::vector<char>().swap(in->owned);
				in->heap = out;
				in->data = out;
				in->size = total;
				return 0;
			}
		}
		std::vector<char> out;
		out.resize(std::max<size_t>(in->size * 4, 1 << 16));
		z_stream zs;
		memset(&zs, 0, sizeof(zs));
		if (inflateInit2(&zs, 15 + 32) != Z_OK) return -1;
		zs.next_in = (Bytef*)in->data;
		size_t in_left = in->size, produced = 0;
		bool complete = false;  // the last member ended with Z_STREAM_END and no input is left
		for (;;) {
			if (zs.avail_in == 0 && in_left) {
				uInt c = (uInt)std::min<size_t>(in_left, 1u << 30);
				zs.avail_in = c;
				in_left -= c;
			}
			if (out.size() - produced < (1 << 16)) out.resize(out.size() * 2);
			zs.next_out = (Bytef*)out.data() + produced;
			uInt room = (uInt)std::min<size_t>(out.size() - produced, 1u << 30);
			zs.avail_out = room;
			int rc = inflate(&zs, Z_NO_FLUSH);
			produced += room - zs.avail_out;
			if (rc == Z_STREAM_END) {
				if (zs.avail_in == 0 && in_left == 0) {
					complete = true;
					break;
				}
				inflateReset(&zs);  // concatenated members (bgzip)
			} else if (rc != Z_OK && rc != Z_BUF_ERROR) {
				break;
			} else if (rc == Z_BUF_ERROR && zs.avail_in == 0 && in_left == 0) {
				break;
			}
		}
		inflateEnd(&zs);
		if (!complete) return -2;
		out.resize(produced);
		if (in->map) munmap(in->map, in->map_size);
		in->map = nullptr;
		in->owned.swap(out);
		in->data = in->owned.data();
		in->size = in->owned.size();
	}
	return 0;
}

// ---- tokenising ------------------------------------------------------------------------

inline bool is_ws(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f'; }

inline const char* skip_ws(const char* p, const char* e) {
	while (p < e && is_ws(*p)) ++p;
	return p;
}
inline const char* token_end(const char* p, const char* e) {
	while (p < e && !is_ws(*p)) ++p;
	return p;
}

// `ss >> unsigned int` (optional sign, digits)
inline bool parse_u32(const char*& p, const char* e, uint32_t* v) {
	p = skip_ws(p, e);
	bool neg = false;
	if (p < e && (*p == '+' || *p == '-')) neg = (*p++ == '-');
	uint64_t x = 0;
	auto r = std::from_chars(p, e, x);
	if (r.ec != std::errc() || r.ptr == p) return false;
	p = r.ptr;
	if (x > 0xffffffffull) x = 0xffffffffull;
	*v = neg ? (uint32_t)(0u - (uint32_t)x) : (uint32_t)x;
	return true;
}
inline bool parse_i32(const char*& p, const char* e, int32_t* v) {
	p = skip_ws(p, e);
	bool neg = false;
	if (p < e && (*p == '+' || *p == '-')) neg = (*p++ == '-');
	uint64_t x = 0;
	auto r = std::from_chars(p, e, x);
	if (r.ec != std::errc() || r.ptr == p) return false;
	p = r.ptr;
	if (x > 0x7fffffffull) x = 0x7fffffffull;
	*v = neg ? -(int32_t)x : (int32_t)x;
	return true;
}
inline bool parse_f64(const char*& p, const char* e, double* v) {
	p = skip_ws(p, e);
	if (p < e && *p == '+') ++p;
	auto r = std::from_chars(p, e, *v, std::chars_format::general);
	if (r.ec == std::errc::result_out_of_range) {
		// strtod semantics: +-HUGE_VAL or (sub)zero; let strtod decide
		std::string tmp(p, r.ptr);
		*v = strtod(tmp.c_str(), nullptr);
		p = r.ptr;
		return true;
	}
	if (r.ec != std::errc() || r.ptr == p) return false;
	p = r.ptr;
	return true;
}

// ---- single-pass fast path for the common line shape -----------------------------------------
//
// `name <blanks> digits <blanks> number [<blanks> number] [\r]\n` with plain decimals: one pass over
// the bytes, no separate search for the line end.  Exactness: <= 9 position digits fit uint32
// arithmetic checked against 2^32; a decimal with <= 15 digits in total is m / 10^f with m < 2^53
// and 10^f exact, and ONE IEEE division of two exact doubles is the correctly rounded value of the
// string -- the double strtod / std::from_chars return (Clinger's fast path).  Anything else (signs
// on the position, exponents, more digits, inf/nan, missing fields, other white space) makes the
// function return false WITHOUT side effects and the caller parses that line the general way.
inline bool fast_decimal(const char*& p, const char* e, double* v) {
	static const double kPow10[16] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15};
	const char* q = p;
	bool neg = false;
	if (q < e && *q == '-') {
		neg = true;
		++q;
	}
	uint64_t m = 0;
	int nd = 0;
	while (q < e && (unsigned)(*q - '0') <= 9u) {
		m = m * 10u + (unsigned)(*q - '0');
		++q;
		++nd;
	}
	int frac = 0;
	if (q < e && *q == '.') {
		++q;
		const char* f0 = q;
		while (q < e && (unsigned)(*q - '0') <= 9u) {
			m = m * 10u + (unsigned)(*q - '0');
			++q;
		}
		frac = (int)(q - f0);
		nd += frac;
	}
	if (nd == 0 || nd > 15) return false;
	if (q < e && *q != ' ' && *q != '\t' && *q != '\n' && *q != '\r') return false;  // exponent, letters, ...
	const double r = (double)m / kPow10[frac];
	*v = neg ? -r : r;
	p = q;
	return true;
}
inline const char* skip_blanks(const char* p, const char* e) {
	while (p < e && (*p == ' ' || *p == '\t')) ++p;
	return p;
}
// On success: [*name_b, *name_e) = first token, *pos, vals[0..nvals), *next = first byte of the next line.
template <int NVALS, bool INTVALS>
inline bool fast_line(const char* p, const char* e, const char** name_b, const char** name_e, uint32_t* pos, double* vals, int32_t* ivals,
                      const char** next) {
	const char* s = p;
	const char* t = s;
	while (t < e && *t != ' ' && *t != '\t' && *t != '\n' && *t != '\r' && *t != '\v' && *t != '\f') ++t;
	if (t == s || t >= e || (*t != ' ' && *t != '\t')) return false;
	const char* q = skip_blanks(t, e);
	uint64_t x = 0;
	int nd = 0;
	while (q < e && (unsigned)(*q - '0') <= 9u) {
		x = x * 10u + (unsigned)(*q - '0');
		++q;
		++nd;
	}
	if (nd == 0 || nd > 9 || q >= e || (*q != ' ' && *q != '\t')) return false;
	double dv[NVALS > 0 ? NVALS : 1];
	int32_t iv[NVALS > 0 ? NVALS : 1];
	for (int k = 0; k < NVALS; ++k) {
		q = skip_blanks(q, e);
		if (INTVALS) {
			bool neg = false;
			if (q < e && *q == '-') {
				neg = true;
				++q;
			}
			uint32_t g = 0;
			int gd = 0;
			while (q < e && (unsigned)(*q - '0') <= 9u) {
				g = g * 10u + (unsigned)(*q - '0');
				++q;
				++gd;
			}
			if (gd == 0 || gd > 9) return false;
			if (q < e && *q != ' ' && *q != '\t' && *q != '\n' && *q != '\r') return false;
			iv[k] = neg ? -(int32_t)g : (int32_t)g;
		} else if (!fast_decimal(q, e, &dv[k])) {
			return false;
		}
	}
	q = skip_blanks(q, e);
	if (q < e && *q == '\r') ++q;
	if (q < e && *q != '\n') return false;  // extra fields: let the general path decide
	*name_b = s;
	*name_e = t;
	*pos = (uint32_t)x;
	for (int k = 0; k < NVALS; ++k) {
		if (INTVALS) ivals[k] = iv[k];
		else vals[k] = dv[k];
	}
	*next = q < e ? q + 1 : e;
	return true;
}

// ---- line-chunked parallel parsing ------------------------------------------------------

struct ContigRun {
	std::string name;
	uint64_t count;
};

// inputs smaller than this are parsed on one thread (PGT_PARALLEL_MIN_BYTES overrides: the tests
// use 1 to push tiny fuzzed files through the multi-chunk path)
inline size_t parallel_min_bytes() {
	const char* env = getenv("PGT_PARALLEL_MIN_BYTES");
	return env ? (size_t)strtoull(env, nullptr, 10) : (size_t)(1u << 20);
}

// The reference stops at the first EMPTY line (fstWindow.cpp:125 `while (!sitedata.empty())`): the
// bytes before it, i.e. up to and including the '\n' that is followed by another '\n'.
// first_empty_line: smallest q in [lo, hi) with d[q] == d[q+1] == '\n' (q + 1 < n), or n
inline size_t first_empty_line(const char* d, size_t n, size_t lo, size_t hi) {
	const char* p = d + lo;
	const char* e = d + hi;
	while (p < e) {
		const char* q = (const char*)memchr(p, '\n', (size_t)(e - p));
		if (!q) break;
		if (q + 1 < d + n && q[1] == '\n') return (size_t)(q - d);
		p = q + 1;
	}
	return n;
}
// One pass over the whole text, so it runs on all parser threads (byte ranges; a pair is found by
// the range that holds its first '\n'): serial it was 0.3-0.45 s of a 0.6 s parse at 48 M lines.
inline size_t effective_size(const char* d, size_t n) {
	if (n == 0 || d[0] == '\n') return 0;
	const unsigned nt = n < parallel_min_bytes() ? 1 : parse_threads();
	size_t q = n;
	if (nt == 1) {
		q = first_empty_line(d, n, 0, n);
	} else {
		std::vector<size_t> hit(nt, n);
		std::vector<std::thread> th;
		for (unsigned t = 0; t < nt; ++t)
			th.emplace_back([&, t]() { hit[t] = first_empty_line(d, n, (size_t)((unsigned __int128)n * t / nt), (size_t)((unsigned __int128)n * (t + 1) / nt)); });
		for (auto& x : th) x.join();
		for (unsigned t = 0; t < nt; ++t) q = std::min(q, hit[t]);
	}
	return q < n ? q + 1 : n;
}

// A line-aligned byte range of the text.  Its lines are counted first, so that its parser thread writes rows
// [row0, row0 + nlines) straight into the final columns: no per-chunk vectors and no serial concatenation (that
// was 100 of 170 ms per 3 M-line MAF on 8 threads).
struct TextChunk {
	size_t begin = 0, end = 0;  // byte range
	uint64_t nlines = 0;        // lines in the range (a last line without '\n' counts)
	uint64_t row0 = 0;          // first output row
	std::vector<ContigRun> runs;
	long bad_line = -1;         // chunk-local index of the first malformed line

	// the next row's contig name is [s, e): it extends the last run or starts a new one
	void add_row(const char* s, const char* e) {
		const size_t len = (size_t)(e - s);
		if (runs.empty() || runs.back().name.size() != len || memcmp(runs.back().name.data(), s, len) != 0)
			runs.push_back(ContigRun{std::string(s, e), 0});
		runs.back().count++;
	}
};

// run `fn(chunk, index)` over all chunks on nt threads (the calling thread is one of them), chunks taken in file order
template <class Fn>
inline void for_chunks(std::vector<TextChunk>& chunks, unsigned nt, Fn fn) {
	std::atomic<size_t> next{0};
	auto worker = [&]() {
		for (size_t i = next++; i < chunks.size(); i = next++) fn(chunks[i], i);
	};
	std::vector<std::thread> th;
	for (unsigned t = 1; t < nt && t < chunks.size(); ++t) th.emplace_back(worker);
	worker();
	for (auto& x : th) x.join();
}

// [begin, end) of d cut at line starts into at most nchunks chunks (at least one), their lines counted on nt threads
// and row0 set; *nrows = the lines of all chunks
inline std::vector<TextChunk> split_lines(const char* d, size_t begin, size_t end, unsigned nchunks, unsigned nt, uint64_t* nrows) {
	std::vector<TextChunk> chunks(1);
	chunks[0].begin = begin;
	for (unsigned t = 1; t < nchunks; ++t) {
		const size_t guess = begin + (end - begin) / nchunks * t;
		if (guess <= chunks.back().begin) continue;
		const char* q = (const char*)memchr(d + guess, '\n', end - guess);
		if (!q) break;
		const size_t s = (size_t)(q + 1 - d);
		if (s > chunks.back().begin && s < end) {
			chunks.back().end = s;
			chunks.emplace_back();
			chunks.back().begin = s;
		}
	}
	chunks.back().end = end;
	for_chunks(chunks, nt, [d](TextChunk& c, size_t) {
		for (const char *p = d + c.begin, *e = d + c.end; p < e; ++c.nlines) {
			const char* q = (const char*)memchr(p, '\n', (size_t)(e - p));
			p = q ? q + 1 : e;
		}
	});
	uint64_t n = 0;
	for (TextChunk& c : chunks) {
		c.row0 = n;
		n += c.nlines;
	}
	*nrows = n;
	return chunks;
}

// Appends the chunks' runs to *runs in file order (a run cut by a chunk boundary becomes one again).  Returns the row
// of the first malformed line in file order, or -1 when there is none.
inline int64_t merge_chunks(const std::vector<TextChunk>& chunks, std::vector<ContigRun>* runs) {
	for (const TextChunk& c : chunks) {
		if (c.bad_line >= 0) return (int64_t)c.row0 + c.bad_line;
		for (const ContigRun& r : c.runs) {
			if (!runs->empty() && runs->back().name == r.name) runs->back().count += r.count;
			else runs->push_back(r);
		}
	}
	return -1;
}

// ---- output ----------------------------------------------------------------------------

inline char* put_u32(char* p, uint32_t v) { return std::to_chars(p, p + 12, v).ptr; }
inline char* put_i32(char* p, int32_t v) { return std::to_chars(p, p + 12, v).ptr; }
// `ostream << double` = printf("%g"): std::to_chars(general, precision 6) is specified to produce exactly
// that text (checked against snprintf on 4e6 values incl. rounding ties, inf and nan) and is ~2.5x faster
inline char* put_g_general(char* p, double v) { return std::to_chars(p, p + 32, v, std::chars_format::general, 6).ptr; }
// The same text ~4x faster for the values the tools print by the hundred million (one row per site with the default
// arguments): |v| in [1e-5, 1e15) is scaled to six digits with ONE exactly-rounded operation (times or over an exact
// power of ten <= 1e10: error < 2e-10 on a number below 1e6), and whenever the scaled value lies within 1e-6 of a
// rounding boundary -- the only place where that error could change the sixth digit, exact ties included -- the
// general routine decides.  Zero, subnormals, huge values, inf and nan go there too.
inline char* put_g(char* p, double v) {
	static const double kP10[16] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15};
	static const char kPairs[201] =
	    "00010203040506070809101112131415161718192021222324252627282930313233343536373839404142434445464748495051525354555657585960616263646566676869707172737475767778798081828384858687888990919293949596979899";
	const double x = v < 0 ? -v : v;
	if (!(x >= 1e-5 && x < 1e15)) return put_g_general(p, v);
	// decimal exponent of the leading digit: estimated from the binary exponent (log10(2) = 0.30103), then one exact
	// comparison.  (The thresholds below 1 are nearest doubles: a value one ulp off a power of ten may land one decade
	// off, which the range check on n catches.)
	uint64_t bits;
	memcpy(&bits, &x, 8);
	const int e2 = (int)(bits >> 52) - 1023;
	int X = (e2 * 1233) >> 12;  // floor(e2 * log10(2)) or one less, for |e2| <= 64
	double scaled;
	if (X >= 0) {
		if (x >= kP10[X + 1 < 16 ? X + 1 : 15]) ++X;  // (x < 1e15, so X + 1 <= 15 whenever the comparison can hold)
		scaled = X <= 5 ? x * kP10[5 - X] : x / kP10[X - 5];
	} else {
		static const double kNeg[7] = {1e0, 1e-1, 1e-2, 1e-3, 1e-4, 1e-5, 1e-6};
		if (X < -6) X = -6;
		if (x >= kNeg[-X - 1]) ++X;  // X + 1 <= 0 here
		if (X < -5) return put_g_general(p, v);
		scaled = x * kP10[5 - X];
	}
	const double fl = (double)(int64_t)scaled;
	const double frac = scaled - fl;
	if (frac > 0.499999 && frac < 0.500001) return put_g_general(p, v);
	uint32_t n = (uint32_t)(int64_t)fl + (frac > 0.5 ? 1u : 0u);
	if (n == 1000000u) {  // 999999.6 -> 1.00000 of the next decade
		n = 100000u;
		++X;
	}
	if (n < 100000u || n > 999999u) return put_g_general(p, v);
	const int tz = (n % 10u == 0) + (n % 100u == 0) + (n % 1000u == 0) + (n % 10000u == 0) + (n % 100000u == 0);
	const int sig = 6 - tz;
	char d[16];  // the six digits, then slack for the fixed-size copies below
	memcpy(d, kPairs + 2 * (n / 10000u), 2);
	memcpy(d + 2, kPairs + 2 * (n / 100u % 100u), 2);
	memcpy(d + 4, kPairs + 2 * (n % 100u), 2);
	memset(d + 6, '0', 10);
	*p = '-';
	p += v < 0;
	// (every branch writes at most 16 bytes from p; callers reserve 32 per value)
	if (X >= 0 && X < 6) {  // %g: fixed notation when -4 <= X < precision
		memcpy(p, d, 8);
		if (sig <= X + 1) return p + X + 1;
		p[X + 1] = '.';
		memcpy(p + X + 2, d + X + 1, 8);
		return p + sig + 1;
	}
	if (X < 0 && X >= -4) {
		memcpy(p, "0.0000", 6);
		p += 1 - X;
		memcpy(p, d, 8);
		return p + sig;
	}
	p[0] = d[0];
	p[1] = '.';
	memcpy(p + 2, d + 1, 8);
	p += sig > 1 ? sig + 1 : 1;
	int e = X;
	p[0] = 'e';
	p[1] = e < 0 ? '-' : '+';
	if (e < 0) e = -e;
	memcpy(p + 2, kPairs + 2 * e, 2);
	return p + 4;
}

// format rows [lo, hi) with `fn(char* p, uint64_t row) -> char*` on several threads, write in order
template <class Fn>
inline void write_rows(FILE* f, uint64_t nrows, size_t max_row_bytes, Fn fn) {
	if (nrows == 0) return;
	unsigned nt = parse_threads();
	if (nrows < 4096) nt = 1;
	const uint64_t block = 1u << 16;
	std::vector<std::vector<char>> bufs(nt);
	for (uint64_t base = 0; base < nrows; base += block * nt) {
		std::vector<std::thread> th;
		std::vector<size_t> used(nt, 0);
		for (unsigned t = 0; t < nt; ++t) {
			uint64_t lo = base + block * t, hi = std::min<uint64_t>(nrows, lo + block);
			if (lo >= hi) break;
			auto work = [&, t, lo, hi]() {
				bufs[t].resize((size_t)(hi - lo) * max_row_bytes);
				char* p = bufs[t].data();
				for (uint64_t r = lo; r < hi; ++r) p = fn(p, r);
				used[t] = (size_t)(p - bufs[t].data());
			};
			if (nt == 1) work();
			else th.emplace_back(work);
		}
		for (auto& x : th) x.join();
		for (unsigned t = 0; t < nt; ++t)
			if (used[t]) fwrite(bufs[t].data(), 1, used[t], f);
	}
}

// ---- device ----------------------------------------------------------------------------

struct DeviceWorkspace {
	void* p = nullptr;
	size_t bytes = 0;
	~DeviceWorkspace() {
		if (p) pgt_device_free(p);
	}
};

// The tools use one GPU (PGT_DEVICE, default 0) or several of one box (PGT_DEVICES=0,1,...: the window list is
// sharded over them by pgt_scan_sharded, one host thread per GPU, same stdout).  CUDA start-up enumerates and
// initialises every visible device (~0.3 s each on an 8-GPU box), so unless the user already set
// CUDA_VISIBLE_DEVICES the process restricts itself to its devices before the first CUDA call; they are then
// indices 0..n-1.
inline std::vector<int>& device_list() {
	static std::vector<int> list;
	return list;
}
inline int chosen_device() {
	std::vector<int>& list = device_list();
	if (!list.empty()) return list[0];
	std::vector<int> want;
	if (const char* env = getenv("PGT_DEVICES")) {
		for (const char* p = env; *p;) {
			char* e = nullptr;
			const long v = strtol(p, &e, 10);
			if (e == p) break;
			if (v >= 0) want.push_back((int)v);
			p = (*e == ',') ? e + 1 : e;
			if (*e != ',' && *e != 0) break;
		}
	}
	if (want.empty()) {
		const char* env = getenv("PGT_DEVICE");
		want.push_back(env ? atoi(env) : 0);
	}
	if (!getenv("CUDA_VISIBLE_DEVICES") && want[0] >= 0) {
		std::string vis;
		for (size_t i = 0; i < want.size(); ++i) vis += (i ? "," : "") + std::to_string(want[i]);
		setenv("CUDA_VISIBLE_DEVICES", vis.c_str(), 1);
		for (size_t i = 0; i < want.size(); ++i) list.push_back((int)i);
	} else {
		list = want;
	}
	return list[0];
}

inline int select_device() {
	const int dev = chosen_device();
	int n = pgt_device_count();
	if (n <= 0) {
		fprintf(stderr, "No usable CUDA device: %s\n", n < 0 ? pgt_last_error() : "device count is 0");
		return -1;
	}
	if (pgt_set_device(dev) != PGT_OK) {
		fprintf(stderr, "%s\n", pgt_last_error());
		return -1;
	}
	return 0;
}

// CUDA start-up (driver + context, ~1-2 s on a B200 box) overlaps with text parsing: helper threads bring the
// device(s) up while the parser threads run; the main thread joins them before the scan.
struct DeviceWarmup {
	std::thread th;
	std::atomic<int> state{0};  // 0 = not started / running, 1 = device(s) up, -1 = failed
	int rc = 0;
	double ms = 0;
	std::string err;
	void start() {
		chosen_device();  // on the calling thread, before any CUDA call
		const std::vector<int> devs = device_list();
		th = std::thread([this, devs]() {
			const double t0 = now_ms();
			int n = pgt_device_count();
			if (n <= 0) {
				rc = -1;
				err = n < 0 ? pgt_last_error() : "device count is 0";
			} else {
				std::vector<std::thread> per;
				std::vector<std::string> errs(devs.size());
				for (size_t i = 0; i < devs.size(); ++i)
					per.emplace_back([&errs, &devs, i]() {
						void* p = nullptr;  // forces context creation
						if (pgt_set_device(devs[i]) != PGT_OK) errs[i] = pgt_last_error();
						else if (pgt_device_alloc(&p, 1 << 20) == PGT_OK) pgt_device_free(p);
					});
				for (auto& t : per) t.join();
				for (const std::string& e : errs)
					if (!e.empty()) {
						rc = -1;
						err = e;
					}
			}
			ms = now_ms() - t0;
			state.store(rc == 0 ? 1 : -1);
		});
	}
	// 0 ok; on failure prints the same message as select_device()
	int finish() {
		if (th.joinable()) th.join();
		if (rc != 0) {
			fprintf(stderr, "No usable CUDA device: %s\n", err.c_str());
			return -1;
		}
		return select_device();  // cudaSetDevice is per-thread state: cheap now
	}
	~DeviceWarmup() {
		if (th.joinable()) th.join();
	}
};

// The scan of a tool: one device -> pgt_scan with a workspace from pgt_device_alloc; PGT_DEVICES with several
// devices -> pgt_scan_sharded (the whole window table, same rows).  Prints nothing; pgt_last_error() on failure.
inline int scan_on_devices(const pgt_plan* plan, const pgt_range* range, pgt_stat stat, const pgt_columns* cols, int minind,
                           const uint64_t* site_offsets, const pgt_windows* out) {
	const std::vector<int>& devs = device_list();
	if (devs.size() > 1) return pgt_scan_sharded(plan, stat, cols, minind, site_offsets, out, devs.data(), (uint32_t)devs.size(), nullptr, nullptr);
	DeviceWorkspace ws;
	ws.bytes = pgt_scan_workspace_bytes(plan, range, stat, PGT_MEM_HOST);
	const int rc = pgt_device_alloc(&ws.p, ws.bytes);
	if (rc != PGT_OK) return rc;
	return pgt_scan(plan, range, stat, cols, minind, site_offsets, out, ws.p, ws.bytes, PGT_MEM_HOST, nullptr);
}

struct Timing {
	double parse_ms = 0, scan_ms = 0, format_ms = 0, total_ms = 0, cuda_init_ms = 0;
	double upload_tail_ms = 0;      // streaming upload: what was left to wait for when parsing / loading had finished
	double upload_gbs = 0;          // bytes sent / (first byte queued .. last byte on the device)
	uint64_t upload_bytes = 0;
	const char* mode = "host";      // "host": columns handed to pgt_scan(PGT_MEM_HOST); "stream": resident columns via the uploader
	uint64_t sites = 0, windows = 0;
	unsigned threads = 0;
	void report(const char* tool) const {
		if (!getenv("PGT_TIMING")) return;
		fprintf(stderr,
		        "{\"tool\":\"%s\",\"sites\":%llu,\"windows\":%llu,\"parse_ms\":%.3f,\"scan_ms\":%.3f,\"format_ms\":%.3f,"
		        "\"total_ms\":%.3f,\"parse_threads\":%u,\"cuda_init_ms_overlapped_with_parse\":%.3f,\"mode\":\"%s\","
		        "\"upload_bytes\":%llu,\"upload_gbs\":%.2f,\"upload_tail_ms\":%.3f}\n",
		        tool, (unsigned long long)sites, (unsigned long long)windows, parse_ms, scan_ms, format_ms, total_ms, threads, cuda_init_ms, mode,
		        (unsigned long long)upload_bytes, upload_gbs, upload_tail_ms);
	}
};

// ---- streaming upload of the tools' columns (pgt_uploader, include/pgt_scan.h) -----------------------------
//
// One GPU, an input of some size: the columns become device-resident while the producer is still running.
// Text: the parser thread that finishes a chunk queues that chunk's rows (rows_ready only enqueues, any order);
// the uploader's copy threads stage them through the pinned ring, so the wall time is max(parse, upload), not
// their sum.  Columnar cache: the file's column blocks are read with pread straight into the ring (no
// page-cache mapping handed to the driver).  Afterwards the scan runs in PGT_MEM_DEVICE and only the window rows
// come back.  Falls back (finish() != 0) when the columns do not fit the free HBM, several GPUs are selected
// (PGT_DEVICES: the sharded host-memory scan), the input is small, or PGT_STREAM=0.
struct StreamColumn {
	const void* host;   // the column in host memory (text parser output / cache mapping)
	uint32_t elem;      // bytes per site
	uint64_t file_off;  // columnar cache: byte offset of the column in the file
	int field;          // index into pgt_columns: 0 pos, 1 a, 2 b, 3 geno, 4 f1, 5 f2, 6 n1, 7 n2
};

struct ColumnStreamer {
	bool on = false;
	std::atomic<bool> failed{false};
	std::thread th;
	std::mutex mu;
	bool ready = false;
	pgt_uploader* up = nullptr;
	StreamColumn cols[8];
	void* dcol[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
	int ncol = 0;
	uint64_t n = 0;
	int fd = -1;
	double t_first = 0;
	std::vector<std::pair<uint64_t, uint64_t>> pending;  // row ranges that became ready before the device was up
	std::string why;

	bool active() const { return on; }

	static uint64_t min_sites() {
		const char* e = getenv("PGT_STREAM_MIN_SITES");
		return e ? strtoull(e, nullptr, 10) : (uint64_t)8 << 20;
	}

	void put_rows_locked(uint64_t lo, uint64_t hi) {
		if (hi <= lo || failed.load()) return;
		if (t_first == 0) t_first = now_ms();
		for (int c = 0; c < ncol; ++c) {
			char* dst = (char*)dcol[c] + lo * cols[c].elem;
			const size_t bytes = (size_t)(hi - lo) * cols[c].elem;
			const int rc = fd >= 0 ? pgt_uploader_put_file(up, dst, fd, cols[c].file_off + lo * cols[c].elem, bytes)
			                       : pgt_uploader_put(up, dst, (const char*)cols[c].host + lo * cols[c].elem, bytes);
			if (rc != PGT_OK) {
				why = pgt_last_error();
				failed.store(true);
				return;
			}
		}
	}

	// nwin_est / out_row_bytes: room to leave for the window table and the scan's workspace
	void start(DeviceWarmup* warm, const StreamColumn* c, int nc, uint64_t nrows, uint64_t nwin_est, size_t out_row_bytes, const char* file_path) {
		const char* env = getenv("PGT_STREAM");
		if ((env && atoi(env) == 0) || nrows < min_sites()) return;
		chosen_device();
		if (device_list().size() != 1) return;
		ncol = nc;
		n = nrows;
		for (int i = 0; i < nc; ++i) cols[i] = c[i];
		if (file_path) {
			fd = open(file_path, O_RDONLY);
			if (fd < 0) return;
		}
		on = true;
		const int dev = device_list()[0];
		th = std::thread([this, warm, dev, nwin_est, out_row_bytes]() {
			while (warm->state.load() == 0) std::this_thread::sleep_for(std::chrono::microseconds(200));
			auto give_up = [this](const std::string& m) {
				std::lock_guard<std::mutex> lk(mu);
				why = m;
				failed.store(true);
			};
			if (warm->state.load() < 0 || pgt_set_device(dev) != PGT_OK) return give_up("device not available");
			size_t free_b = 0, total_b = 0;
			if (pgt_device_mem_info(&free_b, &total_b) != PGT_OK) return give_up(pgt_last_error());
			uint64_t need = (uint64_t)nwin_est * out_row_bytes + ((uint64_t)1 << 30);
			for (int i = 0; i < ncol; ++i) need += n * cols[i].elem;
			if ((double)need > 0.92 * (double)free_b) return give_up("columns do not fit the free device memory");
			for (int i = 0; i < ncol; ++i)
				if (pgt_device_alloc(&dcol[i], (size_t)(n * cols[i].elem)) != PGT_OK) return give_up(pgt_last_error());
			// text: the parser threads own the cores and produce ~8 GB/s of columns; cache: nothing else runs
			const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
			unsigned nthreads = fd >= 0 ? std::min(16u, hw) : std::min(4u, hw);
			if (const char* e = getenv("PGT_UPLOAD_THREADS")) nthreads = std::max(1, atoi(e));
			pgt_uploader* u = nullptr;
			if (pgt_uploader_create(&u, nullptr, 0, 2 * nthreads, (size_t)16 << 20, nthreads) != PGT_OK) return give_up(pgt_last_error());
			std::lock_guard<std::mutex> lk(mu);
			up = u;
			ready = true;
			if (fd >= 0) put_rows_locked(0, n);  // the whole file, read with pread by the copy threads
			for (auto& r : pending) put_rows_locked(r.first, r.second);
			pending.clear();
		});
	}

	// rows [lo, hi) of every column are final in host memory (called by the parser threads, one range per chunk)
	void rows_ready(uint64_t lo, uint64_t hi) {
		if (!on || failed.load()) return;
		std::lock_guard<std::mutex> lk(mu);
		if (!ready) pending.emplace_back(lo, hi);
		else put_rows_locked(lo, hi);
	}

	// 0: every column is resident; otherwise the caller falls back to the host-memory scan
	int finish(Timing* tm) {
		if (!on) return -1;
		const double t0 = now_ms();
		if (th.joinable()) th.join();
		uint64_t sent = 0, want = 0;
		for (int c = 0; c < ncol; ++c) want += n * cols[c].elem;
		if (!failed.load() && pgt_uploader_drain(up, &sent) != PGT_OK) {
			why = pgt_last_error();
			failed.store(true);
		} else if (!failed.load() && sent != want) {  // rows never queued: the scan would read unwritten device memory
			why = "uploaded " + std::to_string(sent) + " of " + std::to_string(want) + " column bytes";
			failed.store(true);
		}
		if (failed.load()) {
			if (getenv("PGT_TIMING")) fprintf(stderr, "{\"stream_fallback\":\"%s\"}\n", why.c_str());
			release();
			return -1;
		}
		const double t1 = now_ms();
		tm->mode = "stream";
		tm->upload_bytes = sent;
		tm->upload_tail_ms = t1 - t0;
		tm->upload_gbs = t1 > t_first && t_first > 0 ? (double)sent / ((t1 - t_first) * 1e6) : 0.0;
		return 0;
	}

	// device-mode scan over the resident columns; `out` holds HOST arrays of nwin rows (any may be NULL)
	int scan(const pgt_plan* plan, pgt_stat stat, const pgt_windows* out, uint64_t nwin, int minind = 1, const pgt_range* range = nullptr,
	         const uint64_t* site_offsets = nullptr) {
		pgt_columns dc;
		memset(&dc, 0, sizeof(dc));
		const void** slots[8] = {(const void**)&dc.pos, (const void**)&dc.a, (const void**)&dc.b, (const void**)&dc.geno,
		                         (const void**)&dc.f1, (const void**)&dc.f2, (const void**)&dc.n1, (const void**)&dc.n2};
		for (int c = 0; c < ncol; ++c) *slots[cols[c].field] = dcol[c];
		struct Field {
			void* host;
			void** dev;
			size_t elem;
		};
		pgt_windows dw;
		memset(&dw, 0, sizeof(dw));
		Field f[14] = {{out->label, (void**)&dw.label, 4},       {out->start_pos, (void**)&dw.start_pos, 4}, {out->end_pos, (void**)&dw.end_pos, 4},
		               {out->mid_pos, (void**)&dw.mid_pos, 4},   {out->nsites, (void**)&dw.nsites, 4},       {out->sum_a, (void**)&dw.sum_a, 8},
		               {out->sum_b, (void**)&dw.sum_b, 8},       {out->fst, (void**)&dw.fst, 8},             {out->nhet, (void**)&dw.nhet, 4},
		               {out->nonmissing, (void**)&dw.nonmissing, 4}, {out->het, (void**)&dw.het, 8},         {out->dxy, (void**)&dw.dxy, 8},
		               {out->neffective, (void**)&dw.neffective, 4}, {out->nskip, (void**)&dw.nskip, 4}};
		std::vector<void*> owned;
		auto cleanup = [&]() {
			for (void* p : owned) pgt_device_free(p);
		};
		int rc = PGT_OK;
		for (Field& x : f) {
			if (!x.host) continue;
			void* p = nullptr;
			if ((rc = pgt_device_alloc(&p, (size_t)std::max<uint64_t>(nwin, 1) * x.elem)) != PGT_OK) break;
			owned.push_back(p);
			*x.dev = p;
		}
		void* dglobal = nullptr;
		if (rc == PGT_OK && out->dxy_global) {
			if ((rc = pgt_device_alloc(&dglobal, 3 * sizeof(double))) == PGT_OK) {
				owned.push_back(dglobal);
				dw.dxy_global = (double*)dglobal;
			}
		}
		void* ws = nullptr;
		size_t ws_bytes = 0;
		if (rc == PGT_OK) {
			ws_bytes = pgt_scan_workspace_bytes(plan, range, stat, PGT_MEM_DEVICE);
			if ((rc = pgt_device_alloc(&ws, ws_bytes)) == PGT_OK) owned.push_back(ws);
		}
		if (rc == PGT_OK) rc = pgt_scan(plan, range, stat, &dc, minind, site_offsets, &dw, ws, ws_bytes, PGT_MEM_DEVICE, nullptr);
		for (Field& x : f)
			if (rc == PGT_OK && x.host) rc = pgt_memcpy_to_host(x.host, *x.dev, (size_t)nwin * x.elem);
		if (rc == PGT_OK && out->dxy_global) rc = pgt_memcpy_to_host(out->dxy_global, dglobal, 3 * sizeof(double));
		cleanup();
		return rc;
	}

	void release() {
		if (up) pgt_uploader_destroy(up);
		up = nullptr;
		for (int c = 0; c < 8; ++c) {
			if (dcol[c]) pgt_device_free(dcol[c]);
			dcol[c] = nullptr;
		}
		if (fd >= 0) close(fd);
		fd = -1;
	}
	~ColumnStreamer() {
		if (th.joinable()) th.join();
		release();
	}
};

}  // namespace pgtcli
#endif
