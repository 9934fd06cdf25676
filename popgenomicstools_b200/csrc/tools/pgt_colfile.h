// pgt_colfile.h -- binary columnar cache of the tools' text inputs (SURVEY.md §8f rank 1).
//
// The reference re-parses its text input on every run, and that is >= 95 % of its wall time
// (getline + stringstream, /root/reference/fstWindow.cpp:123-146).  A `.pgtc` file holds exactly what
// the text parser of the drop-in CLIs produces -- the columns libpgtscan reads plus the chromosome
// runs -- so a later run maps the file and goes straight to the H2D copies.  Writing: run any CLI
// with PGT_PACK=<out.pgtc> (dxyWindow: PGT_PACK for pop 1, PGT_PACK2 for pop 2): it parses, writes
// the cache and exits without touching the GPU.  Reading: give the `.pgtc` file where the text file
// went; the tools sniff the magic bytes, as the reference sniffs gzip (dxyWindow.cpp:82-83).
//
// Layout (little endian):
//   0   char     magic[8]  = "PGTCOL\x01\n"
//   8   uint32   version   = 1
//   12  uint32   kind        1 fst (pos u32, a f64, b f64)        fstWindow.cpp:17-21
//                            2 het (pos u32, geno i8)             hetWindow.cpp:18
//                            3 maf (pos u32, freq f64, nInd i32)  dxyWindow.cpp:24-32 (one population)
//                            4 score (pos u32, score f64)         ihsWindow.cpp:119,160 / xpehhWindow.cpp:165
//                            5 dxy (pos u32, f1 f64, f2 f64, n1 i32, n2 i32): the SYNCED sites of two MAFs, written by
//                              dxyWindow with PGT_PACK_SYNCED=<out> (inspection / tests of the two-file sync, dxyWindow.cpp:315-331)
//   16  uint64   nsites
//   24  uint32   nruns       runs of equal chromosome name, in file order
//   28  uint32   ncols
//   32  uint64   names_bytes
//   40  uint64   data_offset (multiple of 4096)
//   48  uint64   reserved[2]
//   64  uint64   run_count[nruns]
//       char     names[names_bytes]   NUL-terminated, in run order
//   data_offset: the columns back to back, each padded to a multiple of 4096 bytes
#ifndef PGT_COLFILE_H
#define PGT_COLFILE_H

#include "pgt_cli.h"

namespace pgtcol {

enum Kind : uint32_t { KIND_FST = 1, KIND_HET = 2, KIND_MAF = 3, KIND_SCORE = 4, KIND_DXY = 5 };
static const char kMagic[8] = {'P', 'G', 'T', 'C', 'O', 'L', 1, '\n'};
static const uint64_t kAlign = 4096;

inline const uint32_t* elem_sizes(uint32_t kind, uint32_t* ncols) {
	static const uint32_t fst[3] = {4, 8, 8}, het[2] = {4, 1}, maf[3] = {4, 8, 4}, score[2] = {4, 8}, dxy[5] = {4, 8, 8, 4, 4};
	switch (kind) {
		case KIND_FST: *ncols = 3; return fst;
		case KIND_HET: *ncols = 2; return het;
		case KIND_MAF: *ncols = 3; return maf;
		case KIND_SCORE: *ncols = 2; return score;
		case KIND_DXY: *ncols = 5; return dxy;
	}
	*ncols = 0;
	return nullptr;
}

inline uint64_t pad(uint64_t x) { return (x + kAlign - 1) / kAlign * kAlign; }

struct Header {
	char magic[8];
	uint32_t version, kind;
	uint64_t nsites;
	uint32_t nruns, ncols;
	uint64_t names_bytes, data_offset, reserved[2];
};
static_assert(sizeof(Header) == 64, "header layout");

inline bool is_colfile(const char* d, size_t n) { return n >= sizeof(Header) && memcmp(d, kMagic, 8) == 0; }

// 0 ok, -1 I/O error
inline int write_file(const char* path, uint32_t kind, const std::vector<pgtcli::ContigRun>& runs, uint64_t nsites,
                      const void* const* cols) {
	uint32_t ncols = 0;
	const uint32_t* es = elem_sizes(kind, &ncols);
	if (!es) return -1;
	Header h;
	memset(&h, 0, sizeof(h));
	memcpy(h.magic, kMagic, 8);
	h.version = 1;
	h.kind = kind;
	h.nsites = nsites;
	h.nruns = (uint32_t)runs.size();
	h.ncols = ncols;
	for (const auto& r : runs) h.names_bytes += r.name.size() + 1;
	h.data_offset = pad(sizeof(Header) + 8ull * runs.size() + h.names_bytes);
	FILE* f = fopen(path, "wb");
	if (!f) return -1;
	bool ok = fwrite(&h, sizeof(h), 1, f) == 1;
	for (const auto& r : runs) ok = ok && fwrite(&r.count, 8, 1, f) == 1;
	for (const auto& r : runs) ok = ok && fwrite(r.name.c_str(), 1, r.name.size() + 1, f) == r.name.size() + 1;
	static const char zeros[4096] = {0};
	auto pad_to = [&](uint64_t target) {
		long at = ftell(f);
		while (ok && at >= 0 && (uint64_t)at < target) {
			size_t k = (size_t)std::min<uint64_t>(target - (uint64_t)at, sizeof(zeros));
			ok = fwrite(zeros, 1, k, f) == k;
			at += (long)k;
		}
	};
	pad_to(h.data_offset);
	uint64_t at = h.data_offset;
	for (uint32_t c = 0; ok && c < ncols; ++c) {
		const uint64_t bytes = nsites * es[c];
		const char* p = (const char*)cols[c];
		uint64_t done = 0;
		while (ok && done < bytes) {  // fwrite in 1 GiB pieces
			size_t k = (size_t)std::min<uint64_t>(bytes - done, 1ull << 30);
			ok = fwrite(p + done, 1, k, f) == k;
			done += k;
		}
		at = pad(at + bytes);
		pad_to(at);
	}
	ok = fclose(f) == 0 && ok;
	return ok ? 0 : -1;
}

struct View {
	uint32_t kind = 0;
	uint64_t nsites = 0;
	std::vector<pgtcli::ContigRun> runs;
	const void* col[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
};

// 0 ok; -1 malformed (err says why)
inline int open_view(const char* d, size_t n, View* v, std::string* err) {
	if (!is_colfile(d, n)) {
		*err = "not a .pgtc columnar file";
		return -1;
	}
	Header h;
	memcpy(&h, d, sizeof(h));
	uint32_t ncols = 0;
	const uint32_t* es = elem_sizes(h.kind, &ncols);
	if (h.version != 1 || !es || h.ncols != ncols) {
		*err = "unsupported .pgtc version or kind";
		return -1;
	}
	// every 64-bit header field is checked against the file size BEFORE it enters a product or a sum
	// (a crafted nsites ~ 2^61 would wrap nsites * 8 to something small)
	if (h.names_bytes > n || (uint64_t)h.nruns > n / 8 || h.nsites > n) {
		*err = "corrupt .pgtc header";
		return -1;
	}
	const uint64_t meta_end = sizeof(Header) + 8ull * h.nruns + h.names_bytes;
	if (h.data_offset % kAlign || meta_end > h.data_offset || h.data_offset > n) {
		*err = "corrupt .pgtc header";
		return -1;
	}
	v->kind = h.kind;
	v->nsites = h.nsites;
	const char* names = d + sizeof(Header) + 8ull * h.nruns;
	const char* names_end = names + h.names_bytes;
	uint64_t total = 0;
	for (uint32_t r = 0; r < h.nruns; ++r) {
		uint64_t cnt;
		memcpy(&cnt, d + sizeof(Header) + 8ull * r, 8);
		const char* z = names < names_end ? (const char*)memchr(names, 0, (size_t)(names_end - names)) : nullptr;
		if (!z || cnt == 0 || cnt > h.nsites - total) {
			*err = "corrupt .pgtc run table";
			return -1;
		}
		v->runs.push_back(pgtcli::ContigRun{std::string(names, z), cnt});
		names = z + 1;
		total += cnt;
	}
	if (total != h.nsites) {
		*err = "corrupt .pgtc run table (counts do not add up)";
		return -1;
	}
	uint64_t at = h.data_offset;
	for (uint32_t c = 0; c < ncols; ++c) {
		if (at > n || h.nsites > (n - at) / es[c]) {
			*err = "truncated .pgtc file";
			return -1;
		}
		const uint64_t bytes = h.nsites * es[c];
		if (at + bytes > n) {
			*err = "truncated .pgtc file";
			return -1;
		}
		v->col[c] = d + at;
		at = pad(at + bytes);
	}
	return 0;
}

// open_view for a tool that reads `kind`: 0 ok; otherwise prints "<tool>: <path>: <why>" and returns -1
inline int open_view_of(const char* d, size_t n, uint32_t kind, View* v, const char* tool, const char* path) {
	std::string err;
	if (open_view(d, n, v, &err) == 0 && v->kind == kind) return 0;
	fprintf(stderr, "%s: %s: %s\n", tool, path, err.empty() ? "columnar file of another tool" : err.c_str());
	return -1;
}

}  // namespace pgtcol
#endif
