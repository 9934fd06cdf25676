// pgt_cuda.h -- error, launch-geometry, table and timing helpers of the host code that launches kernels (pgt_scan.cu,
// pgt_extreme.cu).
#ifndef PGT_CUDA_H
#define PGT_CUDA_H

#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "pgt_internal.h"

static inline int cuda_fail(cudaError_t e, const char* what) {
	return pgt_set_error(PGT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}
#define PGT_CUDA(call)                                         \
	do {                                                       \
		cudaError_t e__ = (call);                              \
		if (e__ != cudaSuccess) return cuda_fail(e__, #call);  \
	} while (0)
#define PGT_TRY(call)                    \
	do {                                 \
		int rc__ = (call);               \
		if (rc__ != PGT_OK) return rc__; \
	} while (0)

static inline int num_sms() {
	int dev = 0, n = 0;
	if (cudaGetDevice(&dev) != cudaSuccess) return 0;
	cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
	return n;
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Grid of a grid-stride kernel: the blocks that are resident at once (one wave), or fewer when the work is small.
// (A fixed cap of 8 blocks per SM launched the per-site kernel -- 6 resident blocks at 40 registers -- as one full wave
// plus a third of one: ncu "waves per SM 1.33", profiles/r02h_persite_ncu_details.txt.)
template <class K>
static unsigned one_wave_grid(K kern, int threads, uint64_t want_blocks, size_t smem = 0) {
	int per_sm = 0;
	if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
	const uint64_t cap = (uint64_t)num_sms() * per_sm;
	return (unsigned)(want_blocks < cap ? (want_blocks ? want_blocks : 1) : cap);
}

// A plan's device tables (pgt_plan_bind_device, pgt_xplan_bind_device): two host tables a | b in a caller's buffer,
// each at a 256-byte boundary whatever the buffer's alignment.  table_pair_bytes is the buffer size they need.
// bind_table_pair copies them (an empty table is skipped), waits for the copies and sets *base to where a begins;
// b begins align_up(a_bytes, 256) after it.
static inline size_t table_pair_bytes(size_t a_bytes, size_t b_bytes) { return align_up(a_bytes, 256) + align_up(b_bytes, 256) + 256; }

static inline int bind_table_pair(void* buffer, const void* a, size_t a_bytes, const void* b, size_t b_bytes, void* stream,
                                  unsigned char** base) {
	cudaStream_t st = (cudaStream_t)stream;
	unsigned char* p = (unsigned char*)align_up((uintptr_t)buffer, 256);
	cudaError_t e = cudaSuccess;
	if (a_bytes) e = cudaMemcpyAsync(p, a, a_bytes, cudaMemcpyHostToDevice, st);
	if (e == cudaSuccess && b_bytes) e = cudaMemcpyAsync(p + align_up(a_bytes, 256), b, b_bytes, cudaMemcpyHostToDevice, st);
	if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(plan table -> device)");
	PGT_CUDA(cudaStreamSynchronize(st));
	*base = p;
	return PGT_OK;
}

// Optional per-kernel timing (pgt_profile): CUDA events on `st` around the launches of a scope, read back by
// pgt_profile_read*.  kinds: 0 = level 1 (k_units*), 1 = level 2 (k_windows*), 2 / 3 = level 1 / 2 of the extreme scan
struct ProfScope {
	cudaStream_t st;
	cudaEvent_t a = nullptr, b = nullptr;
	int kind;
	bool on;
	ProfScope(int k, cudaStream_t s) : st(s), kind(k), on(pgt_profile_enabled()) {
		if (!on) return;
		if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) {
			on = false;
			return;
		}
		cudaEventRecord(a, st);
	}
	~ProfScope() {
		if (!on) return;
		cudaEventRecord(b, st);
		pgt_profile_push(kind, a, b);
	}
};

#endif
