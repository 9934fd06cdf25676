// pgt_cuda.h -- error and timing helpers of the host code that launches kernels (pgt_scan.cu, pgt_extreme.cu).
#ifndef PGT_CUDA_H
#define PGT_CUDA_H

#include <cuda_runtime.h>

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
