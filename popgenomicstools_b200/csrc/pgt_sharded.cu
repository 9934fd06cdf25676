// pgt_sharded.cu -- one host column set, several GPUs of ONE process (SURVEY.md §8b threading row:
// "one host thread per GPU"; §8e: shards by site range, halo = W - S, no data-path collective).
//
// The reference is a single-threaded process (/root/reference/fstWindow.cpp:109-155); a user of the
// drop-in tools on an 8-GPU box should not have to split the input or launch eight processes.  Here the
// window list is cut by pgt_plan_shard; every shard runs the ordinary host-memory scan (pgt_scan,
// PGT_MEM_HOST) on its own device from its own host thread and stream, reads only the slabs of the
// caller's columns that its windows cover, and copies its rows device -> host straight into the
// caller's result arrays at its window offset.  Nothing is gathered afterwards: the table is complete
// when the threads have joined.  Per-window results are bit-identical for any device count (the
// summation order is a function of (W, S, unit) only); dxyWindow's global line is the sum of the
// shards' disjoint partial lines in shard order.
#include <cuda_runtime.h>

#include <string>
#include <thread>
#include <vector>

#include "pgt_internal.h"

namespace {

struct ShardJob {
	uint32_t shard = 0;
	int device = 0;
	uint64_t w_lo = 0, w_hi = 0;
	void* ws = nullptr;
	size_t ws_bytes = 0;
	bool own_ws = false;
	double global3[3] = {0.0, 0.0, 0.0};
	int rc = PGT_OK;
	std::string err;
};

pgt_windows rows_from(const pgt_windows& o, uint64_t d) {
	pgt_windows r = o;
	for_each_field([d](auto*& p) { p = p ? p + d : p; }, r);
	return r;
}

void run_shard(const pgt_plan* plan, pgt_stat stat, const pgt_columns* cols, int minind, const uint64_t* site_offsets, const pgt_windows* out,
               ShardJob* job) {
	auto fail = [job](int rc, const std::string& msg) {
		job->rc = rc;
		job->err = msg;
	};
	cudaError_t e = cudaSetDevice(job->device);
	if (e != cudaSuccess) return fail(PGT_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
	// the whole axis is addressable from element 0 of the caller's columns; the scan touches only its slabs
	pgt_range range;
	range.w_lo = job->w_lo;
	range.w_hi = job->w_hi;
	range.site_origin = 0;
	range.site_count = 0;
	if (job->w_lo == job->w_hi && (pgt_plan_num_windows(plan) != 0 || job->shard != 0)) {
		// a shard without windows has nothing to do ({0, 0} would even mean "all windows" to pgt_scan) -- except
		// shard 0 of a plan without any window: it owns the axis, whose sites still count for the global line
		return;
	}
	if (!job->ws) {
		job->ws_bytes = pgt_scan_workspace_bytes(plan, &range, stat, PGT_MEM_HOST);
		e = cudaMalloc(&job->ws, job->ws_bytes ? job->ws_bytes : 1);
		if (e != cudaSuccess) return fail(PGT_ERR_CUDA, std::string("cudaMalloc(workspace): ") + cudaGetErrorString(e));
		job->own_ws = true;
	}
	cudaStream_t st = nullptr;
	e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
	if (e != cudaSuccess) return fail(PGT_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
	pgt_windows rows = rows_from(*out, job->w_lo);
	rows.dxy_global = out->dxy_global ? job->global3 : nullptr;
	const int rc = pgt_scan(plan, &range, stat, cols, minind, site_offsets, &rows, job->ws, job->ws_bytes, PGT_MEM_HOST, st);
	if (rc != PGT_OK) fail(rc, pgt_last_error());
	cudaStreamDestroy(st);
	if (job->own_ws) {
		cudaFree(job->ws);
		job->ws = nullptr;
	}
}

int shard_ranges(const pgt_plan* plan, uint32_t ndev, std::vector<ShardJob>* jobs) {
	jobs->resize(ndev);
	for (uint32_t i = 0; i < ndev; ++i) {
		ShardJob& j = (*jobs)[i];
		j.shard = i;
		const int rc = pgt_plan_shard(plan, i, ndev, &j.w_lo, &j.w_hi, nullptr, nullptr);
		if (rc != PGT_OK) return rc;
	}
	return PGT_OK;
}

}  // namespace

extern "C" size_t pgt_scan_sharded_workspace_bytes(const pgt_plan* plan, pgt_stat stat, uint32_t shard, uint32_t nshards) {
	if (!plan || nshards == 0 || shard >= nshards) return 0;
	pgt_range range;
	range.site_origin = 0;
	range.site_count = 0;
	if (pgt_plan_shard(plan, shard, nshards, &range.w_lo, &range.w_hi, nullptr, nullptr) != PGT_OK) return 0;
	if (range.w_lo == 0 && range.w_hi == 0 && pgt_plan_num_windows(plan) != 0) return 256;
	return pgt_scan_workspace_bytes(plan, &range, stat, PGT_MEM_HOST);
}

extern "C" int pgt_scan_sharded(const pgt_plan* plan, pgt_stat stat, const pgt_columns* cols, int minind, const uint64_t* site_offsets,
                                const pgt_windows* out, const int* devices, uint32_t ndev, void* const* workspaces,
                                const size_t* workspace_bytes) {
	if (!plan || !cols || !out) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_sharded: plan, cols and out must not be NULL");
	if (!devices || ndev == 0) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_sharded: no devices given");
	if ((workspaces == nullptr) != (workspace_bytes == nullptr))
		return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_sharded: workspaces and workspace_bytes go together (both NULL = allocate per call)");
	int have = 0;
	if (cudaGetDeviceCount(&have) != cudaSuccess || have == 0)
		return pgt_set_error(PGT_ERR_CUDA, "no usable CUDA device (libpgtscan has no CPU fallback)");
	if (plan->d_tables) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_sharded: the plan is bound to one device (pgt_plan_bind_device); unbind it first");
	// (a device may be listed more than once: its shards then run side by side on it, each on its own stream)
	for (uint32_t i = 0; i < ndev; ++i)
		if (devices[i] < 0 || devices[i] >= have) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_sharded: device index out of range");
	std::vector<ShardJob> jobs;
	const int rc0 = shard_ranges(plan, ndev, &jobs);
	if (rc0 != PGT_OK) return rc0;
	for (uint32_t i = 0; i < ndev; ++i) {
		jobs[i].device = devices[i];
		if (workspaces) {
			jobs[i].ws = workspaces[i];
			jobs[i].ws_bytes = workspace_bytes[i];
		}
	}
	int prev = 0;
	cudaGetDevice(&prev);
	if (ndev == 1) {
		run_shard(plan, stat, cols, minind, site_offsets, out, &jobs[0]);
	} else {
		std::vector<std::thread> th;
		for (uint32_t i = 0; i < ndev; ++i) th.emplace_back(run_shard, plan, stat, cols, minind, site_offsets, out, &jobs[i]);
		for (auto& t : th) t.join();
	}
	cudaSetDevice(prev);
	for (const ShardJob& j : jobs)
		if (j.rc != PGT_OK) return pgt_set_error(j.rc, "shard " + std::to_string(j.shard) + " on device " + std::to_string(j.device) + ": " + j.err);
	if (out->dxy_global) {  // the shards own disjoint parts of the axis (pgt_plan_shard): their lines add up, in shard order
		double g3[3] = {0.0, 0.0, 0.0};
		for (const ShardJob& j : jobs)
			for (int q = 0; q < 3; ++q) g3[q] += j.global3[q];
		for (int q = 0; q < 3; ++q) out->dxy_global[q] = g3[q];
	}
	return PGT_OK;
}

// ---- the bp-window extreme-score scan (ihsWindow / xpehhWindow), same scheme: windows do not overlap, so the
// shards need no halo; a shard's columns start at its first site.
extern "C" int pgt_scan_extreme_sharded(const pgt_xplan* plan, pgt_xstat stat, double cutoff, const uint32_t* pos, const double* score,
                                        const pgt_xwindows* out, const int* devices, uint32_t ndev) {
	if (!plan || !score || !out) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme_sharded: plan, score and out must not be NULL");
	if (!devices || ndev == 0) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme_sharded: no devices given");
	int have = 0;
	if (cudaGetDeviceCount(&have) != cudaSuccess || have == 0)
		return pgt_set_error(PGT_ERR_CUDA, "no usable CUDA device (libpgtscan has no CPU fallback)");
	for (uint32_t i = 0; i < ndev; ++i)
		if (devices[i] < 0 || devices[i] >= have) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme_sharded: device index out of range");
	struct XJob {
		int device = 0;
		pgt_range range;
		int rc = PGT_OK;
		std::string err;
	};
	std::vector<XJob> jobs(ndev);
	for (uint32_t i = 0; i < ndev; ++i) {
		uint64_t slo = 0, shi = 0;
		jobs[i].device = devices[i];
		const int rc = pgt_xplan_shard(plan, i, ndev, &jobs[i].range.w_lo, &jobs[i].range.w_hi, &slo, &shi);
		if (rc != PGT_OK) return rc;
		jobs[i].range.site_origin = slo;
		jobs[i].range.site_count = shi - slo;
	}
	auto run = [&](XJob* job) {
		if (job->range.w_hi <= job->range.w_lo) return;
		cudaError_t e = cudaSetDevice(job->device);
		void* ws = nullptr;
		const size_t bytes = pgt_scan_extreme_workspace_bytes(plan, &job->range, PGT_MEM_HOST);
		if (e == cudaSuccess) e = cudaMalloc(&ws, bytes ? bytes : 1);
		cudaStream_t st = nullptr;
		if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
		if (e != cudaSuccess) {
			job->rc = PGT_ERR_CUDA;
			job->err = cudaGetErrorString(e);
			if (ws) cudaFree(ws);
			return;
		}
		pgt_xwindows rows = *out;
		const uint64_t d = job->range.w_lo;
		for_each_xfield([d](auto*& p) { p = p ? p + d : p; }, rows);
		const uint64_t s0 = job->range.site_origin;
		const int rc = pgt_scan_extreme(plan, &job->range, stat, cutoff, pos ? pos + s0 : nullptr, score + s0, &rows, ws, bytes, PGT_MEM_HOST, st);
		if (rc != PGT_OK) {
			job->rc = rc;
			job->err = pgt_last_error();
		}
		cudaStreamDestroy(st);
		cudaFree(ws);
	};
	int prev = 0;
	cudaGetDevice(&prev);
	if (ndev == 1) {
		run(&jobs[0]);
	} else {
		std::vector<std::thread> th;
		for (uint32_t i = 0; i < ndev; ++i) th.emplace_back(run, &jobs[i]);
		for (auto& t : th) t.join();
	}
	cudaSetDevice(prev);
	for (uint32_t i = 0; i < ndev; ++i)
		if (jobs[i].rc != PGT_OK)
			return pgt_set_error(jobs[i].rc, "shard " + std::to_string(i) + " on device " + std::to_string(jobs[i].device) + ": " + jobs[i].err);
	return PGT_OK;
}
