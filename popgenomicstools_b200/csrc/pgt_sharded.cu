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

#include "pgt_cuda.h"

namespace {

// One shard of a multi-GPU scan.  The caller's describe() sets its windows (and sites), whether it is idle (nothing to
// scan) and its workspace: the caller's own, or ws = nullptr and the bytes to allocate for the call.
struct Shard {
	pgt_range range{};
	bool idle = false;
	void* ws = nullptr;
	size_t ws_bytes = 0;
	double global3[3] = {0.0, 0.0, 0.0};  // the window scan's part of dxyWindow's global line
	int rc = PGT_OK;
	std::string err;
};

// The shards of a multi-GPU scan: after the device list is checked, describe(i, shard) sets up shard i, and every shard
// that is not idle runs scan(shard, stream) on devices[i] from a host thread of its own (inline for one device), on a
// stream of its own and in its workspace.  The caller's current device is restored; the first failing shard is reported.
template <class Describe, class Scan>
int run_shards(const char* who, const int* devices, uint32_t ndev, std::vector<Shard>& shards, Describe&& describe, Scan&& scan) {
	if (!devices || ndev == 0) return pgt_set_error(PGT_ERR_ARGS, std::string(who) + ": no devices given");
	int have = 0;
	if (cudaGetDeviceCount(&have) != cudaSuccess || have == 0)
		return pgt_set_error(PGT_ERR_CUDA, "no usable CUDA device (libpgtscan has no CPU fallback)");
	// (a device may be listed more than once: its shards then run side by side on it, each on its own stream)
	for (uint32_t i = 0; i < ndev; ++i)
		if (devices[i] < 0 || devices[i] >= have) return pgt_set_error(PGT_ERR_ARGS, std::string(who) + ": device index out of range");
	shards.assign(ndev, Shard());
	for (uint32_t i = 0; i < ndev; ++i) PGT_TRY(describe(i, shards[i]));
	auto run = [&](uint32_t i) {
		Shard& s = shards[i];
		if (s.idle) return;
		auto fail = [&s](int rc, const std::string& msg) {
			s.rc = rc;
			s.err = msg;
		};
		cudaError_t e = cudaSetDevice(devices[i]);
		if (e != cudaSuccess) return fail(PGT_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
		const bool own_ws = !s.ws;
		if (own_ws) {
			e = cudaMalloc(&s.ws, s.ws_bytes ? s.ws_bytes : 1);
			if (e != cudaSuccess) return fail(PGT_ERR_CUDA, std::string("cudaMalloc(workspace): ") + cudaGetErrorString(e));
		}
		cudaStream_t st = nullptr;
		e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
		if (e != cudaSuccess) {
			fail(PGT_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
		} else {
			const int rc = scan(s, st);
			if (rc != PGT_OK) fail(rc, pgt_last_error());
			cudaStreamDestroy(st);
		}
		if (own_ws) cudaFree(s.ws);
	};
	int prev = 0;
	cudaGetDevice(&prev);
	if (ndev == 1) {
		run(0);
	} else {
		std::vector<std::thread> th;
		for (uint32_t i = 0; i < ndev; ++i) th.emplace_back(run, i);
		for (auto& t : th) t.join();
	}
	cudaSetDevice(prev);
	for (uint32_t i = 0; i < ndev; ++i)
		if (shards[i].rc != PGT_OK)
			return pgt_set_error(shards[i].rc, "shard " + std::to_string(i) + " on device " + std::to_string(devices[i]) + ": " + shards[i].err);
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
	if ((workspaces == nullptr) != (workspace_bytes == nullptr))
		return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_sharded: workspaces and workspace_bytes go together (both NULL = allocate per call)");
	if (plan->d_tables) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_sharded: the plan is bound to one device (pgt_plan_bind_device); unbind it first");
	auto describe = [&](uint32_t i, Shard& s) -> int {
		// the whole axis is addressable from element 0 of the caller's columns; the scan touches only its slabs
		PGT_TRY(pgt_plan_shard(plan, i, ndev, &s.range.w_lo, &s.range.w_hi, nullptr, nullptr));
		// a shard without windows has nothing to do ({0, 0} would even mean "all windows" to pgt_scan) -- except
		// shard 0 of a plan without any window: it owns the axis, whose sites still count for the global line
		s.idle = s.range.w_lo == s.range.w_hi && (pgt_plan_num_windows(plan) != 0 || i != 0);
		if (workspaces && workspaces[i]) {
			s.ws = workspaces[i];
			s.ws_bytes = workspace_bytes[i];
		} else if (!s.idle) {
			s.ws_bytes = pgt_scan_workspace_bytes(plan, &s.range, stat, PGT_MEM_HOST);
		}
		return PGT_OK;
	};
	auto scan = [&](Shard& s, cudaStream_t st) {
		pgt_windows rows = *out;
		for_each_field([d = s.range.w_lo](auto*& p) { p = p ? p + d : p; }, rows);
		rows.dxy_global = out->dxy_global ? s.global3 : nullptr;
		return pgt_scan(plan, &s.range, stat, cols, minind, site_offsets, &rows, s.ws, s.ws_bytes, PGT_MEM_HOST, st);
	};
	std::vector<Shard> shards;
	PGT_TRY(run_shards("pgt_scan_sharded", devices, ndev, shards, describe, scan));
	if (out->dxy_global) {  // the shards own disjoint parts of the axis (pgt_plan_shard): their lines add up, in shard order
		double g3[3] = {0.0, 0.0, 0.0};
		for (const Shard& s : shards)
			for (int q = 0; q < 3; ++q) g3[q] += s.global3[q];
		for (int q = 0; q < 3; ++q) out->dxy_global[q] = g3[q];
	}
	return PGT_OK;
}

// ---- the bp-window extreme-score scan (ihsWindow / xpehhWindow), same scheme: windows do not overlap, so the
// shards need no halo; a shard's columns start at its first site.
extern "C" int pgt_scan_extreme_sharded(const pgt_xplan* plan, pgt_xstat stat, double cutoff, const uint32_t* pos, const double* score,
                                        const pgt_xwindows* out, const int* devices, uint32_t ndev) {
	if (!plan || !score || !out) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_extreme_sharded: plan, score and out must not be NULL");
	auto describe = [&](uint32_t i, Shard& s) -> int {
		uint64_t slo = 0, shi = 0;
		PGT_TRY(pgt_xplan_shard(plan, i, ndev, &s.range.w_lo, &s.range.w_hi, &slo, &shi));
		s.range.site_origin = slo;
		s.range.site_count = shi - slo;
		s.idle = s.range.w_hi <= s.range.w_lo;
		if (!s.idle) s.ws_bytes = pgt_scan_extreme_workspace_bytes(plan, &s.range, PGT_MEM_HOST);
		return PGT_OK;
	};
	auto scan = [&](Shard& s, cudaStream_t st) {
		pgt_xwindows rows = *out;
		for_each_xfield([d = s.range.w_lo](auto*& p) { p = p ? p + d : p; }, rows);
		const uint64_t s0 = s.range.site_origin;
		return pgt_scan_extreme(plan, &s.range, stat, cutoff, pos ? pos + s0 : nullptr, score + s0, &rows, s.ws, s.ws_bytes, PGT_MEM_HOST, st);
	};
	std::vector<Shard> shards;
	return run_shards("pgt_scan_extreme_sharded", devices, ndev, shards, describe, scan);
}

// ---- the extreme score over a window plan, same scheme as pgt_scan_sharded: windows cut by pgt_plan_shard, every shard
// the ordinary host-memory scan over the whole columns (element 0 = site 0); the reduction is exact, so any cut gives
// the same rows.
extern "C" int pgt_scan_plan_extreme_sharded(const pgt_plan* plan, pgt_xstat stat, double cutoff, const uint32_t* pos, const double* score,
                                             const uint64_t* site_offsets, const pgt_windows* rows, const pgt_xwindows* out, const int* devices,
                                             uint32_t ndev) {
	if (!plan || !score || !out) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme_sharded: plan, score and out must not be NULL");
	if (stat != PGT_XSTAT_IHS && stat != PGT_XSTAT_XPEHH) return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme_sharded: unknown statistic");
	if (plan->d_tables)
		return pgt_set_error(PGT_ERR_ARGS, "pgt_scan_plan_extreme_sharded: the plan is bound to one device (pgt_plan_bind_device); unbind it first");
	auto describe = [&](uint32_t i, Shard& s) -> int {
		PGT_TRY(pgt_plan_shard(plan, i, ndev, &s.range.w_lo, &s.range.w_hi, nullptr, nullptr));
		s.idle = s.range.w_lo == s.range.w_hi;  // ({0, 0} would mean "all windows")
		if (!s.idle) s.ws_bytes = pgt_scan_plan_extreme_workspace_bytes(plan, &s.range, PGT_MEM_HOST);
		return PGT_OK;
	};
	auto scan = [&](Shard& s, cudaStream_t st) {
		auto shift = [d = s.range.w_lo](auto*& p) { p = p ? p + d : p; };
		pgt_windows r;
		if (rows) {
			r = *rows;
			for_each_field(shift, r);
		}
		pgt_xwindows x = *out;
		for_each_xfield(shift, x);
		return pgt_scan_plan_extreme(plan, &s.range, stat, cutoff, pos, score, site_offsets, rows ? &r : nullptr, &x, s.ws, s.ws_bytes,
		                             PGT_MEM_HOST, st);
	};
	std::vector<Shard> shards;
	return run_shards("pgt_scan_plan_extreme_sharded", devices, ndev, shards, describe, scan);
}
