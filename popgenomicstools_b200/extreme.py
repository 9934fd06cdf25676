"""Host-side mirror of ihsWindow / xpehhWindow over the C ABI (include/pgt_extreme.h).

Argument names follow the tools: ``winsize`` (bp, /root/reference/ihsWindow.cpp:47-52),
``cutoff`` (ihsWindow.cpp:54-59; positional for xpehhWindow, xpehhWindow.cpp:55) and ``chrlen``
(the -chrlen table, ihsWindow.cpp:60-65).  PyTorch is plumbing only (device memory, current
stream); the reduction runs in libpgtscan.so's kernels and nothing here computes on the CPU
except the window bookkeeping the library itself does on the host (pgt_xplan_create).
"""
import ctypes as C

import numpy as np

from . import _cabi
from ._cabi import PgtRange, PgtWindows, PgtXWindows, check
from .scan import WindowPlan, _Plan, _columns, _range, _table, _torch

XWINDOW_FIELDS = _cabi.XWINDOW_FIELDS
_X_DTYPES = {"ext_value": "float64", "ext_pos": "uint32", "ext_site": "uint64", "nbig": "uint32", "nsites": "uint32",
             "prop": "float64"}
_XFIELDS_NO_POS = tuple(k for k in XWINDOW_FIELDS if k != "ext_pos")
# rows of a scan over a WindowPlan: pgt_scan's geometry beside the extreme fields (whose nsites counts score sites)
_GEO_FIELDS = ("label", "start_pos", "end_pos", "mid_pos")
_PLAN_DTYPES = dict(_X_DTYPES, **dict.fromkeys(_GEO_FIELDS, "uint32"))


def _plan_tables(out, pos, nrows, device):
    """Result table of pgt_scan_plan_extreme: (out, PgtWindows with the geometry columns only, PgtXWindows).  Without
    `pos` there are no positions: label and the extreme fields but ext_pos."""
    names = ("label",) + _XFIELDS_NO_POS if pos is None else _GEO_FIELDS + XWINDOW_FIELDS
    out, x = _table(PgtXWindows, out, names, _PLAN_DTYPES, nrows, device)
    g = PgtWindows()
    for k in _GEO_FIELDS:
        v = out.get(k)
        if v is not None:
            setattr(g, k, v.ctypes.data if device is None else v.data_ptr())
    return out, g, x


def _site_offsets(plan, site_offsets):
    if plan.mode == _cabi.PGT_MODE_BP and site_offsets is None:
        raise ValueError("a bp plan needs site_offsets (cumulative sites per chromosome)")
    return None if site_offsets is None else np.ascontiguousarray(site_offsets, dtype=np.uint64)


class ExtremePlan(_Plan):
    """Window bookkeeping of ihsWindow / xpehhWindow (pgt_xplan_*): which rows the reference prints
    and which sites each window holds.

    pos: HOST position column (numpy uint32, file order); contig_offsets: cumulative site counts of
    the runs of equal chromosome name; chrlen: per-run -chrlen length (0 = not listed) or None.
    """
    _destroy, _device_bytes, _bind_device, _shard = (
        "pgt_xplan_destroy", "pgt_xplan_device_bytes", "pgt_xplan_bind_device", "pgt_xplan_shard")

    def __init__(self, pos, contig_offsets, winsize=100000, chrlen=None, unit_sites=0):
        super().__init__()
        self.pos = np.ascontiguousarray(pos, dtype=np.uint32)
        self.offsets = np.ascontiguousarray(contig_offsets, dtype=np.uint64)
        ncontig = len(self.offsets) - 1
        if self.offsets.ndim != 1 or ncontig < 1:
            raise ValueError("contig_offsets must be a 1-D array of length ncontig+1")
        if len(self.pos) != int(self.offsets[-1]):
            raise ValueError("pos must hold contig_offsets[-1] sites")
        self.chrlen = None if chrlen is None else np.ascontiguousarray(chrlen, dtype=np.uint32)
        if self.chrlen is not None and len(self.chrlen) != ncontig:
            raise ValueError("chrlen must have one entry per contig run")
        if not 0 <= int(winsize) < 2**32:
            raise _cabi.PgtError(_cabi.PGT_ERR_ARGS, "winsize out of range")
        self.winsize = int(winsize)
        h = C.c_void_p()
        check(self._lib.pgt_xplan_create(C.byref(h), self.pos.ctypes.data, self.offsets.ctypes.data,
                                         self.chrlen.ctypes.data if self.chrlen is not None else None, ncontig, self.winsize,
                                         int(unit_sites)))
        self._h = h

    @property
    def num_windows(self):
        return int(self._lib.pgt_xplan_num_windows(self._h))

    @property
    def num_units(self):
        return int(self._lib.pgt_xplan_num_units(self._h))

    @property
    def num_sites(self):
        return int(self._lib.pgt_xplan_num_sites(self._h))

    def windows(self):
        """dict(label, start, end, first_site, nsites): the printed window table (numpy)."""
        n = self.num_windows
        o = dict(label=np.empty(n, np.uint32), start=np.empty(n, np.uint32), end=np.empty(n, np.uint32),
                 first_site=np.empty(n, np.uint64), nsites=np.empty(n, np.uint32))
        check(self._lib.pgt_xplan_windows(self._h, *[o[k].ctypes.data for k in ("label", "start", "end", "first_site", "nsites")]))
        return o

    def _workspace_bytes(self, mem, window_range, site_origin):
        r = _xrange(self, window_range, site_origin)
        return int(self._lib.pgt_scan_extreme_workspace_bytes(self._h, C.byref(r), mem))

    def workspace(self, device, mem, window_range=None, site_origin=0):
        return self._workspace(device, mem, window_range, site_origin)


def _xrange(plan, window_range, site_origin):
    lo, hi = (0, plan.num_windows) if window_range is None else window_range
    return PgtRange(int(lo), int(hi), int(site_origin), 0)


def scan_extreme(plan, stat, cutoff, pos, score, window_range=None, site_origin=0, out=None, device=None, site_offsets=None):
    """pgt_scan_extreme over an ExtremePlan (ihsWindow's windows), or pgt_scan_plan_extreme over a WindowPlan (sliding
    site / bp windows whose rows line up with fst_window's over the same plan; `site_offsets` as for fst_window, required
    for a bp plan; label, start_pos, end_pos, mid_pos come back too, and nsites counts score sites).  CUDA tensors
    select PGT_MEM_DEVICE (enqueued on the current stream, CUDA tensors back, not synchronised -- except over a bp
    WindowPlan, where the call waits for the stream to report a position outside its chromosome, as bp_window_sites);
    numpy arrays select PGT_MEM_HOST (numpy arrays back).  The rows do not depend on the plan's unit_sites; long windows
    scan fastest over a plan built with unit_sites=2048 (1e9 sites at 50000/10000: 1.29 ms against 2.06 ms)."""
    if isinstance(plan, WindowPlan):
        return _scan_plan_extreme(plan, stat, cutoff, pos, score, window_range, site_origin, out, device, site_offsets)
    if site_offsets is not None:
        raise ValueError("site_offsets applies to a WindowPlan")
    torch = _torch()
    lib = plan._lib
    on_device = isinstance(score, torch.Tensor) and score.is_cuda
    r = _xrange(plan, window_range, site_origin)
    ptrs, keep = _columns(dict(pos=pos, score=score), ("pos", "score"), (), on_device)
    dev = score.device if on_device else torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    names = XWINDOW_FIELDS if pos is not None else _XFIELDS_NO_POS
    out, w = _table(PgtXWindows, out, names, _X_DTYPES, r.w_hi - r.w_lo, dev if on_device else None)
    mem = _cabi.PGT_MEM_DEVICE if on_device else _cabi.PGT_MEM_HOST
    if on_device:
        plan.bind(dev)
    elif plan._bound is not None and plan._bound[0] != dev:
        raise ValueError(f"plan is bound to {plan._bound[0]}, scan requested on {dev}")
    ws = plan._workspace(dev, mem, window_range, site_origin)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(lib.pgt_scan_extreme(plan.handle, C.byref(r), int(stat), float(cutoff), ptrs.get("pos"), ptrs.get("score"), C.byref(w),
                                   ws.data_ptr(), ws.numel(), mem, C.c_void_p(stream)))
    return out


def _scan_plan_extreme(plan, stat, cutoff, pos, score, window_range, site_origin, out, device, site_offsets):
    torch = _torch()
    lib = plan._lib
    on_device = isinstance(score, torch.Tensor) and score.is_cuda
    so = _site_offsets(plan, site_offsets)
    r = _range(plan, window_range, site_origin)
    ptrs, keep = _columns(dict(pos=pos, score=score), ("pos", "score"), ("score",), on_device)
    dev = score.device if on_device else torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    out, g, x = _plan_tables(out, pos, r.w_hi - r.w_lo, dev if on_device else None)
    mem = _cabi.PGT_MEM_DEVICE if on_device else _cabi.PGT_MEM_HOST
    if on_device:
        plan.bind(dev)
    elif plan._bound is not None and plan._bound[0] != dev:
        raise ValueError(f"plan is bound to {plan._bound[0]}, scan requested on {dev}")
    ws = plan._workspace(dev, "extreme", mem, window_range, site_origin)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(lib.pgt_scan_plan_extreme(plan.handle, C.byref(r), int(stat), float(cutoff), ptrs.get("pos"), ptrs["score"],
                                        so.ctypes.data if so is not None else None, C.byref(g), C.byref(x), ws.data_ptr(), ws.numel(),
                                        mem, C.c_void_p(stream)))
    return out


def scan_extreme_sharded(plan, stat, cutoff, pos, score, devices, site_offsets=None):
    """pgt_scan_extreme_sharded (ExtremePlan) or pgt_scan_plan_extreme_sharded (WindowPlan, rows as scan_extreme's):
    numpy columns over ALL sites, one shard of windows per entry of `devices` (CUDA device indices of this process);
    numpy arrays over all windows back, bit-identical for any list."""
    lib = plan._lib
    pos = None if pos is None else np.ascontiguousarray(pos, np.uint32)
    score = np.ascontiguousarray(score, np.float64)
    dev = (C.c_int * len(devices))(*[int(d) for d in devices])
    if isinstance(plan, WindowPlan):
        so = _site_offsets(plan, site_offsets)
        out, g, x = _plan_tables(None, pos, plan.num_windows, None)
        check(lib.pgt_scan_plan_extreme_sharded(plan.handle, int(stat), float(cutoff), pos.ctypes.data if pos is not None else None,
                                                score.ctypes.data, so.ctypes.data if so is not None else None, C.byref(g), C.byref(x),
                                                dev, len(devices)))
        return out
    if site_offsets is not None:
        raise ValueError("site_offsets applies to a WindowPlan")
    out, w = _table(PgtXWindows, None, XWINDOW_FIELDS if pos is not None else _XFIELDS_NO_POS, _X_DTYPES, plan.num_windows, None)
    check(lib.pgt_scan_extreme_sharded(plan.handle, int(stat), float(cutoff), pos.ctypes.data if pos is not None else None,
                                       score.ctypes.data, C.byref(w), dev, len(devices)))
    return out


def ihs_window(plan, pos, score, cutoff=2.0, **kw):
    """Most extreme |iHS| per bp window and the proportion of |iHS| > cutoff
    (/root/reference/ihsWindow.cpp:93-187).  Returns ext_value (signed score), ext_pos, ext_site,
    nbig, nsites, prop per window; empty windows have nsites 0 and NaN ext_value / prop.  `plan` an ExtremePlan
    (ihsWindow's windows) or a WindowPlan (sliding windows, see scan_extreme)."""
    return scan_extreme(plan, _cabi.PGT_XSTAT_IHS, cutoff, pos, score, **kw)


def xpehh_window(plan, pos, score, cutoff, **kw):
    """Most extreme XP-EHH per bp window: cutoff < 0 -> minimum and proportion below the cutoff,
    else maximum and proportion above it (/root/reference/xpehhWindow.cpp:87-193)."""
    return scan_extreme(plan, _cabi.PGT_XSTAT_XPEHH, cutoff, pos, score, **kw)


def synth_score(seed, site0, n, device="cuda"):
    torch = _torch()
    s = torch.empty(n, dtype=torch.float64, device=device)
    with torch.cuda.device(s.device):
        check(_cabi.load().pgt_synth_score(seed, site0, n, s.data_ptr(), C.c_void_p(torch.cuda.current_stream(s.device).cuda_stream)))
    return s


def profile_read_extreme():
    """-> dict(units_ms, units_launches, windows_ms, windows_launches) of the extreme scan since the last read."""
    um, wm = C.c_double(), C.c_double()
    un, wn = C.c_uint64(), C.c_uint64()
    check(_cabi.load().pgt_profile_read_extreme(C.byref(um), C.byref(un), C.byref(wm), C.byref(wn)))
    return dict(units_ms=um.value, units_launches=un.value, windows_ms=wm.value, windows_launches=wn.value)
