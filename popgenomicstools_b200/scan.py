"""Host-side mirror of the reference's window tools over the C ABI (include/pgt_scan.h).

The reference exposes the path only as CLIs; argument names follow them:
``winsize`` / ``stepsize`` as in /root/reference/fstWindow.cpp:158-162 (number of SITES) and
dxyWindow's ``-winsize -stepsize -minind -fixedsite -skip_missing`` (dxyWindow.cpp:34-61).

PyTorch is plumbing only: device memory for columns/outputs/workspace and the current CUDA
stream.  All arithmetic happens in libpgtscan.so's kernels; nothing here computes on the CPU.
"""
import ctypes as C

import numpy as np

from . import _cabi
from ._cabi import WINDOW_FIELDS, PgtColumns, PgtRange, PgtWindows, check


def _torch():
    import torch
    return torch


class _Plan:
    """What WindowPlan and ExtremePlan share: the library handle, the device tables (bind), shard ranges and the cache
    of scan workspaces.  A subclass names its C functions and answers _workspace_bytes(*key)."""
    _destroy = _device_bytes = _bind_device = _shard = None  # names of the plan kind's pgt_* functions

    def __init__(self):
        self._lib = _cabi.load()
        self._h = None
        self._workspaces = {}
        self._bound = None

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            getattr(self._lib, self._destroy)(h)

    @property
    def handle(self):
        return self._h

    def bind(self, device):
        """Keep the plan's device tables resident on `device`: later scans on that device upload nothing.  Called
        automatically by device-mode scans."""
        torch = _torch()
        device = torch.device(device)
        if self._bound is not None and self._bound[0] == device:
            return
        buf = torch.empty(int(getattr(self._lib, self._device_bytes)(self._h)), dtype=torch.uint8, device=device)
        with torch.cuda.device(device):
            check(getattr(self._lib, self._bind_device)(self._h, buf.data_ptr(), buf.numel(),
                                                        C.c_void_p(torch.cuda.current_stream(device).cuda_stream)))
        self._bound = (device, buf)
        self._workspaces = {}

    def shard(self, rank, nranks):
        """Window range [w_lo, w_hi) and site range [site_lo, site_hi) of shard `rank`."""
        v = [C.c_uint64() for _ in range(4)]
        check(getattr(self._lib, self._shard)(self._h, rank, nranks, *[C.byref(x) for x in v]))
        return tuple(x.value for x in v)

    def _workspace(self, device, *key):
        """Device scratch for a scan, cached per (device, tune epoch, key); `key` are the arguments of _workspace_bytes."""
        full = (str(device), _tune_epoch[0]) + key
        ws = self._workspaces.get(full)
        if ws is None:
            torch = _torch()
            ws = torch.empty(self._workspace_bytes(*key), dtype=torch.uint8, device=device)
            self._workspaces[full] = ws
        return ws


class WindowPlan(_Plan):
    """Closed-form window enumeration (pgt_plan_*): which windows the reference would print.

    contig_offsets: cumulative site counts (mode='sites') or chromosome lengths in bp
    (mode='bp'), length ncontig+1, in file order.
    """
    _destroy, _device_bytes, _bind_device, _shard = (
        "pgt_plan_destroy", "pgt_plan_device_bytes", "pgt_plan_bind_device", "pgt_plan_shard")

    def __init__(self, contig_offsets, winsize=1, stepsize=1, mode="sites", unit_sites=0):
        super().__init__()
        self.offsets = np.ascontiguousarray(contig_offsets, dtype=np.uint64)
        if self.offsets.ndim != 1 or len(self.offsets) < 1:
            raise ValueError("contig_offsets must be a 1-D array of length ncontig+1")
        self.winsize, self.stepsize = int(winsize), int(stepsize)
        self.mode = {"sites": _cabi.PGT_MODE_SITES, "bp": _cabi.PGT_MODE_BP}[mode]
        if not (0 <= self.winsize < 2**32 and 0 <= self.stepsize < 2**32):
            raise _cabi.PgtError(_cabi.PGT_ERR_ARGS, "winsize/stepsize out of range")
        h = C.c_void_p()
        check(self._lib.pgt_plan_create(C.byref(h), self.mode, self.offsets.ctypes.data, len(self.offsets) - 1,
                                        self.winsize, self.stepsize, int(unit_sites)))
        self._h = h

    @property
    def num_windows(self):
        return int(self._lib.pgt_plan_num_windows(self._h))

    @property
    def num_units(self):
        return int(self._lib.pgt_plan_num_units(self._h))

    @property
    def num_segments(self):
        return int(self._lib.pgt_plan_num_segments(self._h))

    @property
    def num_sites(self):
        return int(self._lib.pgt_plan_num_sites(self._h))

    def windows(self):
        """(first, last, label) arrays: inclusive site/entry indices and contig index per window."""
        n = self.num_windows
        first, last, label = np.empty(n, np.uint64), np.empty(n, np.uint64), np.empty(n, np.uint32)
        check(self._lib.pgt_plan_windows(self._h, first.ctypes.data, last.ctypes.data, label.ctypes.data))
        return first, last, label

    def unit(self, j):
        st, ln = C.c_uint64(), C.c_uint32()
        check(self._lib.pgt_plan_unit(self._h, j, C.byref(st), C.byref(ln)))
        return st.value, ln.value

    def window_units(self, w):
        f, c = C.c_uint64(), C.c_uint64()
        check(self._lib.pgt_plan_window_units(self._h, w, C.byref(f), C.byref(c)))
        return f.value, c.value

    def scan_path(self, stat):
        """'units' | 'slide' | 'persite': the kernels a scan of `stat` runs (pgt_plan_scan_path)."""
        return ("units", "slide", "persite")[check(self._lib.pgt_plan_scan_path(self._h, stat))]

    def workspace_bytes(self, stat, mem, window_range=None, site_origin=0, site_count=0):
        r = _range(self, window_range, site_origin, site_count)
        return int(self._lib.pgt_scan_workspace_bytes(self._h, C.byref(r), stat, mem))

    def extreme_workspace_bytes(self, mem, window_range=None, site_origin=0, site_count=0):
        """Device scratch of pgt_scan_plan_extreme (scan_extreme over this plan)."""
        r = _range(self, window_range, site_origin, site_count)
        return int(self._lib.pgt_scan_plan_extreme_workspace_bytes(self._h, C.byref(r), mem))

    def _workspace_bytes(self, stat, *key):
        return self.extreme_workspace_bytes(*key) if stat == "extreme" else self.workspace_bytes(stat, *key)

    def workspace(self, device, stat, mem, window_range=None, site_origin=0, site_count=0):
        """Device scratch for a scan, cached per (device, stat, mem, range)."""
        return self._workspace(device, stat, mem, window_range, site_origin, site_count)


def _range(plan, window_range, site_origin, site_count=0):
    lo, hi = (0, plan.num_windows) if window_range is None else window_range
    return PgtRange(int(lo), int(hi), int(site_origin), int(site_count))


_tune_epoch = [0]

_COL_DTYPES = {"pos": "uint32", "a": "float64", "b": "float64", "geno": "int8", "f1": "float64", "f2": "float64",
               "n1": "int32", "n2": "int32", "score": "float64"}
_W_DTYPES = {k: "float64" if k in ("sum_a", "sum_b", "fst", "het", "dxy", "dxy_global") else "uint32" for k in WINDOW_FIELDS}
_STAT_COLS = {
    _cabi.PGT_STAT_FST: ("a", "b"),
    _cabi.PGT_STAT_HET: ("geno",),
    _cabi.PGT_STAT_DXY: ("f1", "f2", "n1", "n2"),
    _cabi.PGT_STAT_FUSED: ("a", "b", "geno", "f1", "f2", "n1", "n2"),
}
_STAT_OUTS = {
    _cabi.PGT_STAT_FST: ("label", "start_pos", "end_pos", "mid_pos", "nsites", "sum_a", "sum_b", "fst"),
    _cabi.PGT_STAT_HET: ("label", "start_pos", "end_pos", "mid_pos", "nsites", "nhet", "nonmissing", "het"),
    _cabi.PGT_STAT_DXY: ("label", "start_pos", "end_pos", "nsites", "dxy", "neffective", "nskip", "dxy_global"),
    _cabi.PGT_STAT_FUSED: WINDOW_FIELDS,
}


def _columns(cols, names, need, on_device):
    """Data pointers of the columns `names` found in `cols` (name -> array), checked against their dtypes: contiguous
    CUDA tensors if `on_device`, else numpy arrays (CPU tensors are viewed as numpy).  int32 positions are viewed as
    uint32.  Every column of `need` must be present.  Returns (name -> pointer, the arrays to keep alive)."""
    for k in need:
        if cols.get(k) is None:
            raise ValueError(f"column {k!r} is required")
    torch = _torch()
    ptrs, keep = {}, []
    for k in names:
        v = cols.get(k)
        if v is None:
            continue
        want = _COL_DTYPES[k]
        if on_device:
            if not (isinstance(v, torch.Tensor) and v.is_cuda and v.is_contiguous()):
                raise TypeError(f"{k}: expected a contiguous CUDA tensor")
            if k == "pos" and v.dtype == torch.int32:
                v = v.view(torch.uint32)
            if str(v.dtype) != "torch." + want:
                raise TypeError(f"{k}: expected {want}, got {v.dtype}")
            ptrs[k] = v.data_ptr()
        else:
            if isinstance(v, torch.Tensor):
                v = v.numpy()
            if k == "pos" and v.dtype == np.int32:
                v = v.view(np.uint32)
            if v.dtype != np.dtype(want) or not v.flags["C_CONTIGUOUS"]:
                raise TypeError(f"{k}: expected contiguous {want}, got {v.dtype}")
            ptrs[k] = v.ctypes.data
        keep.append(v)
    return ptrs, keep


def _table(struct, out, names, dtypes, nrows, device):
    """A result table: `out` (name -> array), or if it is None new arrays `names` of `nrows` rows (dxy_global: 3) and
    `dtypes` -- CUDA tensors on `device`, numpy arrays if `device` is None.  Returns (out, `struct` pointing at it)."""
    if out is None:
        if device is None:
            out = {k: np.empty(3 if k == "dxy_global" else nrows, dtypes[k]) for k in names}
        else:
            torch = _torch()
            out = {k: torch.empty(3 if k == "dxy_global" else nrows, dtype=getattr(torch, dtypes[k]), device=device) for k in names}
    t = struct()
    for k, _ in struct._fields_:
        v = out.get(k)
        if v is not None:
            setattr(t, k, v.ctypes.data if device is None else v.data_ptr())
    return out, t


def scan(plan, stat, cols, minind=1, site_offsets=None, window_range=None, site_origin=0, site_count=0, out=None,
         device=None):
    """Generic entry (pgt_scan).  `cols`: dict name -> column.  CUDA tensors select
    PGT_MEM_DEVICE (enqueued on the current stream, returns CUDA tensors, not synchronised);
    numpy arrays select PGT_MEM_HOST (staged through the device, returns numpy arrays)."""
    torch = _torch()
    lib = plan._lib
    need = _STAT_COLS[stat]
    sample = cols.get(need[0])
    on_device = isinstance(sample, torch.Tensor) and sample.is_cuda
    ptrs, keep = _columns(cols, ("pos",) + need, need, on_device)
    c = PgtColumns(**ptrs)
    r = _range(plan, window_range, site_origin, site_count)
    dev = sample.device if on_device else torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    out, w = _table(PgtWindows, out, _STAT_OUTS[stat], _W_DTYPES, r.w_hi - r.w_lo, dev if on_device else None)
    so = None
    if site_offsets is not None:
        so = np.ascontiguousarray(site_offsets, dtype=np.uint64)
        keep.append(so)
    mem = _cabi.PGT_MEM_DEVICE if on_device else _cabi.PGT_MEM_HOST
    if on_device:
        plan.bind(dev)
    elif plan._bound is not None and plan._bound[0] != dev:
        raise ValueError(f"plan is bound to {plan._bound[0]}, scan requested on {dev}")
    ws = plan._workspace(dev, stat, mem, window_range, site_origin, site_count)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(lib.pgt_scan(plan.handle, C.byref(r), stat, C.byref(c), int(minind), so.ctypes.data if so is not None else None,
                           C.byref(w), ws.data_ptr(), ws.numel(), mem, C.c_void_p(stream)))
    return out


def scan_sharded(plan, stat, cols, devices, minind=1, site_offsets=None, out=None):
    """One host column set, several GPUs of this process (pgt_scan_sharded): `cols` are numpy arrays over the
    WHOLE axis, `devices` a list of CUDA device indices (one shard per entry).  Returns numpy arrays over all
    windows; per-window results are bit-identical for any device list."""
    lib = plan._lib
    need = _STAT_COLS[stat]
    ptrs, keep = _columns(cols, ("pos",) + need, need, False)
    c = PgtColumns(**ptrs)
    out, w = _table(PgtWindows, out, _STAT_OUTS[stat], _W_DTYPES, plan.num_windows, None)
    so = None if site_offsets is None else np.ascontiguousarray(site_offsets, dtype=np.uint64)
    dev = (C.c_int * len(devices))(*[int(d) for d in devices])
    check(lib.pgt_scan_sharded(plan.handle, stat, C.byref(c), int(minind), so.ctypes.data if so is not None else None, C.byref(w),
                               dev, len(devices), None, None))
    return out


def fst_window(plan, pos, a, b, site_offsets=None, **kw):
    """Sliding-window FST = sum(a)/sum(b) (/root/reference/fstWindow.cpp:69-107).  plan mode 'sites' = windows of
    sites as fstWindow; 'bp' = fixed-bp windows over the sites whose positions fall on them (then site_offsets =
    cumulative sites per chromosome, and nsites counts bp: see bp_window_sites).
    Returns label, start_pos, end_pos, mid_pos, nsites, sum_a, sum_b, fst per window."""
    return scan(plan, _cabi.PGT_STAT_FST, dict(pos=pos, a=a, b=b), site_offsets=site_offsets, **kw)


def het_window(plan, pos, geno, site_offsets=None, **kw):
    """Sliding-window heterozygosity = #(g==1) / #(g>=0) (/root/reference/hetWindow.cpp:66-105).
    The counts are integers, so any unit size gives identical results; build the plan with
    ``unit_sites=4096`` for the fastest scan of the 1-byte genotype column.  plan mode and site_offsets as for
    fst_window.
    Returns label, start_pos, end_pos, mid_pos, nsites, nhet, nonmissing, het per window."""
    return scan(plan, _cabi.PGT_STAT_HET, dict(pos=pos, geno=geno), site_offsets=site_offsets, **kw)


def dxy_window(plan, pos, f1, f2, n1, n2, minind=1, site_offsets=None, **kw):
    """Sliding-window dxy = sum of f1(1-f2)+f2(1-f1) over sites with nInd >= minind in both
    populations (/root/reference/dxyWindow.cpp:172-209,381).  plan mode 'sites' = -fixedsite 1,
    'bp' = -fixedsite 0 (then site_offsets = cumulative sites per chromosome).  -skip_missing 1
    is the row filter ``neffective > 0``.  Returns label, start_pos, end_pos, nsites, dxy,
    neffective, nskip per window and dxy_global[3]."""
    return scan(plan, _cabi.PGT_STAT_DXY, dict(pos=pos, f1=f1, f2=f2, n1=n1, n2=n2), minind=minind,
                site_offsets=site_offsets, **kw)


def fused_window(plan, pos, a, b, geno, f1, f2, n1, n2, minind=1, site_offsets=None, **kw):
    """fst + dxy + het over one site axis in a single pass (BASELINE config 5); plan mode and site_offsets as for
    dxy_window.  Each statistic equals its single scan bit for bit."""
    return scan(plan, _cabi.PGT_STAT_FUSED, dict(pos=pos, a=a, b=b, geno=geno, f1=f1, f2=f2, n1=n1, n2=n2),
                minind=minind, site_offsets=site_offsets, **kw)


def bp_window_sites(plan, pos, site_offsets, window_range=None, site_origin=0, site_count=0, out=None, device=None):
    """Sites per window of a bp plan (pgt_scan_bp_sites): the number of sites whose positions fall on each window's
    bp, for the rows of a scan over the same plan and window range (whose ``nsites`` counts bp).  `pos` a CUDA
    tensor (PGT_MEM_DEVICE: enqueued on the current stream, returns a CUDA uint32 tensor) or a numpy array
    (PGT_MEM_HOST: returns a numpy uint32 array).  Raises PgtError (PGT_ERR_INPUT) when a site lies outside its
    chromosome; the call waits for the stream to report that."""
    torch = _torch()
    lib = plan._lib
    on_device = isinstance(pos, torch.Tensor) and pos.is_cuda
    ptrs, keep = _columns(dict(pos=pos), ("pos",), ("pos",), on_device)
    r = _range(plan, window_range, site_origin, site_count)
    so = np.ascontiguousarray(site_offsets, dtype=np.uint64)
    nrows = r.w_hi - r.w_lo
    dev = pos.device if on_device else torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    if out is None:
        out = torch.empty(nrows, dtype=torch.uint32, device=dev) if on_device else np.empty(nrows, np.uint32)
    mem = _cabi.PGT_MEM_DEVICE if on_device else _cabi.PGT_MEM_HOST
    if on_device:
        plan.bind(dev)
    elif plan._bound is not None and plan._bound[0] != dev:
        raise ValueError(f"plan is bound to {plan._bound[0]}, scan requested on {dev}")
    ws = torch.empty(int(lib.pgt_scan_bp_sites_workspace_bytes(plan.handle, C.byref(r), so.ctypes.data, mem)), dtype=torch.uint8,
                     device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(lib.pgt_scan_bp_sites(plan.handle, C.byref(r), ptrs["pos"], so.ctypes.data,
                                    out.data_ptr() if on_device else out.ctypes.data, ws.data_ptr(), ws.numel(), mem,
                                    C.c_void_p(stream)))
    return out


# ---- synthetic inputs (device) -------------------------------------------------------------

def _stream(t):
    torch = _torch()
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def synth_fst(seed, site0, n, device="cuda"):
    torch = _torch()
    lib = _cabi.load()
    a = torch.empty(n, dtype=torch.float64, device=device)
    b = torch.empty(n, dtype=torch.float64, device=device)
    with torch.cuda.device(a.device):
        check(lib.pgt_synth_fst(seed, site0, n, a.data_ptr(), b.data_ptr(), _stream(a)))
    return a, b


def synth_het(seed, site0, n, device="cuda"):
    torch = _torch()
    lib = _cabi.load()
    g = torch.empty(n, dtype=torch.int8, device=device)
    with torch.cuda.device(g.device):
        check(lib.pgt_synth_het(seed, site0, n, g.data_ptr(), _stream(g)))
    return g


def synth_dxy(seed, site0, n, device="cuda"):
    torch = _torch()
    lib = _cabi.load()
    f1 = torch.empty(n, dtype=torch.float64, device=device)
    f2 = torch.empty(n, dtype=torch.float64, device=device)
    n1 = torch.empty(n, dtype=torch.int32, device=device)
    n2 = torch.empty(n, dtype=torch.int32, device=device)
    with torch.cuda.device(f1.device):
        check(lib.pgt_synth_dxy(seed, site0, n, f1.data_ptr(), f2.data_ptr(), n1.data_ptr(), n2.data_ptr(), _stream(f1)))
    return f1, f2, n1, n2


def synth_pos(seed, site0, n, contig_offsets, density=1, device="cuda"):
    torch = _torch()
    lib = _cabi.load()
    off = np.ascontiguousarray(contig_offsets, dtype=np.uint64)
    pos = torch.empty(n, dtype=torch.uint32, device=device)
    with torch.cuda.device(pos.device):
        check(lib.pgt_synth_pos(seed, site0, n, off.ctypes.data, len(off) - 1, density, pos.data_ptr(), _stream(pos)))
    return pos


def kernel_launch_count():
    return int(_cabi.load().pgt_kernel_launch_count())


def profile(enable):
    """Bracket every level-1 / level-2 launch with CUDA events (see pgt_profile)."""
    check(_cabi.load().pgt_profile(1 if enable else 0))


def profile_read():
    """-> dict(units_ms, units_launches, windows_ms, windows_launches) since the last read."""
    um, wm = C.c_double(), C.c_double()
    un, wn = C.c_uint64(), C.c_uint64()
    check(_cabi.load().pgt_profile_read(C.byref(um), C.byref(un), C.byref(wm), C.byref(wn)))
    return dict(units_ms=um.value, units_launches=un.value, windows_ms=wm.value, windows_launches=wn.value)


def tune(key, value):
    """Kernel-selection knobs for tests/experiments (pgt_tune).  Some knobs change the workspace a scan
    needs, so cached workspaces are re-queried afterwards."""
    check(_cabi.load().pgt_tune(key.encode(), int(value)))
    _tune_epoch[0] += 1
