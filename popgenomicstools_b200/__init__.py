"""popgenomicstools_b200 -- B200-native windowed site-statistic scan (fstWindow / hetWindow / dxyWindow hot path,
plus the bp-window extreme-score scans of ihsWindow / xpehhWindow).

Thin host layer over libpgtscan.so (hand-written sm_100a kernels behind the C ABI of
include/pgt_scan.h).  Importing the package loads the shared library and fails loudly if it is
not built; there is no CPU fallback anywhere in the product path.
"""
from . import _cabi
from ._cabi import PgtError

_cabi.load()

from .scan import (WindowPlan, bp_window_sites, dxy_window, fst_window, fused_window, het_window, kernel_launch_count, scan, scan_sharded,  # noqa: E402
                   synth_dxy, synth_fst, synth_het, synth_pos, profile, profile_read, tune)

from .extreme import (ExtremePlan, ihs_window, profile_read_extreme, scan_extreme, scan_extreme_sharded, synth_score, xpehh_window)  # noqa: E402

__all__ = ["ExtremePlan", "scan_extreme", "scan_extreme_sharded", "ihs_window", "xpehh_window", "synth_score", "WindowPlan", "scan", "scan_sharded", "fst_window", "het_window", "dxy_window", "fused_window", "bp_window_sites", "synth_fst", "synth_het",
           "synth_dxy", "synth_pos", "kernel_launch_count", "PgtError"]
