"""The fused tick with several count lines per stream on host memory (tests/hostemu/dd_hostemu_lines.cpp, g++).  TEST
SCAFFOLDING."""
import ctypes
import os
import subprocess

import numpy as np

from . import build as _build
from .driver import _p
from .tick import HostEmuTickTracker

SO = os.path.join(_build.HERE, "libdd_hostemu_lines.so")
SRC = os.path.join(_build.HERE, "dd_hostemu_lines.cpp")
_lib = None


def build(force=False):
    deps = [SRC] + [os.path.join(_build.CSRC, f) for f in os.listdir(_build.CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(_build.HERE, "..", "..", "include", "deepdish_b200.h"))
    if not force and os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in deps):
        return SO
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++", SRC,
                           "-o", SO])
    return SO


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


class HostEmuLinesTracker(HostEmuTickTracker):
    """HostEmuTickTracker whose tick counts cfg.n_lines > 1 lines per stream: lines f64 [S,L,4]."""

    def __init__(self, cfg, lines):
        super().__init__(cfg)
        self.lines = np.ascontiguousarray(lines, np.float64)
        assert self.lines.shape == (cfg.n_streams, cfg.n_lines, 4)

    def tick(self, tlwh, conf, label, feat, count, present=None):
        self._keep = [np.ascontiguousarray(tlwh, np.float64), np.ascontiguousarray(conf, np.float32),
                      np.ascontiguousarray(label, np.int32), np.ascontiguousarray(feat, np.float32),
                      np.ascontiguousarray(count, np.int32)]
        pr = None if present is None else np.ascontiguousarray(np.asarray(present).astype(np.uint8))
        a = self._keep
        rc = lib().ddh_tracker_tick_lines(_p(self.blob), ctypes.byref(self.cfg), _p(a[0]), _p(a[1]), _p(a[2]),
                                          _p(a[3]), _p(a[4]), _p(pr) if pr is not None else None, _p(self.lines),
                                          _p(self.det_track_id))
        assert rc == 0
        return self.det_track_id

    def events(self):
        """(records this tick, the rows written: int32 [min(n, cap), 4])."""
        ev = self.v["events"]
        n = int(ev[0, 0])
        return n, ev[1:1 + min(n, self.cfg.event_cap)].copy()
