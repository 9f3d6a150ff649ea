"""Host build of the rescoring kernels' shared-memory layout (csrc/stage_window.h, through tests/native/
stage_window_harness.cpp): the staged-row window and the band capacity of every shape, computed by the same code the
library launches with.  Used by test_stage_window_cpu.py, which checks the layout, and by test_rescore_window_gpu.py,
which picks its dims and band sizes from it."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "real-time-brain-inspired-video-memory_b200", "csrc")

SM_COUNT = 148              # B200: CTAs of the tcgen05 scan, half the lists of the CUDA-core scan
KP_TC = (32, 64)            # candidate rows of the tcgen05 scan (k <= 16, k <= 48)
KP_SIMT = (16, 24, 32)      # candidate rows of the CUDA-core scan (k <= 8, k <= 16, k <= 24)
ELEM_BYTES = {"bf16": 2, "f32": 4, "f64": 8}
SLAB = 0                    # key source: the tcgen05 scan's union buffer (SELECT_KEY_CAP keys)


class Harness:
    def __init__(self, out_dir):
        so = os.path.join(str(out_dir), "libstage_window.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                               os.path.join(ROOT, "tests", "native", "stage_window_harness.cpp"), "-o", so])
        L = C.CDLL(so)
        L.select_stage.argtypes = [C.c_int] * 6 + [C.c_void_p]
        L.collect_stage.argtypes = [C.c_int] * 3 + [C.c_void_p]
        L.stage_constants.argtypes = [C.c_void_p]
        L.stage_walk.argtypes = [C.c_int] * 3 + [C.c_void_p] * 2
        L.stage_walk.restype = C.c_int
        self.L = L
        c = np.zeros(9, np.int64)
        L.stage_constants(c.ctypes.data)
        (self.SELECT_KEY_CAP, self.SCAN_DUMP_TILE, self.SCAN_DUMP_MAX_KEYS, self.COLLECT_CAP, self.SR_SMEM_LIMIT,
         self.CR_SMEM_LIMIT, self.BAND_CAP_MIN, self.BAND_CAP_MAX, self.CR_ROWS) = (int(v) for v in c)

    def select(self, elem_bytes, kp, lists=0, list_len=0, dims=(1, 4097)):
        """Layout of select_rescore_kernel for every dim in range(*dims): int64 [n][6] = fits, gpr, pitch (bytes),
        chunks, band_cap, smem.  lists == 0: slab mode; else list mode with lists x list_len keys."""
        out = np.zeros((dims[1] - dims[0], 6), np.int64)
        self.L.select_stage(elem_bytes, kp, lists, list_len, dims[0], dims[1], out.ctypes.data)
        return out

    def collect(self, elem_bytes, dims=(1, 4097)):
        """Layout of collect_rescore_kernel for every dim in range(*dims): int64 [n][5] = rows, gpr, pitch, chunks, smem."""
        out = np.zeros((dims[1] - dims[0], 5), np.int64)
        self.L.collect_stage(elem_bytes, dims[0], dims[1], out.ctypes.data)
        return out

    def walk(self, gpr, pitch, chunks):
        """-> (rule broken or 0, first group of every chunk [chunks + 1], first group of its slot [chunks + 1])."""
        lo = np.zeros(chunks + 1, np.int32)
        slot = np.zeros(chunks + 1, np.int32)
        rc = self.L.stage_walk(int(gpr), int(pitch), int(chunks), lo.ctypes.data, slot.ctypes.data)
        return rc, lo, slot

    def dump_tiles(self, n):
        """Dump-mode key source of an n-row store (every row's key, one 128-key list per tile), or None when the
        store has too many rows for it."""
        tiles = (n + 127) // 128
        ok = tiles <= SM_COUNT and tiles * self.SCAN_DUMP_TILE <= self.SCAN_DUMP_MAX_KEYS
        return (tiles, self.SCAN_DUMP_TILE) if ok else None

    def stage_regime(self, elem_bytes, dim, kp, key_source=SLAB):
        """(chunks, pitch, band_cap) of select_rescore_kernel for one shape.  key_source: SLAB, or (lists, list_len)."""
        lists, list_len = (0, 0) if key_source == SLAB else key_source
        fits, _, pitch, chunks, band_cap, _ = (int(v) for v in self.select(elem_bytes, kp, lists, list_len, (dim, dim + 1))[0])
        assert fits, (elem_bytes, dim, kp, key_source)
        return chunks, pitch, band_cap

    def collect_regime(self, elem_bytes, dim):
        """(chunks, pitch) of collect_rescore_kernel for one shape."""
        _, _, pitch, chunks, _ = (int(v) for v in self.collect(elem_bytes, (dim, dim + 1))[0])
        return chunks, pitch
