"""tests/translate_host.py — TEST INFRASTRUCTURE: runs the translator's GENERATED SOURCE on the CPU.

The CUDA source that fx8010_translate_source emits for a program also compiles as plain C++ with
-DFXT_HOST_CHECK (small shims restate the rounded intrinsics with IEEE operations under -ffp-contract=off).
HostTranslated compiles it with g++ and drives the per-instance function over state arrays laid out like the
device's, so the code generator — operand folding, SKIP branches, counters, TRAM, noise, output latches — is
checked against the oracle in this container, without a GPU.  The product never uses this path.
"""
import ctypes as C
import hashlib
import importlib
import os
import subprocess
import tempfile

import numpy as np

PKG = "fx8010-emulator-core_b200"
SEED1, SEED2 = 0x70f4f854, 0xe1e9f0a7
_cache = {}


def device_tables(tables: np.ndarray) -> np.ndarray:
    """[2][32][64] doubles -> [2][32][64][2] {T[i], (T[i+1]-T[i])/(x2-x1)} as fx8010_gpu_load_program builds them (T[64] = 0)."""
    t = np.ascontiguousarray(tables, dtype=np.float64)
    step = np.float64(2.0) / np.float64(63.0)
    i = np.arange(64, dtype=np.float64)
    x1 = np.float64(-1.0) + i * step
    x2 = np.float64(-1.0) + (i + 1.0) * step
    nxt = np.concatenate([t[:, :, 1:], np.zeros((2, 32, 1))], axis=2)
    out = np.zeros((2, 32, 64, 2), dtype=np.float64)
    out[..., 0] = t
    out[..., 1] = (nxt - t) / (x2 - x1)
    return out


def compile_source(src: str) -> C.CDLL:
    key = hashlib.sha1(src.encode()).hexdigest()
    if key in _cache:
        return _cache[key]
    d = tempfile.mkdtemp(prefix="fxt_")
    cu = os.path.join(d, "t.cpp")
    so = os.path.join(d, "t.so")
    open(cu, "w").write(src)
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-DFXT_HOST_CHECK", "-o", so, cu], check=True)
    lib = C.CDLL(so)
    if hasattr(lib, "fx_translated_host"):
        lib.fx_translated_host.restype = None
        lib.fx_translated_host.argtypes = [C.c_int] + [C.c_void_p] * 12 + [C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int]
    else:                       # stateless program: the streaming kernel, one call per (thread, blockIdx.y)
        lib.fx_translated_sl_host.restype = None
        lib.fx_translated_sl_host.argtypes = [C.c_int, C.c_int, FxtIo] + [C.c_void_p] * 6 + [C.c_size_t, C.c_size_t] + [C.c_int] * 6 + [C.c_void_p] * 3 + [C.c_int] * 6
    _cache[key] = lib
    return lib


class FxtIo(C.Structure):
    _fields_ = [("inp", C.c_void_p * 32), ("out", C.c_void_p * 32)]


class HostTranslated:
    def __init__(self, prog, n: int, channels: int = 1):
        fx = importlib.import_module(PKG)
        src, _ = fx.translate_source(prog, channels, instances=n)
        if src is None:
            raise ValueError("program is not eligible for translation")
        self.src = src
        self.span = None                    # delay lines: periods per emulated launch (the caller sets it from the ring geometry)
        self.lib = compile_source(src)
        self.n, self.c = n, channels
        regs = prog.registers()
        self.registers = np.repeat(np.array([r[1] for r in regs], dtype=np.float32)[:, None], n, axis=1).copy()
        self.acc = np.zeros(n, np.float64)
        self.lfsr = np.stack([np.full(n, SEED1, np.uint32), np.full(n, SEED2, np.uint32)])
        self.out_latch = np.zeros((channels, n), np.float32)
        self.tram_ptrs = np.zeros((4, n), np.int32)
        self.isz, self.xsz = prog.itram_size, prog.xtram_size
        self.itram = np.zeros((max(1, self.isz), n), np.float32)
        self.xtram = np.zeros((max(1, self.xsz), n), np.float32)
        self.counts = np.zeros(n, np.uint64)
        self.flags = np.zeros(1, np.uint32)
        self.tabs = device_tables(prog.tables())

    def process(self, x, inplace=False):
        """x: [C][S][N] float32 or (None, S) -> out [C][S][N].  With `inplace` the streaming kernel writes its outputs over its inputs
        (a copy of x: d_out == d_in)."""
        if isinstance(x, tuple):
            x, s = None, x[1]
        else:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1, self.n)
            s = x.shape[1]
        out = np.zeros((self.c, s, self.n), np.float32)
        cs = s * self.n
        if hasattr(self.lib, "fx_translated_sl_host"):
            if "#define FXT_NTR 0" in self.src:
                return self.process_blocks([x], s, inplace=inplace)[0]
            # a delay line: one emulated launch per stretch of at most `span` periods (what fx8010_gpu.cu::launch_blocks does)
            assert self.span and x is not None
            outs = []
            for a in range(0, s, self.span):
                k = min(self.span, s - a)
                outs.append(self.process_blocks([x[:, a:a + k]], k, seg_len=4, inplace=inplace)[0])
            return np.concatenate(outs, axis=1)
        import re
        lanes = int(re.search(r"#define FXT_K (\d+)", self.src).group(1))
        for i in range(-(-self.n // lanes) + 1):            # one thread past the end: the bounds check
            self.lib.fx_translated_host(i, self.registers.ctypes.data, self.acc.ctypes.data, self.lfsr.ctypes.data, self.out_latch.ctypes.data,
                                        self.tram_ptrs.ctypes.data, self.itram.ctypes.data, self.xtram.ctypes.data, self.counts.ctypes.data,
                                        self.flags.ctypes.data, self.tabs.ctypes.data, x.ctypes.data if x is not None else None, out.ctypes.data,
                                        cs, cs, s, self.n, self.isz, self.xsz)
        return out

    def tram(self, which: int, instance: int):
        return (self.itram if which == 0 else self.xtram)[: (self.isz if which == 0 else self.xsz), instance].copy()

    def process_blocks(self, xs, s, seg_len=8, inplace=False):
        """Stateless programs: consecutive blocks in ONE emulated launch (block x time segment x instance group work items).  With
        `inplace` every block's output buffer is its input buffer (a copy of xs[b], which stays as it was)."""
        assert self.n % 4 == 0
        nb = len(xs)
        xs = [None if x is None else np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, s, self.n) for x in xs]
        if inplace:
            assert all(x is not None for x in xs)
            outs = [x.copy() for x in xs]
        else:
            outs = [np.zeros((self.c, s, self.n), np.float32) for _ in xs]
        ins = outs if inplace else xs
        io = FxtIo()
        for b in range(nb):
            io.inp[b] = ins[b].ctypes.data if ins[b] is not None else None
            io.out[b] = outs[b].ctypes.data
        cs = s * self.n
        n_seg = -(-s // seg_len)
        order = [(tx, by) for by in range(n_seg * nb) for tx in range(self.n // 4 + 1)]     # one thread past the end: the bounds check
        base = [int(v) for v in self.tram_ptrs[:, 0]]      # what the host passes: the (shared) ring pointers at the launch's first period
        rng = np.random.default_rng(0)
        rng.shuffle(order)                                                                 # work items are independent: any order
        for tx, by in order:
            self.lib.fx_translated_sl_host(int(tx), int(by), io, self.registers.ctypes.data, self.acc.ctypes.data, self.out_latch.ctypes.data,
                                           self.counts.ctypes.data, self.flags.ctypes.data, self.tabs.ctypes.data, cs, cs, s, seg_len, n_seg, nb, self.n, 0,
                                           self.tram_ptrs.ctypes.data, self.itram.ctypes.data, self.xtram.ctypes.data, self.isz, self.xsz, *base)
        return outs
