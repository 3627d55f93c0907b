"""tests/chain_host.py — TEST INFRASTRUCTURE: runs the fused kernel of a program chain (fx8010_translate_source_chain) on the CPU.

The generated chain source compiles as plain C++ with -DFXT_HOST_CHECK, like the single-program sources tests/translate_host.py runs.
HostChain compiles it with g++ and calls fx_translated_chain_host for every (thread, time segment) work item, in random order, over
per-stage state arrays laid out like the device's.  The product never uses this path.
"""
import ctypes as C
import hashlib
import importlib
import os
import subprocess
import tempfile

import numpy as np

from translate_host import PKG, device_tables

_cache = {}


class FxtStage(C.Structure):
    _fields_ = [("gpr", C.c_void_p), ("acc", C.c_void_p), ("latch", C.c_void_p), ("counts", C.c_void_p), ("rt_flags", C.c_void_p), ("tabs", C.c_void_p)]


class FxtChain(C.Structure):
    _fields_ = [("s", FxtStage * 8)]


def compile_chain_source(src: str) -> C.CDLL:
    key = hashlib.sha1(src.encode()).hexdigest()
    if key in _cache:
        return _cache[key]
    d = tempfile.mkdtemp(prefix="fxt_chain_")
    cu, so = os.path.join(d, "t.cpp"), os.path.join(d, "t.so")
    with open(cu, "w") as f:
        f.write(src)
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-DFXT_HOST_CHECK", "-o", so, cu], check=True)
    lib = C.CDLL(so)
    lib.fx_translated_chain_host.restype = None
    lib.fx_translated_chain_host.argtypes = [C.c_int, C.c_int, FxtChain, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int]
    _cache[key] = lib
    return lib


class StageState:
    """One stage's state arrays laid out like the device's (as a freshly loaded handle holds them)."""

    def __init__(self, prog, n: int, channels: int):
        self.registers = np.repeat(np.array([r[1] for r in prog.registers()], dtype=np.float32)[:, None], n, axis=1).copy()
        self.acc = np.zeros(n, np.float64)
        self.out_latch = np.zeros((channels, n), np.float32)
        self.counts = np.zeros(n, np.uint64)
        self.flags = np.zeros(1, np.uint32)
        self.tabs = device_tables(prog.tables())


class HostChain:
    """The fused kernel of a chain of stateless programs on the CPU: every (thread, time segment) work item in random order, over
    per-stage state arrays."""

    def __init__(self, progs, n: int, channels: int = 1):
        fx = importlib.import_module(PKG)
        src, _ = fx.translate_source_chain(progs, channels, instances=n)
        if src is None:
            raise ValueError("some stage is not stateless")
        self.src = src
        self.lib = compile_chain_source(src)
        self.n, self.c = n, channels
        self.stages = [StageState(p, n, channels) for p in progs]

    def process(self, x, s=None, seg_len=8, seed=0, inplace=False):
        """x: [C][S][N] float32 (or None with s) -> out [C][S][N].  With `inplace` the kernel writes its outputs over its inputs (a copy
        of x: d_out == d_in)."""
        assert self.n % 4 == 0
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1, self.n)
            s = x.shape[1]
        if inplace:
            out = x = x.copy()
        else:
            out = np.zeros((self.c, s, self.n), np.float32)
        ch = FxtChain()
        for j, st in enumerate(self.stages):
            ch.s[j] = FxtStage(st.registers.ctypes.data, st.acc.ctypes.data, st.out_latch.ctypes.data, st.counts.ctypes.data,
                               st.flags.ctypes.data, st.tabs.ctypes.data)
        cs = s * self.n
        n_seg = -(-s // seg_len)
        order = [(tx, by) for by in range(n_seg) for tx in range(self.n // 4 + 1)]     # one thread past the end: the bounds check
        np.random.default_rng(seed).shuffle(order)
        for tx, by in order:
            self.lib.fx_translated_chain_host(int(tx), int(by), ch, x.ctypes.data if x is not None else None, out.ctypes.data, cs, cs, s, seg_len, self.n)
        return out
