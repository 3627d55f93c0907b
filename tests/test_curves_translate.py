"""Control curves in the translated kernels, checked on the CPU (no GPU needed).

fx8010_translate_source_curves emits the source fx8010_gpu_process_batch_curves compiles with NVRTC.  It is built here as plain C++
(-DFXT_HOST_CHECK) and driven over state arrays laid out like the device's, with the curves passed in the kernels' by-value parameter
block, against the oracle stepped one sample period at a time (set_register before each period): outputs, register file,
accumulator, LFSR, latches, TRAM pointers and contents, counters and runtime flags, bit for bit.  Both generators are covered — the
serial kernel (one thread per instance or group of lanes) and the streaming kernel (work items in random order, delay lines one emulated
launch per stretch of the ring's span).
"""
import ctypes as C
import importlib
import re

import numpy as np
import pytest

import curves_common as cc
import progs
from conftest import assert_bits_equal
from translate_host import FxtIo, compile_source, device_tables, SEED1, SEED2

fx = importlib.import_module("fx8010-emulator-core_b200")


class FxtCurves(C.Structure):
    _fields_ = [("p", C.c_void_p * 8), ("bcast", C.c_int * 8)]


@pytest.fixture(scope="module")
def po():
    from oracle import pyoracle
    return pyoracle


class HostCurves:
    """The automated translation of a program, run on the CPU like fx8010_gpu_process_batch_curves runs it on the device."""

    def __init__(self, prog, n, channels, regs, bcast):
        src, _ = fx.translate_source_curves(prog, list(zip(regs, bcast)), channels, instances=n)
        if src is None:
            raise ValueError("not eligible")
        self.src, self.n, self.c = src, n, channels
        self.regs, self.bcast = list(regs), list(bcast)
        self.lib = compile_source(src)
        self.serial = hasattr(self.lib, "fx_translated_host")
        if self.serial:
            self.lib.fx_translated_host.argtypes = [C.c_int] + [C.c_void_p] * 12 + [C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, FxtCurves]
        else:
            self.lib.fx_translated_sl_host.argtypes = ([C.c_int, C.c_int, FxtIo] + [C.c_void_p] * 6 + [C.c_size_t, C.c_size_t] + [C.c_int] * 6 +
                                                       [C.c_void_p] * 3 + [C.c_int] * 6 + [FxtCurves])
        self.registers = np.repeat(np.array([r[1] for r in prog.registers()], dtype=np.float32)[:, None], n, axis=1).copy()
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
        self.rng = np.random.default_rng(5)

    def kind(self):
        if self.serial:
            return 0
        return 1 if "#define FXT_NTR 0" in self.src else 2

    def _block(self, vals, s0):
        cb = FxtCurves()
        for j, v in enumerate(vals):
            cb.p[j] = v.ctypes.data + 4 * (s0 if self.bcast[j] else s0 * self.n)
            cb.bcast[j] = 1 if self.bcast[j] else 0
        return cb

    def process(self, x, vals, span=None, inplace=False):
        """x [C][S][N]; vals: per curve [S][N] (or [S] broadcast) float32 -> out [C][S][N].  With `inplace` the streaming kernel writes its
        outputs over its inputs (a copy of x: d_out == d_in)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        s = x.shape[1]
        if inplace:
            assert not self.serial
            out = x = x.copy()
        else:
            out = np.zeros((self.c, s, self.n), np.float32)
        cs = s * self.n
        if self.serial:
            lanes = int(re.search(r"#define FXT_K (\d+)", self.src).group(1))
            cb = self._block(vals, 0)
            for i in range(-(-self.n // lanes) + 1):            # one thread past the end: the bounds check
                self.lib.fx_translated_host(i, self.registers.ctypes.data, self.acc.ctypes.data, self.lfsr.ctypes.data, self.out_latch.ctypes.data,
                                            self.tram_ptrs.ctypes.data, self.itram.ctypes.data, self.xtram.ctypes.data, self.counts.ctypes.data,
                                            self.flags.ctypes.data, self.tabs.ctypes.data, x.ctypes.data, out.ctypes.data, cs, cs, s, self.n,
                                            self.isz, self.xsz, cb)
            return out
        span = span or s
        for a in range(0, s, span):                            # one emulated launch per stretch (kind 2; kind 1: the whole call)
            k = min(span, s - a)
            io = FxtIo()
            io.inp[0] = x.ctypes.data + 4 * a * self.n
            io.out[0] = out.ctypes.data + 4 * a * self.n
            seg_len = 4 if k > 4 else 8
            n_seg = -(-k // seg_len)
            base = [int(v) for v in self.tram_ptrs[:, 0]]
            order = [(tx, by) for by in range(n_seg) for tx in range(self.n // 4 + 1)]
            self.rng.shuffle(order)                            # work items are independent: any order
            cb = self._block(vals, a)
            for tx, by in order:
                self.lib.fx_translated_sl_host(int(tx), int(by), io, self.registers.ctypes.data, self.acc.ctypes.data, self.out_latch.ctypes.data,
                                               self.counts.ctypes.data, self.flags.ctypes.data, self.tabs.ctypes.data, cs, cs, k, seg_len, n_seg, 1,
                                               self.n, 0, self.tram_ptrs.ctypes.data, self.itram.ctypes.data, self.xtram.ctypes.data,
                                               self.isz, self.xsz, *base, cb)
        return out


def run_case(po, name, n, blocks, want_kind=None, span=None, seed=0, inplace=False):
    text, ch, cv = cc.programs()[name]
    prog = fx.Program(text, channels=ch)
    assert prog.loaded, prog.errors()
    regs = [prog.reg_index(r) for r, _ in cv]
    bcast = [b for _, b in cv]
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, n, ch)
    ht = HostCurves(prog, n, ch, regs, bcast)
    if want_kind is not None:
        assert ht.kind() == want_kind, (name, n, ht.kind())
    rng = np.random.default_rng(seed)
    for b, s in enumerate(blocks):
        x = (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)
        vals = [cc.make_curve(name, r, bc, s, n, rng) for r, bc in cv]
        got = ht.process(x, vals, span=span, inplace=inplace)
        want = cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s)
        assert_bits_equal(got, want, f"{name} outputs of block {b}")
    assert_bits_equal(ht.registers, orc.registers, name + " registers")
    assert_bits_equal(ht.acc, orc.acc, name + " accumulator")
    assert_bits_equal(ht.lfsr, orc.lfsr, name + " lfsr")
    assert_bits_equal(ht.out_latch, orc.out_latch, name + " latch")
    assert_bits_equal(ht.tram_ptrs, orc.tram_ptrs, name + " tram pointers")
    assert_bits_equal(ht.counts, orc.counts, name + " counters")
    if prog.itram_size:
        for i in sorted({0, n - 1}):
            assert_bits_equal(ht.itram[: prog.itram_size, i], orc.tram(0, i), f"{name} itram[{i}]")
    assert int(ht.flags[0]) == orc.flags, name + " runtime flags"
    return ht, prog, regs, bcast


# (program, instances, kind the automated translation must take)
CASES = [
    ("cfg2_instance", 12, 1), ("cfg2_instance", 7, 0), ("cfg2_broadcast", 12, 1), ("cfg2_broadcast", 5, 0),
    ("cfg4_cutoff", 6, 0), ("delay_fb", 8, 2), ("delay_fb", 6, 0), ("log_select", 8, 1), ("log_select", 3, 0),
    ("skip_data", 5, 0), ("cfg5", 3, 0), ("two_channels", 8, 0), ("delay_mod", 8, 0), ("delay_mod", 5, 0),
]


# ... and the cases on the streaming kernel once more with d_out == d_in
RUNS = ([pytest.param(name, n, kind, False, id=f"{name}-{n}-{kind}") for name, n, kind in CASES] +
        [pytest.param(name, n, kind, True, id=f"{name}-{n}-{kind}-inplace") for name, n, kind in CASES if kind != 0])


@pytest.mark.parametrize("name,n,kind,inplace", RUNS)
def test_curves_match_the_oracle_stepped_per_period(po, name, n, kind, inplace):
    span = 200 if name == "delay_fb" and kind == 2 else None
    blocks = [37, 9, 1] if name != "cfg5" else [9, 4]
    if name in ("delay_fb", "delay_mod"):
        blocks = [70, 333, 1, 250]
    run_case(po, name, n, blocks, want_kind=kind, span=span, seed=sum(map(ord, name)) + n, inplace=inplace)


def test_cfg4_four_instances_per_thread(po, monkeypatch):
    """The serial kernel with 4 lanes per thread: a per-instance curve is one more 16-byte ring row."""
    monkeypatch.setenv("FX8010_TR_K", "4")
    ht, *_ = run_case(po, "cfg4_cutoff", 8, [50, 33], want_kind=0)
    assert "#define FXT_K 4" in ht.src


def test_automated_delay_offsets_are_not_prefetched_streams():
    """A ring whose READ or WRITE offset follows a curve is read and written at its per-period slot, never through the serial kernel's
    prefetched TRAM stream (which fixes the slots at kernel start).  The plain translation of the same program does stream it."""
    text, ch, cv = cc.programs()["delay_mod"]
    prog = fx.Program(text)
    assert "tfast_i" in fx.translate_source(prog, instances=8)[0]
    for curves in ([("roff", False)], [("woff", True)], [("roff", False), ("woff", True)]):
        src, _ = fx.translate_source_curves(prog, [(prog.reg_index(r), b) for r, b in curves], instances=8)
        assert src is not None and "tfast_i" not in src, curves


def test_automated_skip_count_is_not_eligible():
    prog = fx.Program(cc.SKIP_COUNT)
    assert prog.loaded
    n = prog.reg_index("n")
    assert fx.translate_source(prog)[0] is not None                     # a constant count: translated
    assert fx.translate_source_curves(prog, [(n, True)])[0] is None       # automated: SKIP counts must be translation-time constants
    a = prog.reg_index("a")
    assert fx.translate_source_curves(prog, [(a, False)])[0] is not None  # another register automated: still eligible


def test_bad_curve_lists_are_rejected():
    prog = fx.Program(progs.CFG2_LOG_GAIN)
    vol, inp = prog.reg_index("volume"), prog.reg_index("in_l")
    assert fx.translate_source_curves(prog, [(vol, 0), (vol, 1)])[0] is None      # named twice
    assert fx.translate_source_curves(prog, [(inp, 0)])[0] is None                # an INPUT register
    assert fx.translate_source_curves(prog, [(999, 0)])[0] is None                # out of range
    assert fx.translate_source_curves(prog, [(vol, 0)] * 9)[0] is None            # more than 8


def test_no_curves_is_the_plain_source():
    for text in (progs.CFG2_LOG_GAIN, progs.CFG4_ONEPOLE, progs.cfg3_delay(200), cc.SKIP_DATA):
        prog = fx.Program(text)
        for n in (1, 8, 65536):
            assert fx.translate_source_curves(prog, [], instances=n)[0] == fx.translate_source(prog, instances=n)[0]


@pytest.mark.parametrize("name", sorted(cc.programs()))
def test_automated_sources_compile_for_sm_100a(name):
    text, ch, cv = cc.programs()[name]
    prog = fx.Program(text, channels=ch)
    curves = [(prog.reg_index(r), b) for r, b in cv]
    for n in (8, 6):
        src, cubin = fx.translate_source_curves(prog, curves, ch, compile_check=True, instances=n)
        assert src is not None and "FxtCurves" in src
        if cubin == -1:
            pytest.skip("libnvrtc not loadable here")
        assert cubin > 1000
