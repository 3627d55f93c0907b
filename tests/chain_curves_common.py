"""Shared by tests/test_chain_curves_translate.py, tests/test_gpu_chain_curves.py and tests/chain_curves_bench.py: control curves on program
chains (fx8010_chain_process_batch_curves).  The curve mixes the tests run, curve values, the reference for a chain call with curves — the
stages' oracles stepped one sample period at a time, with every curve value of a stage set right before that stage's period — and
HostChainCurves, which runs the generated curve-chain source on the CPU like tests/chain_host.py's HostChain."""
from __future__ import annotations

import ctypes as C
import importlib

import numpy as np

from chain_host import FxtChain, FxtStage, HostChain, StageState, compile_chain_source
from translate_host import PKG

# a gain stage whose gain is a STATIC the plain chain source folds into an immediate
MIDDLE = "\n".join(["static k = 0.75", "input in_l 0", "output out_l 0", "macs out_l, 0, in_l, k", "end"])

REG_STATIC, REG_CONTROL = 0, 2


def written(prog) -> set:
    """Registers some instruction of `prog` writes (its R operand)."""
    return {ins[1] for ins in prog.instructions() if ins[0] != 0x12}


def automatable(prog, kind: str) -> list:
    """Register indices of `prog` a curve may drive: kind "control" (CONTROL registers), "static_ro" (STATICs no instruction writes),
    "written" (STATICs some instruction writes)."""
    w = written(prog)
    out = []
    for i, (t, _, _, name) in enumerate(prog.registers()):
        if name == "noise":
            continue
        if kind == "control" and t == REG_CONTROL:
            out.append(i)
        elif kind == "static_ro" and t == REG_STATIC and i not in w:
            out.append(i)
        elif kind == "written" and t == REG_STATIC and i in w:
            out.append(i)
    return out


def any_reg(prog) -> list:
    return automatable(prog, "control") + automatable(prog, "static_ro") + automatable(prog, "written")


def curve_mix(progs, mix: str) -> list:
    """The curve list of mix `mix` over the stages `progs`: [(stage, register index, broadcast)]."""
    k = len(progs)
    mid = k // 2
    if mix == "first":
        return [(0, any_reg(progs[0])[0], False)]
    if mix == "middle":
        return [(mid, any_reg(progs[mid])[0], False)]
    if mix == "last":
        return [(k - 1, any_reg(progs[k - 1])[0], True)]
    if mix == "several":
        out = [(0, any_reg(progs[0])[0], False), (k - 1, any_reg(progs[k - 1])[-1], True)]
        if 0 < mid < k - 1:
            out.append((mid, any_reg(progs[mid])[0], False))
        return out
    if mix == "written":
        for j, p in enumerate(progs):
            w = automatable(p, "written")
            if w:
                return [(j, w[0], False), (k - 1, any_reg(progs[k - 1])[0], False)]
        raise ValueError("no stage writes a STATIC")
    if mix == "eight":                                 # 8 curves, round robin over the stages, broadcast every third
        cand = [[(j, r) for r in any_reg(p)] for j, p in enumerate(progs)]
        out = []
        while len(out) < 8:
            for c in cand:
                if c and len(out) < 8:
                    j, r = c.pop(0)
                    out.append((j, r, len(out) % 3 == 2))
            assert any(cand) or len(out) == 8, "fewer than 8 automatable registers"
        return out
    raise KeyError(mix)


MIXES = ["first", "middle", "last", "several", "eight", "written"]


def curve_values(curves, s: int, n: int, rng: np.random.Generator) -> list:
    """Values for each curve: per-instance [S][N] in [0.05, 1), broadcast [S] a ramp from 1 down to 0.25."""
    out = []
    for _, _, bc in curves:
        if bc:
            out.append(np.linspace(1.0, 0.25, s, dtype=np.float32))
        else:
            out.append((0.05 + 0.95 * rng.random((s, n))).astype(np.float32))
    return out


def oracle_chain_curves_stepped(orcs, x, s: int, curves, values, n: int):
    """The stages' oracles one sample period at a time, stage after stage; before stage j's period k every curve of stage j sets its
    register to its value of period k.  x [C][S][N] or None.  Returns [C][S][N]."""
    outs = []
    for k in range(s):
        y = None if x is None else np.ascontiguousarray(x[:, k:k + 1, :])
        for j, orc in enumerate(orcs):
            for (st, reg, bc), v in zip(curves, values):
                if st == j:
                    orc.set_register(reg, np.full(n, v[k], np.float32) if bc else np.ascontiguousarray(v[k]))
            y = orc.process(y, 1)
        outs.append(y)
    return np.concatenate(outs, axis=1)


class FxtCurves(C.Structure):
    _fields_ = [("p", C.c_void_p * 8), ("bcast", C.c_int * 8)]


class HostChainCurves(HostChain):
    """HostChain for the curve-chain kernel: the source of fx8010_translate_source_chain_curves, whose fx_translated_chain_host takes the
    curves by value after the chain's parameters."""

    def __init__(self, progs, n: int, channels: int, curves):
        fx = importlib.import_module(PKG)
        src, _ = fx.translate_source_chain_curves(progs, curves, channels, instances=n)
        if src is None:
            raise ValueError("some stage is not stateless")
        self.src = src
        self.lib = compile_chain_source(src)
        self.lib.fx_translated_chain_host.argtypes = list(self.lib.fx_translated_chain_host.argtypes[:10]) + [FxtCurves]
        self.n, self.c = n, channels
        self.curves = list(curves)
        self.stages = [StageState(p, n, channels) for p in progs]

    def process_curves(self, x, values, s=None, seg_len=8, seed=0, inplace=False):
        """x [C][S][N] (or None with s), values: one array per curve (curve_values) -> out [C][S][N]."""
        assert self.n % 4 == 0
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1, self.n)
            s = x.shape[1]
        out = x.copy() if inplace else np.zeros((self.c, s, self.n), np.float32)
        if inplace:
            x = out
        ch = FxtChain()
        for j, st in enumerate(self.stages):
            ch.s[j] = FxtStage(st.registers.ctypes.data, st.acc.ctypes.data, st.out_latch.ctypes.data, st.counts.ctypes.data,
                               st.flags.ctypes.data, st.tabs.ctypes.data)
        keep = [np.ascontiguousarray(v, dtype=np.float32) for v in values]
        cv = FxtCurves()
        for q, ((_, _, bc), v) in enumerate(zip(self.curves, keep)):
            cv.p[q], cv.bcast[q] = v.ctypes.data, 1 if bc else 0
        cs = s * self.n
        n_seg = -(-s // seg_len)
        order = [(tx, by) for by in range(n_seg) for tx in range(self.n // 4 + 1)]     # one thread past the end: the bounds check
        np.random.default_rng(seed).shuffle(order)
        for tx, by in order:
            self.lib.fx_translated_chain_host(int(tx), int(by), ch, x.ctypes.data if x is not None else None, out.ctypes.data, cs, cs, s,
                                              seg_len, self.n, cv)
        return out
