"""Operand edge values on every kernel (tests/edge_operands.py): each opcode at signed zeros, subnormals, the +-1 and int32-conversion
limits, the largest finite values, the infinities and a NaN, against the oracle.

The op programs take A, X and Y from three controls set per instance to the cross product of the 30 edge values (27 000 instances), and
A once more from an input that walks through the edge values period by period.  Every op's result of every period reaches an output
channel, so the kernels' per-period loops are checked, not only the copy that writes the final state.  Two variants of each:
  * hot: nobody reads `ccr`; in the instruction-major kernel the input form runs as a fused producer/consumer pair;
  * ccr: `limit q, 1, ccr, ccr` after each op, which materialises CCR every period (the kernels' CCR-live copies) and outputs it.
Floats are compared with NaN as a class (ledger U11), everything else bit for bit; every NaN the device stores must be 0x7FFFFFFF, or
0xFFC00000 where the oracle holds that pattern too (a NaN born in the FP64 pipe, edge_operands.assert_device_nan).  Every case asserts the
kernel that ran it (launch_info.kernel_variant).
"""
import importlib
import math

import numpy as np
import pytest

import curves_common as ccv
import edge_operands as eo
from chain_common import oracle_chain_stepped
from test_gpu_inplace import kernel_of
from test_gpu_parity import make_pair

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

fx = importlib.import_module("fx8010-emulator-core_b200")
from oracle import pyoracle as po  # noqa: E402

GA, GX, GY = eo.grid()
N = GA.size
GRID = {"ca": GA, "cx": GX, "cy": GY}
BLOCKS = (11, 21)                 # two calls: a ragged batch, then one that ends on a batch boundary of M = 8 minus 3
SAMPLED = (0, 1, 4095, N // 2, N - 1)

OP_GROUPS = [eo.OPS[0:4], eo.OPS[4:8], eo.OPS[8:12], eo.OPS[12:14]]     # a few output channels per program for the interpreters


class Snapshot:
    """The oracle's outputs per call and its final state, kept for the several kernels that run the same program."""

    def __init__(self, orc, outs, tram_instances):
        self.outs = outs
        self.registers, self.acc, self.lfsr = orc.registers.copy(), orc.acc.copy(), orc.lfsr.copy()
        self.out_latch, self.tram_ptrs, self.counts, self.flags = orc.out_latch.copy(), orc.tram_ptrs.copy(), orc.counts.copy(), orc.flags
        self.rings = {(w, i): orc.tram(w, i) for w in (0, 1) for i in tram_instances
                      if (orc.image.itram_size if w == 0 else orc.image.xtram_size)}

    def tram(self, which, i):
        return self.rings[(which, i)]


_expected = {}


def expected(text, ch, n, controls, blocks, key):
    if (text, key) not in _expected:
        prog = fx.Program(text, channels=ch)
        assert prog.loaded, prog.errors()
        img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
        orc = po.Oracle(img, n, ch)
        for nm, v in controls.items():
            orc.set_register(nm, v)
        outs, t0 = [], 0
        for s in blocks:
            outs.append(orc.process(eo.periodic_input(ch, s, n, t0), threads=8))
            t0 += s
        _expected[(text, key)] = Snapshot(orc, outs, [i for i in SAMPLED if i < n])
        prog.close()
    return _expected[(text, key)]


def check_variant(info, kernel, bits_set=0, bits_clear=0, lanes=None, what=""):
    kv = info.kernel_variant
    if kernel == "tr_serial":      # (kernel_of reads 4 instances per thread and TRAM as the time-cut kernel: one time segment tells them apart)
        assert kv & 128 and not kv & 4 and info.last_time_split == 1, f"{what}: expected {kernel}, kernel_variant {kv:#x}"
    else:
        assert kernel_of(kv) == kernel, f"{what}: expected {kernel}, kernel_variant {kv:#x}"
    assert kv & bits_set == bits_set and not kv & bits_clear, f"{what}: kernel_variant {kv:#x}, want bits {bits_set:#x} set, {bits_clear:#x} clear"
    if lanes is not None:
        assert (kv >> 8) & 0xff == lanes, f"{what}: kernel_variant {kv:#x}, want {lanes} instances per thread"


def run_gpu(text, ch, n, controls, blocks, key, kernel, monkeypatch, env=None, mode=0, bits_set=0, bits_clear=0, lanes=None,
            broadcast=(), what=""):
    """`text` on a fresh handle (environment applied first), block by block through process_host; outputs and the whole state
    against the oracle, the kernel of every call asserted."""
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    want = expected(text, ch, n, controls, blocks, key)
    prog = fx.Program(text, channels=ch)
    gpu = fx.Gpu(n, ch)
    try:
        gpu.load_program(prog)
        gpu.set_option(fx.OPT_TRANSLATE, mode)
        for nm, v in controls.items():
            if nm in broadcast:                     # one value for every instance: the host knows it (reg_uniform)
                gpu.set_controls(prog.reg_index(nm), v[:1], broadcast=True)
            else:
                gpu.set_controls(prog.reg_index(nm), v)
        t0 = 0
        for b, s in enumerate(blocks):
            y = gpu.process_host(eo.periodic_input(ch, s, n, t0))
            t0 += s
            check_variant(gpu.launch_info(), kernel, bits_set, bits_clear, lanes, f"{what} call {b} ({gpu.translate_status()['message']})")
            eo.assert_edge_equal(y, want.outs[b], f"{what} call {b} outputs")
            eo.assert_device_nan(y, want.outs[b], f"{what} call {b} outputs")
        eo.compare_state_edges(gpu, want, what, [i for i in SAMPLED if i < n])
        eo.assert_device_nan(gpu.registers(), want.registers, what + " registers")
        return gpu.launch_info().kernel_variant
    finally:
        gpu.close()
        prog.close()


# ---- the op programs on the interpreter kernels ------------------------------------------------------------------------------

# name: (environment, program extras, kernel, bits set, bits clear)
PRED_SKIP = dict(extra_head=["control csk = 0"], lead_body=["skip ccr, ccr, 8, csk"])      # a SKIP count the host cannot know: all predicated
INTERP = {
    "generic": ({"FX8010_NO_STATELESS": "1"}, {}, "generic", 0, 1 | 2),
    "generic_skip": ({"FX8010_NO_STATELESS": "1"}, dict(extra_body=["skip ccr, ccr, 8, 0"]), "generic", 1, 2),
    "generic_predicated": ({"FX8010_NO_STATELESS": "1"}, PRED_SKIP, "generic", 1, 2),
    "generic_ext": ({"FX8010_NO_STATELESS": "1"}, dict(extra_head=["static m"], extra_body=["macmv m, ca, cx, cy"]), "generic", 2, 1),
    "im": ({}, {}, "im", 0, 0),
    "im_M1": ({"FX8010_TUNE_M": "1"}, {}, "im", 0, 0),
    "im_no_pairs": ({"FX8010_NO_PAIRS": "1"}, {}, "im", 0, 64),
}


@pytest.mark.parametrize("variant", ["hot", "ccr"])
@pytest.mark.parametrize("name", sorted(INTERP))
def test_op_grid_interpreters(name, variant, monkeypatch):
    env, extra, kernel, bset, bclear = INTERP[name]
    for ops in OP_GROUPS:
        text, ch = eo.op_program(ops, ccr=variant == "ccr", **extra)
        controls = dict(GRID, csk=np.zeros(N, np.float32)) if "csk" in text else GRID
        pairs = 0
        if kernel == "im":
            pairs = 64 if variant == "hot" and name != "im_no_pairs" else 0
        with monkeypatch.context() as mp:
            run_gpu(text, ch, N, controls, BLOCKS, "grid", kernel, mp, env, bits_set=bset | pairs, bits_clear=bclear | (64 if not pairs else 0),
                    what=f"{name} {variant} {'/'.join(ops)}")


@pytest.mark.parametrize("op", eo.OPS)
def test_op_grid_short_kernel(op, monkeypatch):
    """Per-op programs of three instructions with a value carried from the last instruction to the second (the short-program kernel)."""
    text = "\n".join(["control ca = 0", "control cx = 0", "control cy = 0", "static w", "input in_l 0", "output o0 0", "output o1 1",
                      f"{op} o0, ca, cx, cy", f"{op} o1, in_l, cx, w", "limit w, o0, o0, o0", "end"])
    run_gpu(text, 2, N, GRID, BLOCKS, "grid", "short", monkeypatch, {"FX8010_NO_CARRY": "1"}, what=f"short {op}")


# ---- the op programs on the translated kernels (one program with every op; one NVRTC compile each) ----------------------------

@pytest.mark.parametrize("variant", ["hot", "ccr"])
def test_op_grid_translated_streaming(variant, monkeypatch):
    text, ch = eo.op_program(ccr=variant == "ccr")
    run_gpu(text, ch, N, GRID, BLOCKS, "grid", "tr_stream", monkeypatch, mode=2, lanes=4, what=f"translated streaming {variant}")


@pytest.mark.parametrize("lanes", [1, 4])
def test_op_grid_translated_serial(lanes, monkeypatch):
    """A MACMV makes the program stateful (the serial kernel); at one lane a literal SKIP as well (SKIP runs at one lane only), and the
    CCR variant."""
    extra = ["macmv m, ca, cx, cy"] + (["skip ccr, ccr, 8, 1", "macs m, m, in_l, 0.5"] if lanes == 1 else [])
    text, ch = eo.op_program(ccr=lanes == 1, extra_head=["static m"], extra_body=extra)
    run_gpu(text, ch, N, GRID, BLOCKS, "grid", "tr_serial", monkeypatch, {"FX8010_TR_K": str(lanes)}, mode=2, lanes=lanes,
            what=f"translated serial K={lanes}")


def test_op_grid_curve_kernel():
    """The streaming curve kernel: Y arrives as a per-instance control curve, a different edge value every period."""
    text, ch = eo.op_program()
    prog, img, orc, gpu = make_pair(fx, po, text, N, ch)
    try:
        gpu.set_option(fx.OPT_TRANSLATE, 2)
        for nm in ("ca", "cx"):
            gpu.set_controls(prog.reg_index(nm), GRID[nm]); orc.set_register(nm, GRID[nm])
        ry = prog.reg_index("cy")
        t0 = 0
        for b, s in enumerate(BLOCKS):
            x = eo.periodic_input(ch, s, N, t0)
            cv = eo.EDGE[(np.arange(N)[None, :] + np.arange(t0, t0 + s)[:, None]) % eo.E].astype(np.float32)
            t0 += s
            want = ccv.oracle_stepped(orc, x, [(ry, cv, False)], s)
            d_in, d_cv = torch.from_numpy(x).cuda(), torch.from_numpy(np.ascontiguousarray(cv)).cuda()
            d_out = torch.empty_like(d_in)
            gpu.process_device_curves(d_in, d_out, s, [(ry, d_cv, False)])
            gpu.synchronize()
            check_variant(gpu.launch_info(), "tr_stream", fx.VARIANT_CURVES, 0, 4, f"curves call {b} ({gpu.translate_status_curves()})")
            y = d_out.cpu().numpy()
            eo.assert_edge_equal(y, want, f"curves call {b} outputs")
            eo.assert_device_nan(y, want, f"curves call {b} outputs")
        eo.compare_state_edges(gpu, orc, "curves", SAMPLED)
    finally:
        gpu.close()
        prog.close()


def test_op_grid_fused_chain():
    """The hot op program as the middle stage of a three-stage chain fused into one kernel, against the stages' oracles stepped per
    period.  The outer stages pass every channel through unchanged (`limit o, i, i, i`)."""
    hot, ch = eo.op_program()
    through = "\n".join([f"input i{c} {c}" for c in range(ch)] + [f"output o{c} {c}" for c in range(ch)] +
                        [f"limit o{c}, i{c}, i{c}, i{c}" for c in range(ch)] + ["end"])
    stages = [make_pair(fx, po, t, N, ch) for t in (through, hot, through)]
    chain = None
    try:
        for prog, _, orc, gpu in stages:
            gpu.set_option(fx.OPT_TRANSLATE, 2)
        prog, _, orc, gpu = stages[1]
        for nm, v in GRID.items():
            gpu.set_controls(prog.reg_index(nm), v); orc.set_register(nm, v)
        chain = fx.Chain([st[3] for st in stages])
        t0 = 0
        for b, s in enumerate(BLOCKS):
            x = eo.periodic_input(ch, s, N, t0)
            t0 += s
            want = oracle_chain_stepped([st[2] for st in stages], x, s)
            d_in = torch.from_numpy(x).cuda()
            d_out = torch.empty_like(d_in)
            chain.process_batch(d_in, d_out, s)
            torch.cuda.synchronize()
            st = chain.status()
            assert st["fused_last"] == 1, st
            y = d_out.cpu().numpy()
            eo.assert_edge_equal(y, want, f"chain call {b} outputs")
            eo.assert_device_nan(y, want, f"chain call {b} outputs")
        for k, (_, _, orc, gpu) in enumerate(stages):
            eo.compare_state_edges(gpu, orc, f"chain stage {k}", SAMPLED)
    finally:
        if chain is not None:
            chain.close()
        for prog, _, _, gpu in stages:
            gpu.close()
            prog.close()


# ---- MACMV, SKIP and TRAM offsets from the grid -------------------------------------------------------------------------------

MACMV_PROG = "\n".join(["control ca = 0", "control cx = 0", "control cy = 0", "input in_l 0"] + [f"output o{c} {c}" for c in range(3)] +
                       ["macmv o0, ca, cx, cy", "macmv o1, in_l, cy, cx", "acc3 o2, ca, cx, cy", "macmv o2, o2, cy, cy", "end"])
SKIP_PROG = "\n".join(["control ca = 0", "control cx = 0", "control cy = 0", "input in_l 0"] + [f"output o{c} {c}" for c in range(3)] +
                      ["macs o0, ca, 0, 0", "skip ccr, ccr, cx, cy", "macs o1, in_l, ca, 0.5", "macintw o2, o2, ca, 0.75",
                       "limit o0, 1, ccr, ccr", "end"])
TRAM_PROG = "\n".join(["control ca = 0", "control cx = 0", "control cy = 0", "static rd", "static rx", "input in_l 0", "output o0 0",
                       "output o1 1", "itramsize 40 ", "xtramsize 72 ", "idelay write, in_l, at, cy", "idelay read, rd, at, cx",
                       "xdelay read, rx, at, ca", "xdelay write, in_l, at, cx", "limit o0, rd, rd, rd", "limit o1, rx, rx, rx", "end"])


@pytest.mark.parametrize("kernel", ["generic", "tr_serial"])
def test_macmv_grid(kernel, monkeypatch):
    """MACMV carries the accumulator across periods (operands from the grid)."""
    mode = 2 if kernel == "tr_serial" else 0
    run_gpu(MACMV_PROG, 3, N, GRID, (40, 9), "grid", kernel, monkeypatch, mode=mode, bits_set=2, what=f"macmv on {kernel}")


@pytest.mark.parametrize("mode", [0, 2])
def test_skip_grid(mode, monkeypatch):
    """SKIP compares with X and skips Y instructions, both from the grid (counts past END repeat the period up to the pass cap).  In
    translation mode 2 as well: the translator declines a SKIP count it cannot know, and the interpreter runs the program."""
    run_gpu(SKIP_PROG, 3, N, GRID, (40, 9), "grid", "generic", monkeypatch, mode=mode, bits_set=1, what=f"skip, translation mode {mode}")


@pytest.mark.parametrize("kernel", ["generic", "im"])
def test_tram_offsets_grid(kernel, monkeypatch):
    """IDELAY / XDELAY READ and WRITE offsets from the grid (clamped to the ring after the x86 conversion), over several ring turns;
    the instruction-major kernel's TRAM variant."""
    env = {"FX8010_NO_STATELESS": "1"} if kernel == "generic" else {}
    run_gpu(TRAM_PROG, 2, N, GRID, (90, 77), "grid", kernel, monkeypatch, env, bits_set=2, what=f"tram offsets on {kernel}")


# ---- folded literals ----------------------------------------------------------------------------------------------------------

FA, FX = (v.ravel().copy() for v in np.meshgrid(eo.EDGE, eo.EDGE, indexing="ij"))
FOLD_BLOCKS = (5, 3)


@pytest.mark.parametrize("pos", [0, 1, 2], ids=["A", "X", "Y"])
@pytest.mark.parametrize("kernel", ["tr_stream", "tr_serial", "im", "generic"])
def test_folded_literals(kernel, pos, monkeypatch):
    """Each op with one operand a literal at every edge spelling (an immediate of the translated kernels, NVRTC may fold the whole
    instruction), the other two from a 30 x 30 per-instance grid; results in static registers, compared in the final state."""
    text = eo.folded_program(eo.OPS, pos)
    env, mode, lanes = {}, 0, None
    if kernel == "tr_serial":
        text = text.replace("\nend", "\nstatic m\nmacmv m, ca, cx, cx\nend")
        env, mode, lanes = {"FX8010_TR_K": "1"}, 2, 1
    elif kernel == "tr_stream":
        mode, lanes = 2, 4
    elif kernel == "generic":
        env = {"FX8010_NO_STATELESS": "1"}
    controls = {"ca": FA, "cx": FX}
    run_gpu(text, 1, FA.size, controls, FOLD_BLOCKS, "fold", kernel, monkeypatch, env, mode=mode, lanes=lanes, what=f"folded literals at {'AXY'[pos]} on {kernel}")


# ---- broadcast controls: values the host analyses read ------------------------------------------------------------------------

def cvt_x86(v):
    v = float(v)
    return -2**31 if (math.isnan(v) or v >= 2**31 or v < -2**31) else int(v)


NAN = float(eo.EDGE[-1])             # 0x7FFFFFFF (numpy's float("nan") is 0x7FC00000)
SELECTORS = [NAN, float("-inf"), -1.0, -0.0, 31.0, float(np.float32(31.999998)), 32.0, 2.0**31]
SEL_PROG = "\n".join(["control sel = 3", "input in_l 0", "output o0 0", "output o1 1", "output o2 2", "log o0, in_l, sel, 0",
                      "exp o1, in_l, sel, 1", "log o2, in_l, sel, in_l", "end"])


@pytest.mark.parametrize("kernel", ["im", "generic"])
def test_broadcast_table_selector(kernel, monkeypatch):
    """A LOG / EXP selector set with broadcast: the host places the tables from its value (out of range: clamped, flag set)."""
    env = {"FX8010_NO_STATELESS": "1", "FX8010_NO_SHORT": "1"} if kernel == "generic" else {}
    n = 240
    for v in SELECTORS:
        with monkeypatch.context() as mp:
            run_gpu(SEL_PROG, 3, n, {"sel": np.full(n, v, np.float32)}, (20, 9), f"sel {v!r}", kernel, mp, env, broadcast=("sel",),
                    what=f"selector {v!r} on {kernel}")


SKIP_COUNTS = [NAN, -0.0, -1.0, 1.5, 2.0**31, -2.0**31]
SKIPC_PROG = "\n".join(["control cnt = 0", "input in_l 0", "output o0 0", "output o1 1", "macs o0, in_l, 0, 0", "skip ccr, ccr, ccr, cnt",
                        "macsn o1, in_l, 0.5, 0.5", "limit o0, 1, ccr, ccr", "macs o1, o1, 0.25, 1", "end"])


@pytest.mark.parametrize("mode", [0, 2])
def test_broadcast_skip_count(mode, monkeypatch):
    """A SKIP count set with broadcast: the host's reach analysis reads it through the x86 conversion (NaN and +-2^31 skip one)."""
    n = 240
    for v in SKIP_COUNTS:
        with monkeypatch.context() as mp:
            run_gpu(SKIPC_PROG, 2, n, {"cnt": np.full(n, v, np.float32)}, (20, 9), f"cnt {v!r}", "generic", mp, mode=mode, bits_set=1,
                    broadcast=("cnt",), what=f"skip count {v!r}, translation mode {mode}")


RING = 200
OFFSETS = [NAN, float("inf"), float("-inf"), -1.0, -0.0, RING - 1.0, float(RING), 2.0**31]
OFF_PROG = "\n".join(["static a", "static rd", "control roff = 0", "control woff = 0", "input in_l 0", "output out_l 0", f"itramsize {RING} ",
                      "idelay read, rd, at, roff", "macs a, in_l, rd, 0.5", "idelay write, a, at, woff", "macs out_l, in_l, rd, 0.5", "end"])


def cut_span(roff, woff):
    """The span of independent periods the host derives for OFF_PROG (read before write), None when too short to cut along time."""
    pos, wpos = (min(max(cvt_x86(v), 0), RING - 1) for v in (roff, woff))
    d = (wpos + pos) % RING
    d = RING if d == 0 else d
    span = min(RING, d, RING - d if d < RING else RING)
    return span if span >= 64 else None


@pytest.mark.parametrize("kernel", ["interp", "tr_cut"])
def test_broadcast_tram_offsets(kernel, monkeypatch):
    """TRAM READ / WRITE offsets set with broadcast: the host derives the ring distance and the time-cut span from them."""
    n = 256
    for which in ("roff", "woff"):
        for v in OFFSETS:
            ctl = {"roff": np.full(n, v if which == "roff" else 100.0, np.float32), "woff": np.full(n, v if which == "woff" else 0.0, np.float32)}
            span = cut_span(ctl["roff"][0], ctl["woff"][0])
            if kernel == "interp":
                want, env, mode = "im", {"FX8010_NO_TSPLIT": "1"}, 0
            else:
                want, env, mode = ("tr_cut" if span else "im"), {}, 2
            with monkeypatch.context() as mp:
                run_gpu(OFF_PROG, 1, n, ctl, (300, 1, 150), f"{which} {v!r}", want, mp, env, mode=mode, broadcast=("roff", "woff"),
                        what=f"{which} = {v!r} on {kernel} (span {span})")


def test_signed_zeros_per_instance(monkeypatch):
    """One per-instance array that mixes +0 and -0, as the X and Y of every op (instruction-major and translated streaming)."""
    n = 4096
    z = np.where(np.arange(n) % 3 == 1, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
    ctl = {"ca": np.roll(z, 1), "cx": z, "cy": np.roll(z, 2)}
    text, ch = eo.op_program()
    for kernel, mode in (("im", 0), ("tr_stream", 2)):
        with monkeypatch.context() as mp:
            run_gpu(text, ch, n, ctl, BLOCKS, "zeros", kernel, mp, mode=mode, what=f"signed zeros on {kernel}")
