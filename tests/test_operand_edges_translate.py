"""The translator's generated source at operand edge values, run on the CPU (-DFXT_HOST_CHECK, tests/translate_host.py) against the oracle.

Every opcode sees signed zeros, subnormals, the +-1 and int32-conversion limits, the largest finite values, the infinities and a NaN
(tests/edge_operands.py) as per-instance controls over their cross product, as inputs that change every period, and as literals the
translation folds into immediates, in each operand position.  Outputs and the whole final state are compared with NaN as a class and
everything else bit for bit.  The same values on the device: tests/test_gpu_operand_edges.py."""
import importlib

import numpy as np
import pytest

import edge_operands as eo
from translate_host import HostTranslated

fx = importlib.import_module("fx8010-emulator-core_b200")


def oracle_of(prog, n, channels):
    from oracle import pyoracle as po
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    return po.Oracle(img, n, channels)


def run_both(text, n, channels, controls, x, kernel):
    """One block through the generated source and the oracle; compares outputs and state.  `kernel`: "sl" (streaming) or "serial"."""
    prog = fx.Program(text, channels=channels)
    assert prog.loaded, prog.errors()
    orc = oracle_of(prog, n, channels)
    ht = HostTranslated(prog, n, channels)
    assert ("fx_translated_sl" in ht.src) == (kernel == "sl"), "the program took the other translated kernel"
    for name, v in controls.items():
        r = prog.reg_index(name)
        assert r >= 0, name
        orc.set_register(r, v)
        ht.registers[r, :] = v
    yo = orc.process(x, threads=8)
    yh = ht.process(x)
    eo.assert_edge_equal(yh, yo, "outputs")
    eo.assert_edge_equal(ht.registers, orc.registers, "registers")
    eo.assert_edge_equal(ht.acc, orc.acc, "accumulator")
    eo.assert_edge_equal(ht.out_latch, orc.out_latch, "output latch")
    eo.assert_edge_equal(ht.lfsr, orc.lfsr, "lfsr")
    eo.assert_edge_equal(ht.counts, orc.counts, "instruction counters")
    assert int(ht.flags[0]) == orc.flags, (int(ht.flags[0]), orc.flags)
    return prog, ht


def test_literal_spellings_read_as_their_bits():
    """Every spelling reaches the register file as exactly its edge value (strtof of a long decimal)."""
    sp = eo.LITERAL_SPELLING
    text = "\n".join(["output o 0"] + [f"macs o, {s}, 0, 0" for s in sp.values()] + ["end"])
    prog = fx.Program(text)
    assert prog.loaded, prog.errors()
    values = {name: v for _, v, _, name in prog.registers()}
    for b, s in sp.items():
        assert s in values, s
        got = int(np.float32(values[s]).view(np.uint32))
        assert got == b, f"{s!r} reads as {got:#010x}, not {b:#010x}"
    assert set(sp) == set(eo.EDGE_BITS) - {0x7fffffff}


def test_per_instance_grid_streaming():
    """The stateless op program (hot and CCR variants) on the streaming source: 27 000 instances, A / X / Y from the grid."""
    a, x, y = eo.grid()
    n = a.size
    for ccr in (False, True):
        text, ch = eo.op_program(ccr=ccr)
        run_both(text, n, ch, {"ca": a, "cx": x, "cy": y}, eo.periodic_input(ch, 8, n), "sl")


@pytest.mark.parametrize("lanes", [1, 4])
def test_per_instance_grid_serial(lanes, monkeypatch):
    """The op program with a MACMV (and, at one lane, a literal SKIP; the serial kernel takes a SKIP at one lane only) on the serial
    source.  The MACMV makes the program stateful."""
    monkeypatch.setenv("FX8010_TR_K", str(lanes))
    a, x, y = eo.grid()
    n = a.size
    extra = ["macmv m, ca, cx, cy"]
    if lanes == 1:
        extra += ["skip ccr, ccr, 8, 1", "macs m, m, in_l, 0.5"]
    text, ch = eo.op_program(ccr=(lanes == 1), extra_head=["static m"], extra_body=extra)
    _, ht = run_both(text, n, ch, {"ca": a, "cx": x, "cy": y}, eo.periodic_input(ch, 6, n), "serial")
    assert f"#define FXT_K {lanes}\n" in ht.src


@pytest.mark.parametrize("pos", [0, 1, 2], ids=["A", "X", "Y"])
def test_folded_literals(pos):
    """Each op with one operand a folded literal at every spelling; the other two from a 30 x 30 per-instance grid."""
    a, x = (v.ravel().copy() for v in np.meshgrid(eo.EDGE, eo.EDGE, indexing="ij"))
    text = eo.folded_program(eo.OPS, pos)
    prog, ht = run_both(text, a.size, 1, {"ca": a, "cx": x}, eo.periodic_input(1, 4, a.size), "sl")
    for b in (0x80000000, 0x4f000000, 0xcf000001, 0x7f800000, 0x00000001):       # the edge literals really are immediates
        assert f"__uint_as_float(0x{b:08x}u)" in ht.src, hex(b)


def test_all_literal_instructions():
    """About a hundred instructions with three literal operands: the translation folds them to constants."""
    text = eo.all_literal_program(np.random.default_rng(0x8010), 112)
    run_both(text, 8, 1, {}, eo.periodic_input(1, 3, 8), "sl")
