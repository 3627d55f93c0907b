"""The program translator's code generator, checked on the CPU (no GPU needed).

fx8010_translate_source emits the CUDA source the GPU path compiles with NVRTC; the same source builds as plain
C++ (-DFXT_HOST_CHECK) and is run here against the oracle, bit for bit: outputs, register file, accumulator, LFSR,
latches, TRAM pointers and contents, executed-instruction counters, runtime flags.  A second set of tests runs NVRTC
itself (it needs no device) to make sure the source compiles for sm_100a.
"""
import importlib

import numpy as np
import pytest

import progs
from conftest import assert_bits_equal
from translate_host import HostTranslated

fx = importlib.import_module("fx8010-emulator-core_b200")


@pytest.fixture(scope="module")
def po():
    from oracle import pyoracle
    return pyoracle


def check(po, text, n, blocks, rng, channels=1, controls=None, amp=0.9, what="case", span=None, inplace=False):
    prog = fx.Program(text, channels=channels)
    assert prog.loaded, prog.errors()
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, n, channels)
    ht = HostTranslated(prog, n, channels)
    ht.span = span
    for name, vals in (controls or {}).items():
        idx = prog.reg_index(name)
        orc.set_register(idx, vals)
        ht.registers[idx, :] = np.asarray(vals, dtype=np.float32)
    start = 0
    for s in blocks:
        x = (2 * amp * rng.random((channels, s, n)) - amp).astype(np.float32)
        assert_bits_equal(ht.process(x, inplace=inplace), orc.process(x), f"{what} outputs of block at {start}")
        start += s
    assert_bits_equal(ht.registers, orc.registers, what + " registers")
    assert_bits_equal(ht.acc, orc.acc, what + " accumulator")
    assert_bits_equal(ht.lfsr, orc.lfsr, what + " lfsr")
    assert_bits_equal(ht.out_latch, orc.out_latch, what + " latch")
    assert_bits_equal(ht.tram_ptrs, orc.tram_ptrs, what + " tram pointers")
    assert_bits_equal(ht.counts, orc.counts, what + " counters")
    for which, size in ((0, prog.itram_size), (1, prog.xtram_size)):
        if size:
            for i in sorted({0, n - 1}):
                if orc.tram(which, i).size:          # (a declared size without any TRAM instruction allocates nothing)
                    assert_bits_equal(ht.tram(which, i), orc.tram(which, i), f"{what} tram{which}[{i}]")
    assert int(ht.flags[0]) == orc.flags, what + " runtime flags"
    return ht


@pytest.mark.parametrize("seed", range(8))
def test_random_programs(po, seed):
    rng = np.random.default_rng(1000 + seed)
    text = progs.random_program(rng, 40 + 7 * seed, channels=1 + seed % 2, xtram=bool(seed % 3 == 0))
    check(po, text, 5, [23, 9], rng, channels=1 + seed % 2, what=f"random {seed}")


@pytest.mark.parametrize("seed", range(6))
def test_random_programs_four_instances_per_thread(po, seed, monkeypatch):
    """SKIP-free programs, several instances per thread in the serial kernel (the default above ~38 000 instances is 2; FX8010_TR_K forces it)."""
    monkeypatch.setenv("FX8010_TR_K", "4" if seed % 3 else "2")
    rng = np.random.default_rng(1500 + seed)
    ch = 1 + seed % 2
    text = progs.random_program(rng, 30 + 5 * seed, channels=ch, skip=False, xtram=bool(seed % 2))
    ht = check(po, text, 8, [19, 6, 1], rng, channels=ch, what=f"random K=4 {seed}")
    assert ("#define FXT_K 4" in ht.src or "#define FXT_K 2" in ht.src) and "fx_translated_host" in ht.src


def test_cfg4_onepole_four_instances_per_thread(po, monkeypatch):
    monkeypatch.setenv("FX8010_TR_K", "4")
    rng = np.random.default_rng(17)
    n = 8
    ctl = {"filter_cutoff": (0.001 + 0.998 * np.arange(n) / (n - 1)).astype(np.float32)}
    ht = check(po, progs.CFG4_ONEPOLE, n, [50, 33], rng, controls=ctl, what="cfg4")
    assert "#define FXT_K 4" in ht.src


@pytest.mark.parametrize("seed", range(4))
def test_random_programs_unsafe(po, seed):
    rng = np.random.default_rng(2000 + seed)
    text = progs.random_program(rng, 60, safe=False, wild_tables=True)
    check(po, text, 4, [17], rng, what=f"unsafe {seed}")


def test_cfg5_allops(po):
    rng = np.random.default_rng(progs.SEED)
    n = 6
    ctl = {f"k{i}": rng.random(n).astype(np.float32) for i in range(4)}
    ht = check(po, progs.cfg5_allops(), n, [12, 5], rng, controls=ctl, what="cfg5")
    assert "goto L" in ht.src or "bool sk" in ht.src


def test_skip_past_the_end_and_negative_count(po):
    rng = np.random.default_rng(5)
    text = "\n".join(["static a = 0.25", "static b", "input in_l 0", "output out_l 0",
                      "macs a, in_l, 0.5, 0.5", "skip ccr, ccr, 2, -3", "macs b, a, 0.5, 0.5", "macs out_l, b, a, 1.0",
                      "skip ccr, ccr, 2, 7", "macs b, b, 0.25, 0.25", "end"])
    # the second SKIP would jump past END: END is then not guaranteed, so the translator must decline
    prog = fx.Program(text)
    assert prog.loaded
    src, _ = fx.translate_source(prog)
    assert src is None
    text2 = text.replace("skip ccr, ccr, 2, 7", "skip ccr, ccr, 2, 1")
    check(po, text2, 8, [31], rng, what="negative skip count")


def test_skip_count_from_a_written_register_is_declined():
    text = "\n".join(["static n = 1", "static a", "input in_l 0", "output out_l 0", "macs n, 0, 1, 1", "skip ccr, ccr, 2, n",
                      "macs a, in_l, 0.5, 0.5", "macs out_l, a, 0, 0", "end"])
    prog = fx.Program(text)
    assert prog.loaded
    assert fx.translate_source(prog)[0] is None


def test_two_channels_input_index_quirk(po):
    rng = np.random.default_rng(9)
    text = "\n".join(["input in_l 0", "input in_r 1", "output out_l 0", "output out_r 1", "static t",
                      "macs t, in_l, in_r, 0.5", "skip ccr, ccr, 6, 1", "macs out_l, t, in_r, 0.25", "macs out_r, in_r, in_l, 0.5", "end"])
    check(po, text, 4, [19], rng, channels=2, what="two channels")


def test_noise_macmv_tram(po):
    rng = np.random.default_rng(11)
    text = "\n".join(["static noise", "static a", "static d", "static m", "input in_l 0", "output out_l 0", "itramsize 37 ", "xtramsize 50 ",
                      "macs a, in_l, noise, 0.125", "macmv m, a, in_l, 0.5", "macmv m, m, a, 0.25", "macs a, a, 0, 0",
                      "idelay write, a, at, 0", "idelay read, d, at, 36", "xdelay write, d, at, 3", "xdelay read, m, at, 40",
                      "skip ccr, ccr, 2, 1", "macs d, d, m, 0.5", "macs out_l, d, a, 0.5", "end"])
    check(po, text, 3, [90, 45], rng, what="noise/macmv/tram")


def with_inplace(names):
    """Each case on separate buffers (the case's name) and with d_out == d_in (name-inplace)."""
    return [pytest.param(nm, False, id=nm) for nm in names] + [pytest.param(nm, True, id=nm + "-inplace") for nm in names]


@pytest.mark.parametrize("name,inplace", with_inplace(["cfg1", "cfg2", "logtube", "random_stateless"]))
def test_stateless_programs_streaming_kernel(po, name, inplace):
    """Stateless programs translate into the streaming kernel (fx_translated_sl): blocks x time segments x instance groups.  In place,
    the owner of the last period must re-run it from its input, not from the output it has just stored there."""
    rng = np.random.default_rng(21)
    n = 12
    if name == "random_stateless":
        text = progs.random_program(rng, 24, skip=False, tram=False, noise=False, ops=progs.SAT_OPS + progs.TABLE_OPS + ["limit", "tstneg", "andxor"])
        text = stateless_variant(text)
    else:
        text = {"cfg1": progs.CFG1A_TESTCODE, "cfg2": progs.CFG2_LOG_GAIN, "logtube": progs.CFG1B_LOGTUBE}[name]
    prog = fx.Program(text)
    assert prog.loaded, prog.errors()
    ctl = {nm: rng.random(n).astype(np.float32) for nm in prog.controls()}
    ht = check(po, text, n, [37, 8, 1], rng, controls=ctl, what=name, inplace=inplace)
    assert "fx_translated_sl" in ht.src
    # several blocks in one launch
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, n, 1)
    ht = HostTranslated(prog, n, 1)
    for nm, v in ctl.items():
        orc.set_register(prog.reg_index(nm), v); ht.registers[prog.reg_index(nm), :] = v
    xs = [(1.8 * rng.random((1, 21, n)) - 0.9).astype(np.float32) for _ in range(3)]
    ys = ht.process_blocks(xs, 21, seg_len=4, inplace=inplace)
    for b in range(3):
        assert_bits_equal(ys[b], orc.process(xs[b]), f"{name} fused block {b}")
    assert_bits_equal(ht.registers, orc.registers, name + " registers after fused blocks")
    assert_bits_equal(ht.acc, orc.acc, name + " accumulator after fused blocks")
    assert_bits_equal(ht.out_latch, orc.out_latch, name + " latch after fused blocks")
    assert_bits_equal(ht.counts, orc.counts, name + " counters after fused blocks")


def stateless_variant(text: str) -> str:
    """Keeps a random program only if the product's analysis calls it stateless; otherwise falls back to a fixed one."""
    prog = fx.Program(text)
    src, _ = fx.translate_source(prog)
    if src is not None and "fx_translated_sl" in src:
        return text
    return "\n".join(["static a", "static b", "control g = 0.5", "input in_l 0", "output out_l 0", "macs a, 0, in_l, g", "log b, a, 5, 0",
                      "limit a, b, a, 0.25", "exp b, a, 3, 0", "macsn out_l, b, a, g", "end"])


@pytest.mark.parametrize("name,inplace", with_inplace(["cfg3_200", "tap", "two_rings", "xdelay"]))
def test_delay_lines_streaming_kernel(po, name, inplace):
    """Delay lines whose periods are independent over a stretch (ring positions shared by all instances): the streaming kernel with TRAM
    READs loaded like inputs and WRITEs stored like outputs, one emulated launch per stretch, work items in random order."""
    rng = np.random.default_rng(23)
    n = 8
    if name == "cfg3_200":
        text, span = progs.cfg3_delay(200), 200
    elif name == "tap":          # write first, read 150 periods later (write offset 3): read-after-write distance 153, write-after-read 347
        text = "\n".join(["static a", "static rd", "input in_l 0", "output out_l 0", "itramsize 500 ", "idelay write, in_l, at, 3",
                          "idelay read, rd, at, 150", "macs a, rd, 0.5, 0.5", "macs out_l, in_l, rd, 0.5", "end"])
        span = 153
    elif name == "two_rings":
        text = "\n".join(["static a", "static a2", "static rd", "static rx", "input in_l 0", "output out_l 0", "itramsize 700 ", "xtramsize 300 ",
                          "idelay read, rd, at, 0", "macs a, in_l, rd, 0.5", "idelay write, a, at, 0", "xdelay write, in_l, at, 0", "xdelay read, rx, at, 150",
                          "macs a2, rx, 0.5, 0.5", "macs out_l, a2, rd, 0.5", "end"])
        span = 150
    else:
        text = "\n".join(["static a", "static rd", "input in_l 0", "output out_l 0", "xtramsize 2000 ", "xdelay read, rd, at, 0", "macs a, in_l, rd, 0.5",
                          "xdelay write, a, at, 0", "macs out_l, in_l, rd, 0.5", "end"])
        span = 2000
    ht = check(po, text, n, [70, 400, 33, 1, 250], rng, what=name, span=span, inplace=inplace)
    assert "fx_translated_sl" in ht.src and "#define FXT_NTR 0" not in ht.src


@pytest.mark.parametrize("sel", [*range(32), "dynamic"])
def test_table_sweep_all_selectors(po, sel):
    """The sweep of test_gpu_parity.py::test_table_sweep_all_selectors on the generated streaming kernel: LOG and EXP at every table
    boundary, its neighbours and the U6 inputs (|A| > 1, signed zeros, subnormals, NaN), per selector; the range flag as the oracle's."""
    rng = np.random.default_rng(8)
    n = 512
    grid = progs.table_sweep_grid(n, rng)
    x = np.tile(grid, (3, 1)).reshape(1, 3, n)
    if sel == "dynamic":
        texts = ["static a\ninput in_l 0\ncontrol sel = 3\noutput out_l 0\nlog a, in_l, sel, 0\nexp out_l, a, sel, 0\nend"]
    else:
        texts = [f"static a\ninput in_l 0\noutput out_l 0\n{op} a, in_l, {sel}, 0\nmacs out_l, 0, a, 1.0\nend" for op in ("log", "exp")]
    for text in texts:
        prog = fx.Program(text)
        assert prog.loaded, prog.errors()
        img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
        orc = po.Oracle(img, n, 1)
        ht = HostTranslated(prog, n, 1)
        assert "fx_translated_sl" in ht.src
        if sel == "dynamic":
            v = rng.integers(0, 32, n).astype(np.float32)
            orc.set_register("sel", v); ht.registers[prog.reg_index("sel"), :] = v
        what = text.split("\n")[-3]
        assert_bits_equal(ht.process(x), orc.process(x), what + " outputs")
        assert_bits_equal(ht.registers, orc.registers, what + " registers")
        assert_bits_equal(ht.counts, orc.counts, what + " counters")
        assert orc.flags & fx.RT_TABLE_RANGE and int(ht.flags[0]) == orc.flags, (what, int(ht.flags[0]), orc.flags)


@pytest.mark.parametrize("name", ["cfg5", "random"])
def test_source_compiles_for_sm_100a(name):
    """NVRTC (no device needed) turns the generated source into an sm_100a CUBIN."""
    text = progs.cfg5_allops() if name == "cfg5" else progs.random_program(np.random.default_rng(3), 64, xtram=True)
    prog = fx.Program(text)
    src, cubin = fx.translate_source(prog, 1, compile_check=True)
    assert src is not None
    if cubin == -1:
        pytest.skip("libnvrtc not loadable here")
    assert cubin > 1000


def test_branch_free_table_index_matches_the_reference_rule(tmp_path):
    """fxt_table_index (no branch, U6 clamp by clamping x) against the branchy rule of the interpreter kernels / the oracle, over every
    5th binary32 bit pattern (tests/table_index_check.c; `table_index_check 1` sweeps all 2^32 and was run once: 0 mismatches)."""
    import os, subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    exe = str(tmp_path / "table_index_check")
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-o", exe, os.path.join(here, "table_index_check.c"), "-lm"], check=True)
    r = subprocess.run([exe, "5"], capture_output=True, text=True)
    assert r.returncode == 0 and "mismatches: 0" in r.stdout, r.stdout
