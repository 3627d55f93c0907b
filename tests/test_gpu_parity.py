"""GPU parity: the CUDA interpreter (through the C ABI) against the oracle, bit for bit.

Every case parses the program with the product's host front-end, hands the same decoded image to
oracle/liboracle.so and to fx8010_gpu_load_program, feeds both the same seeded inputs and controls
and compares outputs, the whole register file, accumulator, LFSR, output latch, TRAM pointers,
TRAM contents, executed-instruction counters and runtime flags as raw bit patterns (tolerance: 0).
"""
import os

import numpy as np
import pytest

import progs
from conftest import assert_bits_equal

pytestmark = pytest.mark.gpu


def make_pair(fx, po, text, n, channels=1):
    prog = fx.Program(text, channels=channels)
    assert prog.loaded, prog.errors()
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, n, channels)
    gpu = fx.Gpu(n, channels)
    gpu.load_program(prog)
    return prog, img, orc, gpu


def compare_state(gpu, orc, img, what, tram_instances=(0,)):
    assert_bits_equal(gpu.registers(), orc.registers, what + " registers")
    acc, lfsr, latch, ptrs = gpu.scalars()
    assert_bits_equal(acc, orc.acc, what + " accumulator")
    assert_bits_equal(lfsr, orc.lfsr, what + " lfsr")
    assert_bits_equal(latch, orc.out_latch, what + " out latch")
    assert_bits_equal(ptrs, orc.tram_ptrs, what + " tram pointers")
    assert_bits_equal(gpu.counts(), orc.counts, what + " instruction counters")
    d = gpu.dims()
    for which, size in ((0, d.itram_size), (1, d.xtram_size)):
        if size:
            for i in tram_instances:
                assert_bits_equal(gpu.tram(which, i), orc.tram(which, i), f"{what} tram{which}[{i}]")
    assert gpu.flags() == orc.flags, what + " runtime flags"


def run_case(fx, po, text, n, blocks, rng, channels=1, controls=None, stimulus=None, what="case"):
    prog, img, orc, gpu = make_pair(fx, po, text, n, channels)
    try:
        for name, vals in (controls or {}).items():
            idx = prog.reg_index(name)
            assert idx >= 0
            gpu.set_controls(idx, vals)
            orc.set_register(idx, vals)
        start = 0
        for s in blocks:
            if stimulus is not None:
                x = stimulus(start, s)
            else:
                x = (1.8 * rng.random((channels, s, n)) - 0.9).astype(np.float32)
            yo = orc.process(x)
            yg = gpu.process_host(x)
            assert_bits_equal(yg, yo, f"{what} outputs of block at {start}")
            start += s
        inst = sorted({0, n - 1, n // 2})
        compare_state(gpu, orc, img, what, inst)
        return gpu.launch_info()
    finally:
        gpu.close()


# ---- BASELINE.json configs at sizes the oracle finishes in seconds --------------------------------

def test_cfg1_testcode_shipped(fx, po):
    rng = np.random.default_rng(progs.SEED)
    n = 64
    vol = rng.random(n).astype(np.float32)
    x = progs.sine_bank(n, 257, rng)
    run_case(fx, po, progs.CFG1A_TESTCODE, n, [100, 157], rng, controls={"volume": vol},
             stimulus=lambda a, s: x[a:a + s].reshape(1, s, n), what="cfg1a")


def test_cfg1b_logtube_edges(fx, po):
    n = 16
    edge = np.array([1.0, -1.0, 0.0, -0.0, 1 / 63, -1 / 63, 0.99999994, -0.99999994, 0.5, -0.5, 0.0159, 0.9375,
                     1e-30, -1e-30, 0.031746034, 0.96825397], dtype=np.float32)
    rng = np.random.default_rng(1)
    run_case(fx, po, progs.CFG1B_LOGTUBE, n, [8], rng, stimulus=lambda a, s: np.tile(edge, (s, 1)).reshape(1, s, n), what="cfg1b")


@pytest.mark.parametrize("n", [4096, 1000, 333])
def test_cfg2_log_gain(fx, po, n):
    rng = np.random.default_rng(progs.SEED)
    vol = rng.random(n).astype(np.float32)
    x = progs.sine_bank(n, 1024 + 40, rng)
    info = run_case(fx, po, progs.CFG2_LOG_GAIN, n, [1024, 40], rng, controls={"volume": vol},
                    stimulus=lambda a, s: x[a:a + s].reshape(1, s, n), what=f"cfg2 n={n}")
    assert info.kernel_variant & 4, "cfg2 is stateless: the time axis must be splittable"


@pytest.mark.parametrize("size", [100, 1000, 8192])
def test_cfg3_delay(fx, po, size):
    rng = np.random.default_rng(progs.SEED)
    n = 256
    s = min(2 * size + 33, 2500)
    x = progs.impulse_noise(n, s, rng)
    run_case(fx, po, progs.cfg3_delay(size), n, [s // 2, s - s // 2], rng,
             stimulus=lambda a, k: x[a:a + k].reshape(1, k, n), what=f"cfg3 S={size}")


def test_cfg3_delay_65536(fx, po):
    rng = np.random.default_rng(progs.SEED)
    n = 32
    x = progs.impulse_noise(n, 1500, rng)
    run_case(fx, po, progs.cfg3_delay(65536), n, [1500], rng, stimulus=lambda a, k: x[a:a + k].reshape(1, k, n), what="cfg3 S=65536")


def test_cfg4_onepole_sweep(fx, po):
    rng = np.random.default_rng(progs.SEED)
    n = 2048
    cutoff = (0.001 + 0.998 * np.arange(n) / (n - 1)).astype(np.float32)
    x = progs.sine_bank(n, 700, rng)
    run_case(fx, po, progs.CFG4_ONEPOLE, n, [512, 188], rng, controls={"filter_cutoff": cutoff},
             stimulus=lambda a, s: x[a:a + s].reshape(1, s, n), what="cfg4")


def test_cfg5_allops_512(fx, po):
    rng = np.random.default_rng(progs.SEED)
    n = 512
    text = progs.cfg5_allops()
    ctl = {f"k{i}": rng.random(n).astype(np.float32) for i in range(4)}
    x = progs.sine_bank(n, 96, rng, amp_lo=0.9, amp_hi=0.9)
    info = run_case(fx, po, text, n, [64, 32], rng, controls=ctl, stimulus=lambda a, s: x[a:a + s].reshape(1, s, n), what="cfg5")
    assert info.kernel_variant & 1


# ---- one program per feature snippet of the reference's testcode.da ----------------------------------

@pytest.mark.parametrize("name", sorted(progs.SNIPPETS))
def test_snippets(fx, po, name):
    rng = np.random.default_rng(7)
    run_case(fx, po, progs.SNIPPETS[name], 96, [50, 31], rng, what=name)


# ---- random programs over every opcode, with SKIP / TRAM / noise / xTRAM -------------------------------

@pytest.mark.parametrize("seed", range(12))
def test_random_programs(fx, po, seed):
    rng = np.random.default_rng(1000 + seed)
    n = [128, 100, 37, 64][seed % 4]
    ch = 1 + seed % 2
    text = progs.random_program(rng, 60 + 10 * seed, channels=ch, xtram=(seed % 3 == 0), read_offsets=(seed % 4 == 1))
    run_case(fx, po, text, n, [40, 25], rng, channels=ch, what=f"random {seed}")


@pytest.mark.parametrize("seed", range(4))
def test_random_programs_unsafe(fx, po, seed):
    """Operands may leave [-1,1], ccr appears as an operand, LOG/EXP may see out-of-range input
    (rule U6: clamped + flagged identically by oracle and kernel)."""
    rng = np.random.default_rng(2000 + seed)
    text = progs.random_program(rng, 80, safe=False, skip=(seed % 2 == 0), wild_tables=True)
    run_case(fx, po, text, 64, [30, 30], rng, what=f"unsafe {seed}")


def test_end_skipped_wraps_and_cap(fx, po):
    """END skipped: the program runs again carrying the skip count (reference :1243); a program that
    always skips END is cut off after FX8010_MAX_PASSES and flagged (rule U9)."""
    rng = np.random.default_rng(3)
    wrap = progs.END_SKIPPED_WRAP
    run_case(fx, po, wrap, 64, [40], rng, what="end skipped sometimes")
    forever = "static a\noutput out_l 0\nmacs a, 0, 0.5, 0.5\nmacs out_l, a, 0.1, 0.1\nskip ccr, ccr, 2, 1\nend"
    prog, img, orc, gpu = make_pair(fx, po, forever, 8)
    try:
        assert_bits_equal(gpu.process_host(None, 3), orc.process(None, 3), "capped outputs")
        assert gpu.flags() & fx.RT_END_SKIPPED_CAP
        compare_state(gpu, orc, img, "capped")
    finally:
        gpu.close()


def test_two_channels_input_index_quirk(fx, po):
    """X and Y operands of INPUT type read the channel of A (reference :1057-1060)."""
    rng = np.random.default_rng(4)
    text = "static a\ninput in_l 0\ninput in_r 1\noutput out_l 0\noutput out_r 1\nmacs out_r, 0, in_r, 1.0\nmacs out_l, in_r, in_l, 0.5\nmacs a, 0.1, 0.5, in_r\nend"
    run_case(fx, po, text, 40, [33], rng, channels=2, what="two channels")


def test_state_roundtrip_checkpoint(fx, po):
    """get_state -> new handle -> set_state continues bit-identically (checkpoint / resume)."""
    rng = np.random.default_rng(5)
    text = progs.random_program(rng, 50, xtram=True)
    n = 32
    prog, img, orc, gpu = make_pair(fx, po, text, n)
    gpu2 = fx.Gpu(n, 1)
    try:
        x1 = (1.8 * rng.random((1, 64, n)) - 0.9).astype(np.float32)
        x2 = (1.8 * rng.random((1, 64, n)) - 0.9).astype(np.float32)
        gpu.process_host(x1); orc.process(x1)
        gpu2.load_program(prog)
        gpu2.set_registers(gpu.registers())
        acc, lfsr, latch, ptrs = gpu.scalars()
        gpu2.set_scalars(acc, lfsr, latch, ptrs)
        d = gpu.dims()
        for i in range(n):
            if d.itram_size: gpu2.set_tram(0, i, gpu.tram(0, i))
            if d.xtram_size: gpu2.set_tram(1, i, gpu.tram(1, i))
        yo = orc.process(x2)
        assert_bits_equal(gpu2.process_host(x2), yo, "resumed outputs")
        assert_bits_equal(gpu2.registers(), orc.registers, "resumed registers")
    finally:
        gpu.close(); gpu2.close()


def test_device_pointers_and_streams(fx, po):
    import torch
    rng = np.random.default_rng(6)
    n, s = 4096, 256
    prog, img, orc, gpu = make_pair(fx, po, progs.CFG4_ONEPOLE, n)
    try:
        cut = rng.random(n).astype(np.float32)
        idx = prog.reg_index("filter_cutoff")
        st = torch.cuda.Stream()
        d_cut = torch.from_numpy(cut).cuda()
        x = progs.sine_bank(n, 2 * s, rng).reshape(1, 2 * s, n)
        d_x = torch.from_numpy(x).cuda()
        torch.cuda.synchronize()
        gpu.set_controls_device(idx, d_cut, st.cuda_stream)
        a = d_x[0, :s].contiguous(); b = d_x[0, s:].contiguous()
        ya = torch.empty_like(a); yb = torch.empty_like(b)
        torch.cuda.synchronize()
        gpu.process_device(a, ya, s, st.cuda_stream)
        gpu.process_device(b, yb, s, st.cuda_stream)
        gpu.synchronize(st.cuda_stream)
        orc.set_register(idx, cut)
        yo = orc.process(x)
        assert_bits_equal(np.concatenate([ya.cpu().numpy(), yb.cpu().numpy()])[None], yo, "device path outputs")
        compare_state(gpu, orc, img, "device path")
    finally:
        gpu.close()


def test_table_sweep_all_selectors(fx, po):
    """LOG and EXP over a dense grid of inputs (every table boundary and its neighbours, and the U6 inputs: |A| > 1, signed zeros,
    subnormals, NaN) for each of the 32 selectors and for a per-instance selector held in a control, on the interpreter (translate
    mode 0) and on the translated streaming kernel (mode 2: the programs are stateless and 4 096 instances allow its 16-byte
    accesses).  The runtime flags follow the oracle's."""
    n = 4096
    grid = progs.table_sweep_grid(n, np.random.default_rng(8))
    x = np.tile(grid, (3, 1)).reshape(1, 3, n)
    dynamic = "static a\ninput in_l 0\ncontrol sel = 3\noutput out_l 0\nlog a, in_l, sel, 0\nexp out_l, a, sel, 0\nend"
    texts = [f"static a\ninput in_l 0\noutput out_l 0\n{op} a, in_l, {sel}, 0\nmacs out_l, 0, a, 1.0\nend" for sel in range(32) for op in ("log", "exp")]
    for mode in (0, 2):
        for text in texts + [dynamic]:
            what = f"{text.split(chr(10))[-3]}, mode {mode}"
            prog, img, orc, gpu = make_pair(fx, po, text, n)
            try:
                gpu.set_option(fx.OPT_TRANSLATE, mode)
                if text is dynamic:         # the selector is a control, per instance: the global-memory table path
                    v = np.random.default_rng(9).integers(0, 32, n).astype(np.float32)
                    gpu.set_controls(prog.reg_index("sel"), v); orc.set_register("sel", v)
                assert_bits_equal(gpu.process_host(x), orc.process(x), what + " outputs")
                compare_state(gpu, orc, img, what, (0, 200, n - 1))
                assert orc.flags & fx.RT_TABLE_RANGE and gpu.flags() == orc.flags, (what, gpu.flags(), orc.flags)
                assert bool(gpu.launch_info().kernel_variant & 128) == (mode == 2), (what, hex(gpu.launch_info().kernel_variant))
            finally:
                gpu.close()


@pytest.mark.parametrize("k,b", [(1, 32), (2, 64), (4, 128), (4, 32)])
def test_forced_geometries(fx, po, k, b, monkeypatch):
    """Every contexts-per-thread / block-size variant of the kernel gives the same bits."""
    monkeypatch.setenv("FX8010_TUNE_K", str(k))
    monkeypatch.setenv("FX8010_TUNE_B", str(b))
    rng = np.random.default_rng(9)
    text = progs.random_program(rng, 70, xtram=True)
    run_case(fx, po, text, 200, [37, 20], rng, what=f"K={k} B={b}")
    run_case(fx, po, progs.CFG2_LOG_GAIN, 256, [100], rng, what=f"cfg2 K={k} B={b}")


STATELESS_PROGS = {
    "cfg2": progs.CFG2_LOG_GAIN,
    "testcode": progs.CFG1A_TESTCODE,
    "exp": progs.SNIPPETS["exp"],
    "interp_const": progs.SNIPPETS["interp_const"],
    "andxor": progs.SNIPPETS["andxor"],
    # ccr read as an operand (kept per sample), a temp written twice, two outputs, dynamic table selector
    "ccr_operand": "static a\nstatic b\ninput in_l 0\ncontrol sel = 5\noutput out_l 0\nmacs a, 0, in_l, 0.5\nmacs b, ccr, a, 0.25\n"
                   "log a, b, sel, 0\nmacsn a, a, in_l, 0.125\nmacs out_l, a, b, ccr\nend",
    "two_outputs": "static a\ninput in_l 0\ninput in_r 1\noutput out_l 0\noutput out_r 1\nmacw a, in_l, 0.75, 0.5\nlimit out_r, in_r, a, 0.25\n"
                   "tstneg out_l, in_l, a, 0\nmacintw out_l, out_l, a, 0.75\nend",
}


@pytest.mark.parametrize("name", sorted(STATELESS_PROGS))
@pytest.mark.parametrize("mode", ["M1", "M2", "M4", "M8", "generic", "M8tma"])
def test_stateless_kernel_modes(fx, po, name, mode, monkeypatch):
    """Stateless programs through the sample-batched kernel at every batch length and through the
    generic kernel: identical bits, identical final state (several calls, ragged lengths)."""
    if mode == "M8tma":                 # input stage filled by bulk tensor copies (TMA) instead of cp.async
        monkeypatch.setenv("FX8010_USE_TMA", "2")
        mode = "M8"
    if mode == "generic":
        monkeypatch.setenv("FX8010_NO_STATELESS", "1")
    else:
        monkeypatch.setenv("FX8010_TUNE_M", mode[1:])
    rng = np.random.default_rng(11)
    ch = 2 if name == "two_outputs" else 1
    n = 260
    ctl = {"sel": rng.integers(0, 32, n).astype(np.float32)} if name == "ccr_operand" else None
    info = run_case(fx, po, STATELESS_PROGS[name], n, [1, 37, 8, 3, 100], rng, channels=ch, controls=ctl, what=f"{name} {mode}")
    assert bool(info.kernel_variant & 8) == (mode != "generic"), "wrong kernel took the program"


# Self recurrences: an operand is the instruction's own result of the previous sample period.  They run
# instruction-major, serially in time, with the carried value forwarded in a hardware register.
CARRIED_PROGS = {
    "onepole": progs.CFG4_ONEPOLE,
    "carry_x": "static a = 0.25\ninput in_l 0\noutput out_l 0\nmacs a, in_l, a, 0.9\nmacs out_l, a, in_l, 0.5\nend",
    "carry_y": "static a = 0.5\ninput in_l 0\ncontrol g = 0.7\noutput out_l 0\nmacsn a, in_l, g, a\nlimit out_l, a, in_l, 0.25\nend",
    # two independent recurrences, the second fed by the first; wrap-around arithmetic; the state register is also an output
    "cascade": "static s1 = 0.1\ninput in_l 0\ncontrol c = 0.3\noutput out_l 0\ninterp s1, s1, c, in_l\ninterp out_l, out_l, c, s1\nend",
    "macw_acc": "static ph = 0.0\ninput in_l 0\noutput out_l 0\nmacw ph, ph, in_l, 0.37\nmacintw out_l, ph, ph, 0.5\nend",
    "square": "static a = 0.9\ninput in_l 0\noutput out_l 0\nmacs a, in_l, a, a\nacc3 out_l, a, in_l, 0.125\nend",
    "log_rec": "static a = 0.2\ninput in_l 0\noutput out_l 0\nlog a, a, 3, 0\nmacs a, in_l, a, 0.5\nmacs out_l, a, 0.5, 0.5\nend",
    "log_self": "static a = 0.6\ninput in_l 0\noutput out_l 0\nexp a, a, 2, 0\nmacs out_l, a, in_l, 0.5\nend",
}


@pytest.mark.parametrize("name", sorted(CARRIED_PROGS))
@pytest.mark.parametrize("mode", ["auto", "M2", "M4", "K1", "K2", "nocarry", "noshort", "no_tma", "tma_everywhere"])
def test_carried_recurrences(fx, po, name, mode, monkeypatch):
    if mode == "no_tma":                 # the input stage of a recurrence is filled by bulk tensor copies (TMA) by default
        monkeypatch.setenv("FX8010_USE_TMA", "0")
    elif mode == "tma_everywhere":
        monkeypatch.setenv("FX8010_USE_TMA", "2")
    if mode[0] == "M":
        monkeypatch.setenv("FX8010_TUNE_M", mode[1:])
    elif mode[0] == "K":
        monkeypatch.setenv("FX8010_TUNE_K", mode[1:])
    elif mode == "nocarry":
        monkeypatch.setenv("FX8010_NO_CARRY", "1")
    elif mode == "noshort":
        monkeypatch.setenv("FX8010_NO_CARRY", "1")
        monkeypatch.setenv("FX8010_NO_SHORT", "1")
    rng = np.random.default_rng(21)
    n = 264
    ctl = {}
    if name in ("onepole",):
        ctl["filter_cutoff"] = (0.001 + 0.998 * rng.random(n)).astype(np.float32)
    if name in ("cascade",):
        ctl["c"] = rng.random(n).astype(np.float32)
    info = run_case(fx, po, CARRIED_PROGS[name], n, [1, 2, 37, 8, 16, 3, 100, 1], rng, controls=ctl, what=f"{name} {mode}")
    # log_rec carries `a` from the LAST instruction to the first one: not a self recurrence
    carried = mode not in ("nocarry", "noshort") and name != "log_rec"
    assert bool(info.kernel_variant & 8) == carried, "wrong kernel took the program"
    if mode == "nocarry":
        assert info.kernel_variant & 32, "expected the short-program kernel"
    if mode == "noshort":
        assert not (info.kernel_variant & (8 | 32))


# TRAM programs in the instruction-major kernel: READ streams prefetched a batch ahead when the delay is longer than
# two batches, otherwise the same code one sample at a time.
def _tram_prog(size, order="rw", roff="0", woff="0", x=False, two=None):
    d, sz = ("xdelay", "xtramsize") if x else ("idelay", "itramsize")
    if order == "rw":     # feedback delay line (cfg3): read, mix, write back
        body = f"{d} read, rd, at, {roff}\nmacs a, in_l, rd, 0.5\n{d} write, a, at, {woff}\n"
    else:                 # tap: write the input, read it back delayed (negative ring indices follow rule U1)
        body = f"{d} write, in_l, at, {woff}\n{d} read, rd, at, {roff}\nmacs a, rd, 0.5, 0.5\n"
    decl2, body2 = "", ""
    if two:               # the other TRAM as well: (write offset, read offset)
        decl2 = "xtramsize 300 \n"
        body2 = f"xdelay write, in_l, at, {two[0]}\nxdelay read, rx, at, {two[1]}\nmacs a2, rx, 0.5, 0.5\n"
    return ("static a\nstatic a2\nstatic rd\nstatic rx\ncontrol dly = 5\ninput in_l 0\noutput out_l 0\n"
            f"{sz} {size} \n{decl2}{body}{body2}macs out_l, in_l, rd, 0.5\nend")


TRAM_CASES = {
    "s3": dict(size=3), "s40": dict(size=40), "s64": dict(size=64), "s65": dict(size=65), "s66": dict(size=66), "s100": dict(size=100),
    "s1000": dict(size=1000), "wr_off": dict(size=500, order="wr", roff="200", woff="3"),
    "wr_short": dict(size=500, order="wr", roff="17", woff="0"), "wr_zero": dict(size=90, order="wr"),
    "wr_wrap": dict(size=300, order="wr", roff="5", woff="290"),
    "ctl_off": dict(size=400, order="wr", roff="dly"), "xdelay": dict(size=2000, x=True),
    "two_slow": dict(size=700, two=(7, 2)), "two_fast": dict(size=700, two=(0, 150)),
}


@pytest.mark.parametrize("name", sorted(TRAM_CASES))
@pytest.mark.parametrize("mode", ["auto", "K4", "K2M8", "no_im", "P1", "P2", "K1P4M16", "serial", "tsplitK2M16", "tsplitSEG3"])
def test_tram_instruction_major(fx, po, name, mode, monkeypatch):
    # auto / K4 / K2M8: delay lines whose periods are known to be independent over >= 64 periods are cut along time
    # (blocks longer than that span run as several launches); the other modes switch that off and exercise the serial
    # kernel with its sample split
    if mode in ("P1", "P2", "K1P4M16", "serial"):
        monkeypatch.setenv("FX8010_NO_TSPLIT", "1")
    if mode == "tsplitK2M16":
        monkeypatch.setenv("FX8010_TUNE_K", "2")
        monkeypatch.setenv("FX8010_TUNE_M", "16")
    elif mode == "tsplitSEG3":
        monkeypatch.setenv("FX8010_TUNE_SEG", "3")
    if mode == "K4":
        monkeypatch.setenv("FX8010_TUNE_K", "4")
    elif mode == "K2M8":
        monkeypatch.setenv("FX8010_TUNE_K", "2")
        monkeypatch.setenv("FX8010_TUNE_M", "8")
    elif mode == "no_im":
        monkeypatch.setenv("FX8010_NO_TRAM_IM", "1")
    elif mode in ("P1", "P2"):  # threads per instance column (they split each batch's samples)
        monkeypatch.setenv("FX8010_TUNE_P", mode[1:])
    elif mode == "K1P4M16":
        monkeypatch.setenv("FX8010_TUNE_K", "1")
        monkeypatch.setenv("FX8010_TUNE_P", "4")
        monkeypatch.setenv("FX8010_TUNE_M", "16")
    rng = np.random.default_rng(31)
    n = 136
    text = _tram_prog(**TRAM_CASES[name])
    ctl = {"dly": rng.integers(70, 390, n).astype(np.float32)} if name == "ctl_off" else None
    x = progs.impulse_noise(n, 700, rng)
    info = run_case(fx, po, text, n, [1, 150, 33, 64, 2, 450], rng, controls=ctl,
                    stimulus=lambda a, k: x[a:a + k].reshape(1, k, n), what=f"tram {name} {mode}")
    assert bool(info.kernel_variant & 8) == (mode != "no_im"), "wrong kernel took the program"


def test_input_channel_quirk_takes_generic_kernel(fx, po):
    """X/Y INPUT operands read A's channel (reference :1057-1060): such a program is stateless but must not
    use the stage-aliasing kernel."""
    rng = np.random.default_rng(12)
    text = "input in_l 0\ninput in_r 1\noutput out_l 0\noutput out_r 1\nmacs out_l, in_l, in_r, 0.5\nmacs out_r, 0.25, in_r, in_l\nend"
    info = run_case(fx, po, text, 64, [20, 5], rng, channels=2, what="quirk")
    assert not (info.kernel_variant & 8)


def test_errors_are_loud(fx):
    g = fx.Gpu(8, 1)
    try:
        with pytest.raises(fx.FxError) as e:
            g.process_host(np.zeros((1, 4, 8), np.float32))
        assert e.value.code == 3          # ERR_NO_PROGRAM
        p = fx.Program("static a\nidelay write, a, at, 0\nend")
        assert p.loaded
        with pytest.raises(fx.FxError) as e:
            g.load_program(p)             # IDELAY without itramsize: rule U4
        assert e.value.code == 4
    finally:
        g.close()


def test_facade_per_sample_process_matches_reference_driver(fx, po):
    """The legacy drop-in call: one process() per sample, volume slider changed every 8 samples,
    exactly as the reference's main.cpp:103-122 drives it; anchors from SURVEY.md §8c."""
    p = fx.Program(progs.CFG1A_TESTCODE)
    ramp = np.array([(i - 16) / 16 for i in range(32)], dtype=np.float32)
    out = []
    for i in range(32):
        if i % 8 == 0:
            assert p.set_register("volume", [0.1, 0.25, 0.5, 1.0][i // 8]) == 0
        out.append(p.process(ramp[i:i + 1])[0, 0])
    out = np.array(out, dtype=np.float32)
    want = [0xbdcccccd, 0xbdc00000, 0xbdb33333, 0xbda66667, 0xbd99999a, 0xbd8ccccd, 0xbd800000, 0xbd666667,
            0xbe000000, 0xbde00000, 0xbdc00000, 0xbda00000, 0xbd800000, 0xbd400000, 0xbd000000, 0xbc800000,
            0x00000000, 0x3d000000, 0x3d800000, 0x3dc00000, 0x3e000000, 0x3e200000, 0x3e400000, 0x3e600000] + \
           [0x3f000000 + 0x100000 * k for k in range(8)]
    assert [int(v) for v in out.view(np.uint32)] == want
    assert p.instruction_counter == 64
    assert p.get_register("nonexistent") == 1.0 and p.set_register("nonexistent", 0.0) == 1
    p.close()


# ---- edge cases ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 2, 3, 5])
def test_tiny_instance_counts(fx, po, n):
    rng = np.random.default_rng(20 + n)
    run_case(fx, po, progs.CFG2_LOG_GAIN, n, [9, 1, 30], rng, controls={"volume": rng.random(n).astype(np.float32)}, what=f"cfg2 n={n}")
    run_case(fx, po, progs.random_program(rng, 40, xtram=True), n, [17, 8], rng, what=f"random n={n}")


def test_zero_samples_and_long_batch(fx, po):
    rng = np.random.default_rng(30)
    prog, img, orc, gpu = make_pair(fx, po, progs.CFG4_ONEPOLE, 8)
    try:
        assert gpu.process_host(np.zeros((1, 0, 8), np.float32)).shape == (1, 0, 8)
        x = (1.8 * rng.random((1, 5000, 8)) - 0.9).astype(np.float32)
        assert_bits_equal(gpu.process_host(x), orc.process(x), "5000-sample batch")
        compare_state(gpu, orc, img, "long batch")
    finally:
        gpu.close()


def test_maximum_program_length(fx, po):
    """1 000 instructions (FX8010_MAX_INSTRUCTIONS) run; one more is refused with ERR_CAPACITY."""
    rng = np.random.default_rng(31)
    text = progs.random_program(rng, 999 - 1, skip=True, tram=True, noise=True)      # + 1 output driver + END = 1000
    prog = fx.Program(text)
    assert prog.loaded and len(prog.instructions()) == 1000
    run_case(fx, po, text, 32, [6], rng, what="1000 instructions")
    big = fx.Program(progs.random_program(rng, 999, skip=False, tram=False, noise=False))
    assert big.loaded and len(big.instructions()) == 1001
    g = fx.Gpu(4, 1)
    try:
        with pytest.raises(fx.FxError) as e:
            g.load_program(big)
        assert e.value.code == 5
    finally:
        g.close()


def test_handles_are_not_limited_by_constant_memory(fx):
    """Any number of live handles per device (the reference allows any number of FX8010 objects, include/FX8010.h:51):
    programs share a constant-memory arena and are re-uploaded when evicted (see test_gpu_fullsize.py for the eviction case)."""
    p = fx.Program(progs.CFG1A_TESTCODE)
    hs = [fx.Gpu(4, 1) for _ in range(6)]
    try:
        for g in hs:
            g.load_program(p)
        x = np.full((1, 3, 4), 0.5, np.float32)
        ys = [g.process_host(x) for g in hs]
        for y in ys[1:]:
            assert np.array_equal(ys[0], y)
    finally:
        for g in hs:
            g.close()


def test_full_size_xtram(fx, po):
    """xtramsize 1048576 (MAX_XDELAY_SIZE, include/FX8010.h:42): 4 MiB ring per instance."""
    rng = np.random.default_rng(32)
    text = ("static a\nstatic rd\ninput in_l 0\noutput out_l 0\nxtramsize 1048576 \nxdelay read, rd, at, 0\nmacs a, in_l, rd, 0.5\n"
            "xdelay write, a, at, 0\nxdelay read, rd, at, 5\nmacs out_l, in_l, rd, 0.5\nend")
    prog, img, orc, gpu = make_pair(fx, po, text, 8)
    try:
        ptr = np.zeros((4, 8), np.int32); ptr[2] = 1048570; ptr[3] = 1048572      # pointers about to wrap
        gpu.set_scalars(ptrs=ptr); orc.tram_ptrs[:] = ptr
        x = (1.8 * rng.random((1, 40, 8)) - 0.9).astype(np.float32)
        assert_bits_equal(gpu.process_host(x), orc.process(x), "xtram outputs")
        compare_state(gpu, orc, img, "xtram", tram_instances=(0, 7))
    finally:
        gpu.close()


def test_literal_register_overwritten_through_api(fx, po):
    """setRegisterValue can write ANY register, literals included (source/FX8010.cpp:236-253).  The LOG selector
    '3' and the MACS addend '0' are folded at encode time while they are uniform; writing them must undo that."""
    rng = np.random.default_rng(33)
    n = 128
    prog, img, orc, gpu = make_pair(fx, po, progs.CFG1B_LOGTUBE, n)
    try:
        x = (1.8 * rng.random((1, 20, n)) - 0.9).astype(np.float32)
        assert_bits_equal(gpu.process_host(x), orc.process(x), "before")
        sel = rng.integers(0, 32, n).astype(np.float32); add = (0.2 * rng.random(n)).astype(np.float32)
        for name, v in (("3", sel), ("0", add)):
            gpu.set_controls(prog.reg_index(name), v); orc.set_register(name, v)
        assert_bits_equal(gpu.process_host(x), orc.process(x), "per-instance literals")
        gpu.set_controls(prog.reg_index("3"), [7.0], broadcast=True); orc.set_register("3", np.full(n, 7.0, np.float32))
        assert_bits_equal(gpu.process_host(x), orc.process(x), "broadcast literal")
        compare_state(gpu, orc, img, "literals")
    finally:
        gpu.close()


def test_async_host_batches_chain_in_order(fx, po):
    """fx8010_gpu_process_batch_host_async: queued calls on a stateful program keep their order and their
    state; outputs are complete after fx8010_gpu_synchronize; a device-pointer call afterwards waits for them."""
    import torch
    rng = np.random.default_rng(40)
    n, s, calls = 512, 300, 7
    text = progs.random_program(rng, 30, xtram=True)
    prog, img, orc, gpu = make_pair(fx, po, text, n)
    try:
        ins = [fx.pinned_array((1, s, n)) for _ in range(calls)]
        outs = [fx.pinned_array((1, s, n)) for _ in range(calls)]
        for a, _ in ins:
            a[...] = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
        for (a, _), (b, _) in zip(ins, outs):
            gpu.process_host_ptr(a.ctypes.data, b.ctypes.data, s, wait=False)
        d_x = torch.from_numpy(ins[0][0].copy()).cuda(); d_y = torch.empty_like(d_x)
        torch.cuda.synchronize()
        gpu.process_device(d_x, d_y, s, None)                 # must run after the queued host batches
        gpu.synchronize(None)
        for k, ((a, _), (b, _)) in enumerate(zip(ins, outs)):
            assert_bits_equal(b, orc.process(a), f"async call {k}")
        assert_bits_equal(d_y.cpu().numpy(), orc.process(ins[0][0]), "device call after async")
        compare_state(gpu, orc, img, "async")
    finally:
        gpu.close()


def test_trace_matches_execution(fx, po):
    """fx8010_gpu_trace: same outputs and state as a normal run; per-instruction records are consistent with
    the oracle (executed-instruction count, the values the output drivers leave, the final register file)."""
    rng = np.random.default_rng(50)
    for text in (progs.CFG2_LOG_GAIN, progs.SNIPPETS["skip"], progs.random_program(rng, 40, xtram=True)):
        n, s, inst = 24, 9, 5
        prog, img, orc, gpu = make_pair(fx, po, text, n)
        try:
            x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
            out, rec = gpu.trace(x, inst)
            assert_bits_equal(out, orc.process(x), "trace outputs")
            compare_state(gpu, orc, img, "trace state")
            instrs = prog.instructions()
            assert rec.shape == (s, len(instrs))
            assert [int(v) for v in rec["index"][0]] == list(range(len(instrs)))
            assert [int(v) for v in rec["opcode"][0]] == [i[0] for i in instrs]
            assert int(rec["executed"].sum()) == int(orc.counts[inst])
            regs = prog.registers()
            last = rec[-1]
            for k, ins in enumerate(instrs):                    # a register nobody touches afterwards keeps its traced value
                later = {j[1] for j in instrs[k + 1:]} | {j[2] for j in instrs[k + 1:]}
                if last["executed"][k] and ins[0] < 15 and ins[1] not in later and ins[1] != 0 and regs[ins[1]][0] != 3:
                    assert np.float32(last["r"][k]).view(np.uint32) == orc.registers[ins[1], inst].view(np.uint32)
            # and a normal batch afterwards continues from the traced state
            x2 = (1.8 * rng.random((1, 7, n)) - 0.9).astype(np.float32)
            assert_bits_equal(gpu.process_host(x2), orc.process(x2), "after trace")
        finally:
            gpu.close()


@pytest.mark.parametrize("order", ["rw", "wr"])
def test_tram_pointers_differ_per_instance(fx, po, order):
    """TRAM pointers are per-instance state (set through the checkpoint API here): neighbouring instances then sit
    at different ring positions (no vector access), and some have a delay shorter than two batches, so their warps
    take the one-sample-at-a-time path while others prefetch."""
    rng = np.random.default_rng(51)
    n, size = 192, 400
    text = _tram_prog(size, order=order, roff="30" if order == "wr" else "0", woff="2")
    prog, img, orc, gpu = make_pair(fx, po, text, n)
    try:
        ptrs = np.zeros((4, n), np.int32)
        ptrs[0] = rng.integers(0, size, n)                       # iw
        ptrs[1] = (ptrs[0] + rng.integers(0, size, n)) % size    # ir: any distance, including very short ones
        ptrs[1, 32:64] = (ptrs[0, 32:64] + 200) % size           # one warp (K = 1) / part of one (K = 4) comfortably far
        ptrs[1, 64:68] = (ptrs[0, 64:68] + 1) % size
        acc, lfsr, latch, _ = gpu.scalars()
        gpu.set_scalars(acc, lfsr, latch, ptrs)
        orc.tram_ptrs[...] = ptrs
        ring = (rng.random((n, size)) - 0.5).astype(np.float32)
        for i in range(n):
            gpu.set_tram(0, i, ring[i])
            orc.set_tram(0, i, ring[i])
        for s in (1, 70, 64, 33):
            x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
            assert_bits_equal(gpu.process_host(x), orc.process(x), f"outputs, per-instance pointers, {order}")
        compare_state(gpu, orc, img, "per-instance pointers", (0, 40, 65, n - 1))
        assert gpu.launch_info().kernel_variant & 8
    finally:
        gpu.close()


@pytest.mark.parametrize("seed", range(24))
def test_fuzz_instruction_major(fx, po, seed):
    """Random programs of the instruction-major kernel's data-flow class (self recurrences, same-period flow, one
    READ + one WRITE per TRAM), against the oracle: outputs and the whole state, several ragged calls."""
    rng = np.random.default_rng(1000 + seed)
    tram = ["", "", "i", "x", "ix"][seed % 5]
    ch = 2 if seed % 7 == 3 else 1
    text = progs.random_flow_program(rng, int(rng.integers(2, 14)), channels=ch, tram=tram, size=int(rng.choice([5, 70, 200, 900])))
    n = int(rng.choice([96, 130, 257]))
    info = run_case(fx, po, text, n, [1, 40, 7, 64, 33], rng, channels=ch, what=f"flow fuzz {seed}")
    if ch == 1:     # (with two channels an X / Y input operand reads A's channel, reference :1057-1060: those programs take the generic kernel)
        assert info.kernel_variant & 8, "the generator is meant to stay inside the instruction-major class:\n" + text


@pytest.mark.parametrize("seed", range(6))
def test_fuzz_cross_instruction_carry_leaves_the_instruction_major_kernel(fx, po, seed):
    rng = np.random.default_rng(2000 + seed)
    text = progs.random_flow_program(rng, int(rng.integers(3, 9)), cross=True)
    info = run_case(fx, po, text, 100, [1, 30, 9], rng, what=f"cross fuzz {seed}")
    first = text.split("\n")
    body0 = [l for l in first if l.split(" ")[0] in ("macs", "macsn", "acc3", "macints", "interp", "macw", "macwn", "macintw", "limit", "limitn", "tstneg", "log", "exp", "andxor")][0]
    if not body0.startswith(("log", "exp")):       # LOG/EXP never read Y: nothing is carried there
        assert not (info.kernel_variant & 8), text


# ---- the caller's block loop (SURVEY.md §8f-2): control changes inside a batch, planar audio buffers --------------

@pytest.mark.parametrize("name", ["testcode", "cfg2", "onepole", "delay", "dynsel"])
def test_control_events_inside_a_batch(fx, po, name):
    """The reference driver's pattern (source/main.cpp:107-114): a slider changes every 8 sample periods, between
    process() calls.  One process_batch_events call with the schedule == the oracle stepped stretch by stretch."""
    import torch
    rng = np.random.default_rng(41)
    n = 300
    text, ctl = {
        "testcode": (progs.CFG1A_TESTCODE, "volume"),
        "cfg2": (progs.CFG2_LOG_GAIN, "volume"),
        "onepole": (progs.CFG4_ONEPOLE, "filter_cutoff"),
        "delay": ("static a\nstatic rd\ncontrol fb = 0.5\ninput in_l 0\noutput out_l 0\nitramsize 150 \nidelay read, rd, at, 0\n"
                  "macs a, in_l, rd, fb\nidelay write, a, at, 0\nmacs out_l, in_l, rd, fb\nend", "fb"),
        # the control is a LOG table selector: the literal-selector encoding has to follow it
        "dynsel": ("static a\ninput in_l 0\ncontrol sel = 3\noutput out_l 0\nlog a, in_l, sel, 0\nmacs out_l, 0, a, 0.5\nend", "sel"),
    }[name]
    prog, img, orc, gpu = make_pair(fx, po, text, n)
    try:
        reg = prog.reg_index(ctl)
        s_total = 100
        x = (1.8 * rng.random((1, s_total, n)) - 0.9).astype(np.float32)
        events = []
        for s0 in range(0, s_total, 8):
            if name == "dynsel":
                v = float(rng.integers(0, 32)) if (s0 // 8) % 2 else rng.integers(0, 32, n).astype(np.float32)
            else:
                v = float(rng.random()) if (s0 // 8) % 3 == 0 else rng.random(n).astype(np.float32)
            events.append((s0, reg, v))
        events.insert(3, (16, reg, 0.125))             # two changes at the same sample: the later one wins
        events.sort(key=lambda e: e[0])
        # oracle: stretch by stretch
        yo = np.zeros_like(x)
        bounds = sorted({e[0] for e in events} | {s_total})
        for a, b in zip(bounds[:-1], bounds[1:]):
            for (s, r, v) in events:
                if s == a:
                    orc.set_register(r, np.full(n, v, np.float32) if np.isscalar(v) else v)
            yo[:, a:b] = orc.process(np.ascontiguousarray(x[:, a:b]))
        d_in = torch.from_numpy(x).cuda()
        d_out = torch.empty_like(d_in)
        st = torch.cuda.Stream()
        gpu.process_device_events(d_in, d_out, s_total, events, st.cuda_stream)
        gpu.synchronize(st.cuda_stream)
        assert_bits_equal(d_out.cpu().numpy(), yo, f"{name} outputs with control events")
        compare_state(gpu, orc, img, f"{name} events", (0, n - 1))
    finally:
        gpu.close()


@pytest.mark.parametrize("n,s", [(300, 77), (64, 1024), (1, 5), (33, 1)])
def test_planar_buffers(fx, po, n, s):
    """[channel][instance][sample] device buffers in and out (what an audio host holds)."""
    import torch
    rng = np.random.default_rng(42)
    text = "static a\ninput in_l 0\ninput in_r 1\noutput out_l 0\noutput out_r 1\nmacs a, in_l, in_l, 0.5\nmacs out_l, a, 0.25, 0.5\nmacs out_r, in_r, a, 0.5\nend"
    prog, img, orc, gpu = make_pair(fx, po, text, n, channels=2)
    try:
        for _ in range(2):
            x = (1.8 * rng.random((2, s, n)) - 0.9).astype(np.float32)
            yo = orc.process(x)
            d_in = torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 1))).cuda()      # [C][N][S]
            d_out = torch.empty_like(d_in)
            gpu.process_device_planar(d_in, d_out, s, None)
            gpu.synchronize(None)
            assert_bits_equal(d_out.cpu().numpy().transpose(0, 2, 1), yo, "planar outputs")
        compare_state(gpu, orc, img, "planar", (0, n - 1))
    finally:
        gpu.close()


@pytest.mark.parametrize("text", [progs.CFG2_LOG_GAIN, progs.CFG4_ONEPOLE, progs.cfg3_delay(100)])
def test_null_input_block_is_silence(fx, po, text):
    """process_batch with d_in == NULL: INPUT operands read 0.0 (every kernel family)."""
    import torch
    n, s = 96, 70
    prog, img, orc, gpu = make_pair(fx, po, text, n)
    try:
        x = (np.random.default_rng(61).random((1, s, n)) - 0.5).astype(np.float32)
        assert_bits_equal(gpu.process_host(x), orc.process(x), "warm-up block")
        d_out = torch.empty((1, s, n), dtype=torch.float32, device="cuda")
        gpu.process_device(None, d_out, s, None)
        gpu.synchronize(None)
        assert_bits_equal(d_out.cpu().numpy(), orc.process(np.zeros((1, s, n), np.float32)), "NULL input")
        compare_state(gpu, orc, img, "NULL input", (0, n - 1))
    finally:
        gpu.close()


@pytest.mark.parametrize("text", [
    # a TRAM that is only written, one that is only read (its ring comes from the checkpoint API), both in one program
    "static a\ninput in_l 0\noutput out_l 0\nitramsize 50 \nmacs a, in_l, 0.5, 0.5\nidelay write, a, at, 3\nmacs out_l, a, in_l, 0.25\nend",
    "static rd\ninput in_l 0\noutput out_l 0\nxtramsize 333 \nxdelay read, rd, at, 40\nmacs out_l, rd, in_l, 0.25\nend",
    "static a\nstatic rd\ninput in_l 0\noutput out_l 0\nitramsize 50 \nxtramsize 333 \nxdelay read, rd, at, 40\nmacs a, in_l, rd, 0.5\n"
    "idelay write, a, at, 3\nmacs out_l, a, in_l, 0.25\nend",
])
def test_tram_written_only_or_read_only(fx, po, text):
    rng = np.random.default_rng(71)
    n = 100
    prog, img, orc, gpu = make_pair(fx, po, text, n)
    try:
        d = gpu.dims()
        if d.xtram_size:
            for i in range(n):
                ring = (rng.random(d.xtram_size) - 0.5).astype(np.float32)
                gpu.set_tram(1, i, ring); orc.set_tram(1, i, ring)
        for s in (1, 90, 64, 500):
            x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
            assert_bits_equal(gpu.process_host(x), orc.process(x), "outputs")
        compare_state(gpu, orc, img, "one-sided TRAM", (0, 50, n - 1))
        assert gpu.launch_info().kernel_variant & 8
    finally:
        gpu.close()
