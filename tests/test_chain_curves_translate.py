"""The fused kernel of a program chain with control curves (fx8010_translate_source_chain_curves), checked on the CPU: the generated source
compiled as plain C++ (-DFXT_HOST_CHECK), every (thread, time segment) work item in random order, against the stages' oracles stepped one
period at a time with every curve value of a stage set right before that stage's period — bit for bit in the outputs and in every stage's
registers, accumulator, latches, counters and run-time flags.  Also: NVRTC compiles the source for sm_100a, a chain with a stage that carries
state is declined, refused curve lists return -1, and a chain call without curves keeps the plain chain source."""
import ctypes
import importlib

import numpy as np
import pytest

import chain_common as cc
import chain_curves_common as ccc
import progs
from conftest import assert_bits_equal

fx = importlib.import_module("fx8010-emulator-core_b200")


def load(texts, ch):
    prog_list = [fx.Program(t, channels=ch) for t in texts]
    for p in prog_list:
        assert p.loaded, p.errors()
    return prog_list


def run_chain_curves(po, texts, ch, curves, n, blocks, seg_len, rng, inplace=False, what=""):
    prog_list = load(texts, ch)
    hc = ccc.HostChainCurves(prog_list, n, ch, curves)
    orcs = []
    for j, p in enumerate(prog_list):
        orc = po.Oracle(po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables()), n, ch)
        if j % 2 == 0:                      # per-instance controls on every other stage (the others fold their literals)
            for nm, v in cc.controls(p, n, rng).items():
                orc.set_register(nm, v)
                hc.stages[j].registers[p.reg_index(nm), :] = v
        orcs.append(orc)
    for b, s in enumerate(blocks):
        x = (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)
        values = ccc.curve_values(curves, s, n, rng)
        want = ccc.oracle_chain_curves_stepped(orcs, x, s, curves, values, n)
        got = hc.process_curves(x, values, seg_len=seg_len, seed=b, inplace=inplace)
        assert_bits_equal(got, want, f"{what} outputs of block {b}")
    for j, (orc, st) in enumerate(zip(orcs, hc.stages)):
        w = f"{what} stage {j}"
        assert_bits_equal(st.registers, orc.registers, w + " registers")
        assert_bits_equal(st.acc, orc.acc, w + " accumulator")
        assert_bits_equal(st.out_latch, orc.out_latch, w + " latches")
        assert_bits_equal(st.counts, orc.counts, w + " counters")
        assert int(st.flags[0]) == orc.flags, w + " run-time flags"
    for p in prog_list:
        p.close()
    return hc


@pytest.mark.parametrize("mix", ccc.MIXES)
@pytest.mark.parametrize("name", ["two", "three", "eight", "two_ch_two"])
def test_chain_curves_match_stages_stepped(po, name, mix):
    texts, ch = cc.chain_texts(name)
    curves = ccc.curve_mix(load(texts, ch), mix)
    hc = run_chain_curves(po, texts, ch, curves, 12, [37, 9, 1], 8, np.random.default_rng(7 + len(mix)), what=f"{name} {mix}")
    assert "FxtCurves" in hc.src and hc.src.count("FXT_DEV void fxt_period_s") == len(texts)
    if mix == "eight":
        assert len(curves) == 8


@pytest.mark.parametrize("seg_len", [4, 8, 64])
@pytest.mark.parametrize("inplace", [False, True], ids=["separate", "inplace"])
def test_segment_lengths_and_in_place(po, seg_len, inplace):
    """In place, the owner of the last period re-runs it from its input and that period's curve values."""
    texts, ch = cc.chain_texts("three")
    curves = ccc.curve_mix(load(texts, ch), "several")
    run_chain_curves(po, texts, ch, curves, 12, [37, 9, 1], seg_len, np.random.default_rng(seg_len), inplace=inplace, what=f"seg {seg_len}")


def test_curve_on_a_folded_static(po):
    """k = 0.75 is an immediate of the plain chain source; with a curve on it, the curve source reads it from the curve."""
    texts = [progs.CFG2_LOG_GAIN, ccc.MIDDLE, cc.LIMIT]
    prog_list = load(texts, 1)
    k = prog_list[1].reg_index("k")
    assert "0x3f400000" in fx.translate_source_chain(prog_list)[0]
    curves = [(1, k, False)]
    hc = run_chain_curves(po, texts, 1, curves, 16, [33, 7], 8, np.random.default_rng(3), what="folded static")
    assert "0x3f400000" not in hc.src
    run_chain_curves(po, texts, 1, [(1, k, True)], 16, [21], 4, np.random.default_rng(4), what="folded static, broadcast")


def test_curve_on_a_written_register_is_never_read():
    """A register its stage writes is overwritten before any read: no load for its curve."""
    texts, ch = cc.chain_texts("two")
    prog_list = load(texts, ch)
    a = prog_list[0].reg_index("a")                 # cfg2's LOG output
    assert a in ccc.written(prog_list[0])
    src, _ = fx.translate_source_chain_curves(prog_list, [(0, a, False)], ch, instances=4096)
    assert "FxtCurves" in src and "FXT_LOAD_CV" not in src


def test_without_curves_the_source_is_the_plain_chain_source():
    for name in cc.CHAINS:
        texts, ch = cc.chain_texts(name)
        prog_list = load(texts, ch)
        for n in (1, 4096, 65536):
            assert fx.translate_source_chain_curves(prog_list, [], ch, instances=n)[0] == fx.translate_source_chain(prog_list, ch, instances=n)[0]


@pytest.mark.parametrize("mix", ["several", "eight"])
def test_chain_curves_source_compiles_for_sm_100a(mix):
    texts, ch = cc.chain_texts("three")
    prog_list = load(texts, ch)
    src, cubin = fx.translate_source_chain_curves(prog_list, ccc.curve_mix(prog_list, mix), ch, compile_check=True, instances=65536)
    assert src is not None and "fx_translated_chain" in src
    if cubin == -1:
        pytest.skip("libnvrtc not loadable here")
    assert cubin > 1000


@pytest.mark.parametrize("stateful", ["cfg4", "cfg3", "cfg5"])
def test_chain_with_a_stateful_stage_is_declined(stateful):
    text = {"cfg4": progs.CFG4_ONEPOLE, "cfg3": progs.cfg3_delay(1000), "cfg5": progs.cfg5_allops()}[stateful]
    prog_list = [fx.Program(progs.CFG2_LOG_GAIN), fx.Program(text, relaxed=True)]
    assert all(p.loaded for p in prog_list)
    vol = prog_list[0].reg_index("volume")
    assert fx.translate_source_chain_curves(prog_list, [(0, vol, False)]) == (None, None)
    if stateful == "cfg4":
        cut = prog_list[1].reg_index("filter_cutoff")
        assert fx.translate_source_chain_curves(prog_list, [(1, cut, False)]) == (None, None)


def test_refused_curve_lists():
    texts, ch = cc.chain_texts("three")
    prog_list = load(texts, ch)
    vol = prog_list[1].reg_index("volume")
    in_l = prog_list[1].reg_index("in_l")
    bad = [[(3, vol, False)], [(-1, vol, False)], [(1, 999, False)], [(1, vol, False), (1, vol, True)], [(1, in_l, False)],
           [(1, vol, False)] * 9]
    for curves in bad:
        with pytest.raises(ValueError):
            fx.translate_source_chain_curves(prog_list, curves, ch)
    # the same register on two different stages is two curves
    assert fx.translate_source_chain_curves(prog_list, [(0, prog_list[0].reg_index("volume"), False), (1, vol, False)], ch)[0] is not None
    L = fx.gpu_lib()
    imgs = (ctypes.c_void_p * 3)(*[p.image_ptr() for p in prog_list])
    assert L.fx8010_translate_source_chain_curves(imgs, 3, 1, ch, None, None, None, 1, None, 0, 0, None) == -1
    assert L.fx8010_translate_source_chain_curves(imgs, 3, 1, ch, None, None, None, -1, None, 0, 0, None) == -1
    assert L.fx8010_chain_process_batch_curves(None, None, None, 1, None, 0, None) == 1
    assert L.fx8010_chain_status_curves(None, None, None, None, None, 0) == 1
