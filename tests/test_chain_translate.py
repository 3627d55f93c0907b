"""The fused kernel of a program chain (fx8010_translate_source_chain), checked on the CPU: the generated source compiled as plain C++
(-DFXT_HOST_CHECK) against the stages' oracles stepped one period at a time, stage after stage, bit for bit in the outputs and in every
stage's registers, accumulator, latches, counters and run-time flags.  Also: NVRTC compiles the source for sm_100a, a chain with a stage
that carries state is declined, and fx8010_chain_create refuses malformed stage lists before it touches a device."""
import ctypes
import importlib

import numpy as np
import pytest

import chain_common as cc
import progs
from conftest import assert_bits_equal
from chain_host import HostChain

fx = importlib.import_module("fx8010-emulator-core_b200")


def run_chain(po, name, n, blocks, seg_len, rng, no_input=False, inplace=False):
    texts, ch = cc.chain_texts(name)
    prog_list = [fx.Program(t, channels=ch) for t in texts]
    for p in prog_list:
        assert p.loaded, p.errors()
    hc = HostChain(prog_list, n, ch)
    orcs = []
    for j, p in enumerate(prog_list):
        orc = po.Oracle(po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables()), n, ch)
        if j % 2 == 0:                      # per-instance controls on every other stage (the others fold their literals)
            for nm, v in cc.controls(p, n, rng).items():
                orc.set_register(nm, v)
                hc.stages[j].registers[p.reg_index(nm), :] = v
        orcs.append(orc)
    start = 0
    for b, s in enumerate(blocks):
        x = None if no_input else (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)
        want = cc.oracle_chain_stepped(orcs, x, s)
        got = hc.process(x, s, seg_len=seg_len, seed=b, inplace=inplace)
        assert_bits_equal(got, want, f"{name} outputs of block at {start}")
        start += s
    for j, (orc, st) in enumerate(zip(orcs, hc.stages)):
        what = f"{name} stage {j}"
        assert_bits_equal(st.registers, orc.registers, what + " registers")
        assert_bits_equal(st.acc, orc.acc, what + " accumulator")
        assert_bits_equal(st.out_latch, orc.out_latch, what + " latches")
        assert_bits_equal(st.counts, orc.counts, what + " counters")
        assert int(st.flags[0]) == orc.flags, what + " run-time flags"
    for p in prog_list:
        p.close()
    return hc


@pytest.mark.parametrize("name,seg_len,inplace", [pytest.param(nm, sl, ip, id=f"{nm}-{sl}" + ("-inplace" if ip else ""))
                                                  for ip in (False, True) for nm in cc.CHAINS for sl in (4, 8, 64)])
def test_chain_matches_stages_one_after_another(po, name, seg_len, inplace):
    """In place (d_out == d_in), the owner of the last period must re-run it through every stage from its input, not from the output it
    has just stored there."""
    rng = np.random.default_rng(31 + seg_len)
    hc = run_chain(po, name, 12, [37, 9, 1], seg_len, rng, inplace=inplace)
    assert "fx_translated_chain" in hc.src and hc.src.count("FXT_DEV void fxt_period_s") == len(hc.stages)


def test_chain_without_input(po):
    """A NULL input is zeros for stage 0 (its program still runs every period)."""
    run_chain(po, "three", 8, [13], 4, np.random.default_rng(5), no_input=True)


def test_table_range_flags_per_stage(po):
    """LOG inputs outside [-1, 1] in a middle stage raise that stage's flag only (stage 0 outputs 2 for every input >= 0)."""
    gain = "\n".join(["input in_l 0", "output out_l 0", "limit out_l, in_l, 2, 0", "end"])          # 2 for inputs >= 0, else 0
    texts = [gain, progs.CFG2_LOG_GAIN, cc.LIMIT]
    prog_list = [fx.Program(t) for t in texts]
    assert all(p.loaded for p in prog_list), [p.errors() for p in prog_list]
    n, s = 8, 21
    hc = HostChain(prog_list, n)
    orcs = [po.Oracle(po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables()), n, 1) for p in prog_list]
    x = (1.8 * np.random.default_rng(2).random((1, s, n)) - 0.9).astype(np.float32)
    assert_bits_equal(hc.process(x, s, seg_len=8), cc.oracle_chain_stepped(orcs, x, s), "outputs")
    assert [int(st.flags[0]) for st in hc.stages] == [o.flags for o in orcs]
    assert orcs[1].flags & fx.RT_TABLE_RANGE


@pytest.mark.parametrize("name", ["three", "two_ch_eight"])
def test_chain_source_compiles_for_sm_100a(name):
    texts, ch = cc.chain_texts(name)
    prog_list = [fx.Program(t, channels=ch) for t in texts]
    src, cubin = fx.translate_source_chain(prog_list, ch, compile_check=True, instances=4096)
    assert src is not None and "fx_translated_chain" in src
    if cubin == -1:
        pytest.skip("libnvrtc not loadable here")
    assert cubin > 1000


@pytest.mark.parametrize("stateful", ["cfg4", "cfg3", "cfg5"])
def test_chain_with_a_stateful_stage_is_declined(stateful):
    text = {"cfg4": progs.CFG4_ONEPOLE, "cfg3": progs.cfg3_delay(1000), "cfg5": progs.cfg5_allops()}[stateful]
    prog_list = [fx.Program(progs.CFG2_LOG_GAIN), fx.Program(text, relaxed=True)]
    assert all(p.loaded for p in prog_list)
    assert fx.translate_source_chain(prog_list) == (None, None)
    assert fx.translate_source_chain(prog_list[:1])[0] is not None
    with pytest.raises(ValueError):
        fx.translate_source_chain([])


def test_chain_create_refuses_bad_stage_lists():
    """Checked before any device is touched: a count outside 1..8, a NULL stage."""
    L = fx.gpu_lib()
    out = ctypes.c_void_p(1)
    for arr, n in [((ctypes.c_void_p * 1)(None), 0), ((ctypes.c_void_p * 9)(*([None] * 9)), 9), ((ctypes.c_void_p * 2)(None, None), 2)]:
        assert L.fx8010_chain_create(arr, n, ctypes.byref(out)) == 1
        assert out.value is None
        assert L.fx8010_chain_last_error(None)
    assert L.fx8010_chain_create(None, 1, ctypes.byref(out)) == 1
    assert L.fx8010_chain_process_batch(None, None, None, 1, None) == 1
    assert L.fx8010_chain_status(None, None, None, None, None, None, None, 0) == 1
