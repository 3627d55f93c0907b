"""Edge cases of program chains (fx8010_chain_*) on the GPU.  Every call is compared with the chain's definition — twin handles called one
after another — bit for bit in the output and in every stage's whole final state, and every call asserts which path ran it (fused_last).
Shapes around the launch geometry (partial warps and thread blocks, FXT_U groups and time-segment boundaries, the segment-count cap, forced
geometries), seeded random chains, a NULL input, pass-through latches, more tables than shared-memory slots, edge input samples, edits and
plain calls between chain calls, in-place calls, and the ordering of the stage-by-stage path when every stage is STREAM_EXCLUSIVE."""
import importlib

import numpy as np
import pytest

import chain_common as cc
import progs
from conftest import assert_bits_equal
from test_gpu_chain import Setup, assert_same_state, input_block, run_and_compare

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

fx = importlib.import_module("fx8010-emulator-core_b200")


def calls(su, blocks, what, fused, seed=0):
    for b, s in enumerate(blocks):
        run_and_compare(su, s, seed + b, f"{what} call {b} (S={s})", expect_fused=fused)
    assert_same_state(su, what)


@pytest.mark.parametrize("s", [1, 2, 3, 4, 5, 7, 8, 9, 31, 33, 4097])
@pytest.mark.parametrize("n", [4, 8, 12, 132, 4100])
def test_shapes(n, s):
    """Partial warps and thread blocks (N), FXT_U groups and time-segment boundaries (S); two calls each, so that the second starts from
    the state the first left."""
    texts, ch = cc.chain_texts("three")
    su = Setup(texts, ch, n)
    try:
        calls(su, [s, s], f"N={n} S={s}", True)
    finally:
        su.close()


def test_segment_count_cap(monkeypatch):
    """N = 4, S = 600 000 at 4 periods per segment: 150 000 segments exceed the grid's 65 535, so sl_segments doubles seg_len twice."""
    monkeypatch.setenv("FX8010_TUNE_SEGLEN", "4")
    texts, ch = cc.chain_texts("two")
    su = Setup(texts, ch, 4)
    try:
        calls(su, [600000, 7], "segment cap", True)
    finally:
        su.close()


@pytest.mark.parametrize("env,value", [("FX8010_TUNE_SEGLEN", v) for v in ("4", "8", "64")] + [("FX8010_TUNE_B", v) for v in ("32", "64", "256")] +
                                      [("FX8010_TR_U", v) for v in ("1", "2", "8")])
def test_forced_geometry(env, value, monkeypatch):
    monkeypatch.setenv(env, value)
    texts, ch = cc.chain_texts("two_ch_three")
    su = Setup(texts, ch, 4100)
    try:
        if env == "FX8010_TR_U":
            assert f"#define FXT_U {value}\n" in fx.translate_source_chain(su.progs, ch, instances=4100)[0]
        calls(su, [333, 1, 64], f"{env}={value}", True)
    finally:
        su.close()


@pytest.mark.parametrize("seed", range(16))
def test_random_chains(seed):
    """2 to 8 stages of seeded random stateless programs, one or two channels."""
    rng = np.random.default_rng(700 + seed)
    ch = 1 + seed % 2
    texts = [cc.random_stateless(40 + 10 * seed + j, channels=ch) for j in range(2 + seed % 7)]
    su = Setup(texts, ch, 4096, seed=seed)
    try:
        calls(su, [int(rng.integers(1, 300)), 1, 96], f"random chain {seed}", True, seed=seed)
    finally:
        su.close()


NO_INPUT = "\n".join(["static a", "control g = 0.5", "output out_l 0", "macs a, 0.25, g, 0.125", "macs out_l, 0, a, 0.5", "end"])


@pytest.mark.parametrize("n,fused", [(4096, True), (4094, False)])
def test_null_input(n, fused):
    """Stage 0 reads no input: d_in = NULL on the fused and on the stage-by-stage path."""
    su = Setup([NO_INPUT, progs.CFG1A_TESTCODE, cc.LIMIT], 1, n)
    try:
        for b, s in enumerate([100, 1, 33]):
            d_y, d_r = torch.full((1, s, n), 7.0, device="cuda"), torch.full((1, s, n), -7.0, device="cuda")
            su.chain.process_batch(None, d_y, s)
            su.definition(None, d_r, s)
            torch.cuda.synchronize()
            assert su.chain.status()["fused_last"] == int(fused)
            assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), f"NULL input call {b}")
        assert_same_state(su, "NULL input")
    finally:
        su.close()


# two channels; never writes output channel 1, so that channel's latch passes the value it held through
LEFT_ONLY = "\n".join(["input in_l 0", "input in_r 1", "output out_l 0", "output out_r 1", "macs out_l, in_l, in_r, 0.5", "end"])
# the input-index quirk: X and Y operands of INPUT type read A's channel (test_gpu_parity.py::test_two_channels_input_index_quirk)
QUIRK = "static a\ninput in_l 0\ninput in_r 1\noutput out_l 0\noutput out_r 1\nmacs out_r, 0, in_r, 1.0\nmacs out_l, in_r, in_l, 0.5\nmacs a, 0.1, 0.5, in_r\nend"
QUIRK_GENERIC = "input in_l 0\ninput in_r 1\noutput out_l 0\noutput out_r 1\nmacs out_l, in_l, in_r, 0.5\nmacs out_r, 0.25, in_r, in_l\nend"


@pytest.mark.parametrize("middle", ["left_only", "quirk", "quirk_generic"])
def test_latches_and_channels(middle):
    """A two-channel middle stage: one that leaves output channel 1 alone, and the two programs of the input-index quirk."""
    text = {"left_only": LEFT_ONLY, "quirk": QUIRK, "quirk_generic": QUIRK_GENERIC}[middle]
    su = Setup([cc.TWO_CH_GAIN, text, cc.TWO_CH_MIX], 2, 4096)
    try:
        calls(su, [77, 1, 200], middle, True)
    finally:
        su.close()


def test_more_tables_than_shared_memory_slots():
    """Six distinct (stage, literal selector) LOG / EXP tables: four in shared memory, the others read through L1; and a stage whose
    selector is a control (per instance)."""
    stage = lambda a, b: f"static t\ninput in_l 0\noutput out_l 0\nlog t, in_l, {a}, 0\nexp out_l, t, {b}, 0\nend"
    dyn = "static a\ninput in_l 0\ncontrol sel = 3\noutput out_l 0\nlog a, in_l, sel, 0\nmacs out_l, 0, a, 0.5\nend"
    texts = [stage(1, 2), dyn, stage(3, 4), stage(5, 6)]
    su = Setup(texts, 1, 4096)
    try:
        v = np.random.default_rng(3).integers(0, 32, 4096).astype(np.float32)
        for g in (su.stages[1], su.twins[1]):
            g.set_controls(su.progs[1].reg_index("sel"), v)
        assert "#define FXT_NT 4\n" in fx.translate_source_chain(su.progs, 1, instances=4096)[0]
        calls(su, [300, 1, 64], "table slots", True)
    finally:
        su.close()


def test_edge_input_samples():
    """Signed zeros, subnormals, the largest value below 1, large finite values and the table-edge bit patterns (NaN included) as inputs,
    against the twins only (NaN payloads are the device's on both sides)."""
    n, s = 4096, 16
    edge = np.array([0.0, -0.0, 1e-45, -1e-45, 1.1754942e-38, -1.1754942e-38, 0.99999994, -0.99999994, 1.0, -1.0, 3.4e38, -3.4e38, 65504.0],
                    np.float32)
    vals = np.concatenate([edge, np.asarray(progs.TABLE_EDGE_BITS, np.uint32).view(np.float32)])
    x = np.resize(vals, (1, s, n)).astype(np.float32)
    for name in ("three", "eight"):
        texts, ch = cc.chain_texts(name)
        su = Setup(texts, ch, n)
        try:
            d_x = torch.from_numpy(x).cuda()
            run_and_compare(su, s, 0, f"{name} edge inputs", d_x=d_x, expect_fused=True)
            run_and_compare(su, s, 0, f"{name} edge inputs again", d_x=d_x, expect_fused=True)
            assert_same_state(su, f"{name} edge inputs")
        finally:
            su.close()


def test_edits_and_plain_calls_between_chain_calls():
    """set_controls per instance on a middle stage's non-folded control, set_controls_device on another stream, plain process_batch calls
    of single stages, and a trace of a stage, each between fused chain calls."""
    texts, ch = cc.chain_texts("eight")
    n, s = 4096, 96
    su = Setup(texts, ch, n)
    rng = np.random.default_rng(17)
    other = torch.cuda.Stream()
    try:
        run_and_compare(su, s, 0, "first", expect_fused=True)
        vol = su.progs[2].reg_index("volume")
        v = rng.random(n).astype(np.float32)
        for g in (su.stages[2], su.twins[2]):
            g.set_controls(vol, v)
        run_and_compare(su, s, 1, "after set_controls on stage 2", expect_fused=True)
        d_v = torch.from_numpy(rng.random(n).astype(np.float32)).cuda()
        torch.cuda.synchronize()
        for g in (su.stages[2], su.twins[2]):
            g.set_controls_device(vol, d_v, other.cuda_stream)
        other.synchronize()
        run_and_compare(su, s, 2, "after set_controls_device on another stream", expect_fused=True)
        for j in (0, 3, 7):
            d_x = input_block(ch, 40, n, 50 + j)
            d_a, d_b = torch.empty_like(d_x), torch.empty_like(d_x)
            su.stages[j].process_device(d_x, d_a, 40)
            su.twins[j].process_device(d_x, d_b, 40)
            torch.cuda.synchronize()
            assert_bits_equal(d_a.cpu().numpy(), d_b.cpu().numpy(), f"plain call of stage {j}")
            run_and_compare(su, s, 3 + j, f"after a plain call of stage {j}", expect_fused=True)
        xt = (1.8 * rng.random((ch, 20, n)) - 0.9).astype(np.float32)
        ya, _ = su.stages[4].trace(xt, 5)
        yb, _ = su.twins[4].trace(xt, 5)
        assert_bits_equal(ya, yb, "trace of stage 4")
        run_and_compare(su, s, 20, "after a trace", expect_fused=True)
        assert_same_state(su, "edits between calls")
    finally:
        su.close()


def test_one_handle_in_two_chains():
    """Stage 0 of chain A is also stage 1 of chain B; the chains are called alternately."""
    n, s = 4096, 64
    su = Setup([progs.CFG2_LOG_GAIN, cc.LIMIT, progs.CFG1A_TESTCODE, progs.CFG1B_LOGTUBE], 1, n)
    a_st, b_st = [su.stages[0], su.stages[1]], [su.stages[2], su.stages[0], su.stages[3]]
    a_tw, b_tw = [su.twins[0], su.twins[1]], [su.twins[2], su.twins[0], su.twins[3]]
    ca, cb = fx.Chain(a_st), fx.Chain(b_st)
    try:
        for k in range(4):
            for c, tw, name in ((ca, a_tw, "A"), (cb, b_tw, "B")):
                d_x = input_block(1, s, n, 10 * k + len(name))
                d_y, d_r = torch.empty_like(d_x), torch.empty_like(d_x)
                c.process_batch(d_x, d_y, s)
                cur = d_x
                for j, g in enumerate(tw):
                    out = d_r if j + 1 == len(tw) else torch.empty_like(d_x)
                    g.process_device(cur, out, s)
                    cur = out
                torch.cuda.synchronize()
                assert c.status()["fused_last"] == 1, (name, c.status())
                assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), f"chain {name} call {k}")
        assert_same_state(su, "one handle in two chains")
    finally:
        ca.close(); cb.close(); su.close()


@pytest.mark.parametrize("n,fused", [(4096, True), (4094, False)])
def test_in_place(n, fused):
    """d_out == d_in, on the fused and on the stage-by-stage path."""
    for name in ("three", "two_ch_eight"):
        texts, ch = cc.chain_texts(name)
        su = Setup(texts, ch, n)
        try:
            for b, s in enumerate([300, 1, 37]):
                d_io = input_block(ch, s, n, b)
                d_x, d_r = d_io.clone(), torch.empty_like(d_io)
                su.chain.process_batch(d_io, d_io, s)
                su.definition(d_x, d_r, s)
                torch.cuda.synchronize()
                assert su.chain.status()["fused_last"] == int(fused)
                assert_bits_equal(d_io.cpu().numpy(), d_r.cpu().numpy(), f"{name} N={n} in place call {b}")
            assert_same_state(su, f"{name} N={n} in place")
        finally:
            su.close()


def test_stream_exclusive_stages_wait_for_the_stage_before():
    """Every stage STREAM_EXCLUSIVE, N = 4 094 and mode 0 (the stage-by-stage path), three rotating output buffers over 9 calls.  The last
    stage reads the same intermediate block every call and writes a new buffer, so its own launches alone would let it postpone its wait
    and read that block while the stage before still writes it: a chain's stage launches must wait at their start."""
    n, s = 4094, 256
    texts, ch = cc.chain_texts("three")
    su = Setup(texts, ch, n, mode=0)
    try:
        for g in su.stages:
            g.set_option(fx.OPT_STREAM_EXCLUSIVE, 1)
        d_x = input_block(ch, s, n, 1)
        outs = [torch.full_like(d_x, 7.0) for _ in range(3)]
        refs = [torch.full_like(d_x, -7.0) for _ in range(3)]
        torch.cuda.synchronize()
        for k in range(9):
            su.chain.process_batch(d_x, outs[k % 3], s)
            assert su.chain.status()["fused_last"] == 0
            assert [g.launch_info().last_late_wait for g in su.stages] == [0] * len(su.stages), (k, [g.launch_info().last_late_wait for g in su.stages])
        for k in range(9):
            su.definition(d_x, refs[k % 3], s)
        torch.cuda.synchronize()
        for b in range(3):
            assert_bits_equal(outs[b].cpu().numpy(), refs[b].cpu().numpy(), f"rotating buffer {b}")
        assert_same_state(su, "stream exclusive")
    finally:
        su.close()
