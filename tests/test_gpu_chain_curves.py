"""Control curves on program chains on the GPU (fx8010_chain_process_batch_curves): every call is compared, bit for bit in the output and
in every stage's whole final state, with its definition — twin handles run one after another, fx8010_gpu_process_batch_curves on each
stage with curves and fx8010_gpu_process_batch on the others — and the fused calls also with the stages' oracles stepped per period on
sampled instances.  Covers the fused kernel, the stage-by-stage path and its reasons, the mode-1 switch-over, interleaved plain and
automated calls (one compile per kernel), a folded STATIC that becomes automated, refused lists, in-place calls, stream ordering of a curve
produced by another handle, n_curves == 0, and the facade and its C view."""
import importlib
import time

import numpy as np
import pytest

import chain_common as cc
import chain_curves_common as ccc
import progs
from conftest import assert_bits_equal

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

fx = importlib.import_module("fx8010-emulator-core_b200")


class Setup:
    """Chain stages and their twins: the same programs and per-instance controls on separate handles."""

    def __init__(self, texts, ch, n, mode=2, twin_mode=0, seed=7, relaxed=False):
        self.n, self.ch, self.texts = n, ch, texts
        self.progs = [fx.Program(t, channels=ch, relaxed=relaxed) for t in texts]
        for p in self.progs:
            assert p.loaded, p.errors()
        rng = np.random.default_rng(seed)
        self.ctl = [cc.controls(p, n, rng) if j % 2 == 0 else {} for j, p in enumerate(self.progs)]
        self.stages = [self.handle(j, mode) for j in range(len(texts))]
        self.twins = [self.handle(j, twin_mode) for j in range(len(texts))]
        self.chain = fx.Chain(self.stages)

    def handle(self, j, mode):
        g = fx.Gpu(self.n, self.ch)
        g.load_program(self.progs[j])
        g.set_option(fx.OPT_TRANSLATE, mode)
        for nm, v in self.ctl[j].items():
            g.set_controls(self.progs[j].reg_index(nm), v)
        return g

    def definition(self, d_x, d_y, s, curves, d_vals, stream=None):
        """curves [(stage, reg, broadcast)], d_vals the device buffers: stage j runs process_batch_curves with its curves."""
        t = [torch.empty_like(d_y) for _ in range(2)]
        cur = d_x
        for j, g in enumerate(self.twins):
            out = d_y if j + 1 == len(self.twins) else t[j & 1]
            mine = [(reg, v, bc) for (st, reg, bc), v in zip(curves, d_vals) if st == j]
            if mine:
                g.process_device_curves(cur, out, s, mine, stream)
            else:
                g.process_device(cur, out, s, stream)
            cur = out
        return t

    def close(self):
        self.chain.close()
        for g in self.stages + self.twins:
            g.close()


def full_state(g, tram=False):
    acc, lfsr, latch, ptrs = g.scalars()
    out = {"registers": g.registers(), "acc": acc, "lfsr": lfsr, "latch": latch, "ptrs": ptrs, "counts": g.counts(), "flags": np.array([g.flags()])}
    if tram:
        d = g.dims()
        for which, size in ((0, d.itram_size), (1, d.xtram_size)):
            if size:
                out[f"tram{which}"] = np.stack([g.tram(which, i) for i in (0, g.n // 2, g.n - 1)])
    return out


def assert_same_state(su, what, tram=False):
    for j, (a, b) in enumerate(zip(su.stages, su.twins)):
        sa, sb = full_state(a, tram), full_state(b, tram)
        for k in sa:
            assert_bits_equal(sa[k], sb[k], f"{what}: stage {j} {k}")


def input_block(ch, s, n, seed):
    return torch.from_numpy((1.8 * np.random.default_rng(seed).random((ch, s, n)) - 0.9).astype(np.float32)).cuda()


def device_values(curves, s, n, seed):
    vals = ccc.curve_values(curves, s, n, np.random.default_rng(seed))
    return vals, [torch.from_numpy(v).cuda() for v in vals]


def run_and_compare(su, s, seed, curves, what, d_x=None, d_vals=None, expect_fused=None, tram=False, inplace=False):
    if d_x is None:
        d_x = input_block(su.ch, s, su.n, seed)
    vals = None
    if d_vals is None:
        vals, d_vals = device_values(curves, s, su.n, seed + 1000)
    d_r = torch.full_like(d_x, -7.0)
    su.definition(d_x, d_r, s, curves, d_vals)
    if inplace:
        d_y = d_x.clone()
        su.chain.process_batch_curves(d_y, d_y, s, [(st, reg, v, bc) for (st, reg, bc), v in zip(curves, d_vals)])
    else:
        d_y = torch.full_like(d_x, 7.0)
        su.chain.process_batch_curves(d_x, d_y, s, [(st, reg, v, bc) for (st, reg, bc), v in zip(curves, d_vals)])
    torch.cuda.synchronize()
    assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), what + " output")
    st = su.chain.status()
    if expect_fused is not None:
        assert st["fused_last"] == (1 if expect_fused else 0), (what, st)
    return d_x, d_y, vals, st


def oracle_sampled(po, su, x, y, curves, vals, idx, what):
    """The stages' oracles stepped per period with the curves (the definition), from a freshly loaded state, on the instances idx."""
    orcs = []
    for j, p in enumerate(su.progs):
        orc = po.Oracle(po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables()), len(idx), su.ch)
        for nm, v in su.ctl[j].items():
            orc.set_register(nm, v[idx])
        orcs.append(orc)
    sub = [v if bc else np.ascontiguousarray(v[:, idx]) for (_, _, bc), v in zip(curves, vals)]
    want = ccc.oracle_chain_curves_stepped(orcs, np.ascontiguousarray(x[:, :, idx]), x.shape[1], curves, sub, len(idx))
    assert_bits_equal(np.ascontiguousarray(y[:, :, idx]), want, what + " against the oracle")


@pytest.mark.parametrize("mix", ccc.MIXES)
@pytest.mark.parametrize("name", ["two", "three", "eight", "two_ch_two"])
def test_fused_curve_mixes(po, name, mix):
    texts, ch = cc.chain_texts(name)
    n, s = 4096, 333
    su = Setup(texts, ch, n)
    try:
        curves = ccc.curve_mix(su.progs, mix)
        for b in range(2):
            d_x, d_y, vals, st = run_and_compare(su, s, 100 + b, curves, f"{name} {mix} block {b}", expect_fused=True)
            if b == 0:
                idx = np.random.default_rng(n + s).choice(n, 64, replace=False)
                oracle_sampled(po, su, d_x.cpu().numpy(), d_y.cpu().numpy(), curves, vals, idx, f"{name} {mix}")
        cs = su.chain.status_curves()
        assert cs["state"] == 2 and cs["message"] == "", cs
        assert su.chain.status()["launches"] == 2
        assert_same_state(su, f"{name} {mix}")
    finally:
        su.close()


@pytest.mark.parametrize("s", [1024, 333])
@pytest.mark.parametrize("n", [4096, 65536])
@pytest.mark.parametrize("mix", ["several", "eight"])
def test_fused_sizes(po, mix, n, s):
    texts, ch = cc.chain_texts("three")
    su = Setup(texts, ch, n)
    try:
        curves = ccc.curve_mix(su.progs, mix)
        d_x, d_y, vals, st = run_and_compare(su, s, 7, curves, f"{mix} N={n} S={s}", expect_fused=True)
        idx = np.random.default_rng(n + s).choice(n, 64, replace=False)
        oracle_sampled(po, su, d_x.cpu().numpy(), d_y.cpu().numpy(), curves, vals, idx, f"{mix} N={n} S={s}")
        run_and_compare(su, s, 8, curves, f"{mix} N={n} S={s} second block", expect_fused=True)
        assert_same_state(su, f"{mix} N={n} S={s}")
    finally:
        su.close()


def test_cfg4_stage_runs_on_its_own_curve_kernel():
    su = Setup([progs.CFG2_LOG_GAIN, progs.CFG4_ONEPOLE], 1, 4096)
    try:
        cut = su.progs[1].reg_index("filter_cutoff")
        for b in range(2):
            _, _, _, st = run_and_compare(su, 256, b, [(1, cut, False)], f"cfg4 block {b}", expect_fused=False)
        assert "stage 1 carries state across sample periods" in st["message"], st
        assert st["launches"] == 0
        tc = su.stages[1].translate_status_curves()
        assert tc["state"] == 2 and tc["kind"] == 0, tc                      # the translated serial kernel with the curve
        assert su.stages[1].launch_info().kernel_variant & fx.VARIANT_CURVES
        assert_same_state(su, "cfg4")
    finally:
        su.close()


@pytest.mark.parametrize("case", ["cfg3", "n_not_multiple_of_4", "unaligned_curve", "mode_0"])
def test_unfusable_calls_run_stage_by_stage(case):
    n = 4094 if case == "n_not_multiple_of_4" else 4096
    texts = [progs.CFG2_LOG_GAIN, progs.cfg3_delay(1000), cc.LIMIT] if case == "cfg3" else cc.chain_texts("three")[0]
    su = Setup(texts, 1, n, mode=0 if case == "mode_0" else 2, relaxed=case == "cfg3")
    try:
        s = 200
        curves = [(0, su.progs[0].reg_index("volume"), False), (len(texts) - 1, su.progs[-1].reg_index("ceil"), True)]
        for b in range(2):
            _, d_vals = device_values(curves, s, n, b)
            if case == "unaligned_curve":
                base = torch.zeros(s * n + 1, dtype=torch.float32, device="cuda")
                base[1:].view(s, n).copy_(d_vals[0])
                d_vals[0] = base[1:].view(s, n)
            _, _, _, st = run_and_compare(su, s, b, curves, f"{case} block {b}", d_vals=d_vals, expect_fused=False, tram=case == "cfg3")
        want = {"cfg3": "stage 1 carries state across sample periods", "n_not_multiple_of_4": "multiple of 4",
                "unaligned_curve": "a curve buffer is not 16-byte aligned", "mode_0": "FX8010_OPT_TRANSLATE 0"}[case]
        assert want in st["message"], st
        assert_same_state(su, case, tram=case == "cfg3")
    finally:
        su.close()


def test_mode_1_switches_over_with_identical_bits():
    texts = [progs.CFG2_LOG_GAIN, cc.LIMIT.replace("-0.5", "-0.46875")]        # (a source no other test compiles)
    su = Setup(texts, 1, 8192, mode=1)
    try:
        curves = [(1, su.progs[1].reg_index("ceil"), False)]
        fused = []
        t0 = time.time()
        for b in range(400):
            _, _, _, st = run_and_compare(su, 128, b, curves, f"mode 1 call {b}")
            fused.append(st["fused_last"])
            if st["fused_last"] and len(fused) > 2 and fused[-3:] == [1, 1, 1]:
                break
            if not st["fused_last"]:
                assert "compiling" in st["message"], st
                time.sleep(0.05)
            assert time.time() - t0 < 120, "the chain kernel never came"
        assert fused[0] == 0 and fused[-1] == 1 and fused == sorted(fused), fused
        assert_same_state(su, "mode 1")
    finally:
        su.close()


def test_plain_and_automated_calls_interleave_with_one_compile_each():
    texts = [progs.CFG2_LOG_GAIN, cc.LIMIT.replace("-0.5", "-0.453125")]      # (a source no other test compiles)
    su = Setup(texts, 1, 4096)
    try:
        curves = [(0, su.progs[0].reg_index("volume"), False), (1, su.progs[1].reg_index("ceil"), True)]
        c0 = fx.kernel_cache_stats()["nvrtc_compiles"]
        d_x = input_block(1, 256, 4096, 0)
        d_y, d_r = torch.empty_like(d_x), torch.empty_like(d_x)
        su.chain.process_batch(d_x, d_y, 256)
        su.definition(d_x, d_r, 256, [], [])
        torch.cuda.synchronize()
        assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), "first plain call")
        run_and_compare(su, 256, 1, curves, "first automated call", expect_fused=True)
        c1 = fx.kernel_cache_stats()["nvrtc_compiles"]
        assert c1 <= c0 + 2
        for b in range(3):
            su.chain.process_batch(d_x, d_y, 256)
            su.definition(d_x, d_r, 256, [], [])
            torch.cuda.synchronize()
            assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), f"plain call {b}")
            assert su.chain.status()["fused_last"] == 1
            run_and_compare(su, 256, 10 + b, curves, f"automated call {b}", expect_fused=True)
        assert fx.kernel_cache_stats()["nvrtc_compiles"] == c1
        assert su.chain.status()["launches"] == 8
        assert_same_state(su, "interleaved")
    finally:
        su.close()


def test_folded_static_automated_regenerates_the_plain_kernel_once():
    su = Setup([progs.CFG2_LOG_GAIN, ccc.MIDDLE, cc.LIMIT.replace("-0.5", "-0.4375")], 1, 4096)
    try:
        k = su.progs[1].reg_index("k")
        d_x = input_block(1, 64, 4096, 0)
        d_y, d_r = torch.empty_like(d_x), torch.empty_like(d_x)

        def plain(b):
            su.chain.process_batch(d_x, d_y, 64)
            su.definition(d_x, d_r, 64, [], [])
            torch.cuda.synchronize()
            assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), f"plain call {b}")
            assert su.chain.status()["fused_last"] == 1

        plain(0)
        c0 = fx.kernel_cache_stats()["nvrtc_compiles"]
        run_and_compare(su, 64, 1, [(1, k, False)], "automated k", expect_fused=True)
        assert fx.kernel_cache_stats()["nvrtc_compiles"] == c0 + 1               # the curve kernel
        plain(1)                                                                # k is no longer one known value: the plain kernel once more
        assert fx.kernel_cache_stats()["nvrtc_compiles"] == c0 + 2
        for b in range(3):
            run_and_compare(su, 64, 2 + b, [(1, k, False)], f"automated k {b}", expect_fused=True)
            plain(2 + b)
        assert fx.kernel_cache_stats()["nvrtc_compiles"] == c0 + 2
        assert_same_state(su, "folded static")
    finally:
        su.close()


def test_refused_lists_change_nothing():
    texts, ch = cc.chain_texts("three")
    n, s = 4096, 16
    su = Setup(texts, ch, n)
    try:
        vol = su.progs[1].reg_index("volume")
        in_l = su.progs[1].reg_index("in_l")
        d_x = input_block(ch, s, n, 0)
        d_y = torch.empty_like(d_x)
        d_v = torch.rand(s, n, device="cuda")
        su.chain.process_batch(d_x, d_y, s)
        torch.cuda.synchronize()
        d_y.fill_(3.0)
        before = ([g.launch_info().kernel_launches for g in su.stages], su.chain.status()["launches"], [full_state(g) for g in su.stages])
        bad = [[(3, vol, d_v, False)], [(-1, vol, d_v, False)], [(1, 999, d_v, False)], [(1, vol, d_v, False), (1, vol, d_v, True)],
               [(1, in_l, d_v, False)], [(1, vol, None, False)], [(1, vol, d_v, False)] * 9,
               [(0, su.progs[0].reg_index("volume"), d_v, False), (2, 999, d_v, False)]]     # stage 0 is fine, stage 2 is not
        for curves in bad:
            with pytest.raises(fx.FxError) as e:
                su.chain.process_batch_curves(d_x, d_y, s, curves)
            assert e.value.code == 1, curves
        L = fx.gpu_lib()
        assert L.fx8010_chain_process_batch_curves(su.chain.h, d_x.data_ptr(), d_y.data_ptr(), s, None, 1, None) == 1
        assert L.fx8010_chain_process_batch_curves(su.chain.h, d_x.data_ptr(), d_y.data_ptr(), s, None, -1, None) == 1
        torch.cuda.synchronize()
        after = ([g.launch_info().kernel_launches for g in su.stages], su.chain.status()["launches"], [full_state(g) for g in su.stages])
        assert after[:2] == before[:2]
        for j, (a, b) in enumerate(zip(before[2], after[2])):
            for key in a:
                assert_bits_equal(a[key], b[key], f"stage {j} {key} after refused lists")
        assert bool((d_y == 3.0).all()), "the output buffer was written"
    finally:
        su.close()


def test_in_place_with_curves():
    texts, ch = cc.chain_texts("two_ch_two")
    su = Setup(texts, ch, 4096)
    try:
        curves = ccc.curve_mix(su.progs, "eight")
        for b in range(2):
            run_and_compare(su, 333, b, curves, f"in place block {b}", expect_fused=True, inplace=True)
        assert_same_state(su, "in place")
    finally:
        su.close()


def test_curve_written_by_another_handle_on_a_second_stream():
    """The curve is another handle's output, queued on stream 1 after earlier work of stage 0 there; the chain call on stream 2 reads it
    after that work."""
    texts, ch = cc.chain_texts("three")
    n, s = 65536, 256
    su = Setup(texts, ch, n)
    producer = fx.Gpu(n, 1)
    producer.load_program(fx.Program(progs.CFG2_LOG_GAIN)); producer.set_option(fx.OPT_TRANSLATE, 2)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    try:
        curves = [(1, su.progs[1].reg_index("volume"), False)]
        d_a, d_x, d_p = input_block(ch, s, n, 1), input_block(ch, s, n, 2), input_block(1, s, n, 3)
        junk, d_v, d_y = torch.empty_like(d_a), torch.empty((s, n), device="cuda"), torch.empty_like(d_x)
        torch.cuda.synchronize()
        with torch.cuda.stream(s1):
            su.stages[0].process_device(d_a, junk, s, s1.cuda_stream)
            torch.cuda._sleep(20_000_000)                    # keep stream 1 busy: the chain call on stream 2 must still come after
            producer.process_device(d_p, d_v, s, s1.cuda_stream)
        su.chain.process_batch_curves(d_x, d_y, s, [(1, curves[0][1], d_v, False)], s2.cuda_stream)
        torch.cuda.synchronize()
        assert su.chain.status()["fused_last"] == 1
        r_junk, d_r = torch.empty_like(d_a), torch.empty_like(d_x)
        su.twins[0].process_device(d_a, r_junk, s)
        su.definition(d_x, d_r, s, curves, [d_v])
        torch.cuda.synchronize()
        assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), "chain output with a curve from another stream")
        assert_same_state(su, "second stream")
    finally:
        su.close(); producer.close()


def test_no_curves_is_the_plain_call():
    texts, ch = cc.chain_texts("three")
    su = Setup(texts, ch, 4096)
    try:
        d_x = input_block(ch, 128, 4096, 0)
        d_y, d_r = torch.empty_like(d_x), torch.empty_like(d_x)
        su.chain.process_batch_curves(d_x, d_y, 128, [])
        su.definition(d_x, d_r, 128, [], [])
        torch.cuda.synchronize()
        assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), "n_curves == 0")
        assert su.chain.status()["fused_last"] == 1 and su.chain.status_curves()["state"] == 0
        assert_same_state(su, "no curves")
    finally:
        su.close()


def test_facade_chain_with_curves_by_name():
    n, s = 4096, 128
    texts, ch = cc.chain_texts("three")
    objs = [fx.Program(t, channels=ch, instances=n) for t in texts]
    for o in objs:
        o.set_translation(2)
    pc = objs[0].chain(objs[1:])
    d_x = input_block(ch, s, n, 9)
    d_y, d_r = torch.empty_like(d_x), torch.empty_like(d_x)
    vals, d_vals = device_values([(0, 0, False), (2, 0, True)], s, n, 5)
    pc.process_curves(d_x, d_y, s, [(0, "volume", d_vals[0], False), (2, "ceil", d_vals[1], True)])
    twins = []
    cur = d_x
    for j, t in enumerate(texts):
        g = fx.Gpu(n, ch); g.load_program(objs[j]); g.set_option(fx.OPT_TRANSLATE, 0); twins.append(g)
        out = d_r if j + 1 == len(texts) else torch.empty_like(d_x)
        if j == 0:
            g.process_device_curves(cur, out, s, [(objs[0].reg_index("volume"), d_vals[0], False)])
        elif j == 2:
            g.process_device_curves(cur, out, s, [(objs[2].reg_index("ceil"), d_vals[1], True)])
        else:
            g.process_device(cur, out, s)
        cur = out
    torch.cuda.synchronize()
    assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), "facade chain with curves")
    for bad in ([(3, "volume", d_vals[0], False)], [(1, "no_such_register", d_vals[0], False)]):
        with pytest.raises(fx.FxError):
            pc.process_curves(d_x, d_y, s, bad)
    pc.close()
    for g in twins:
        g.close()
