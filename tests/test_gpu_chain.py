"""Program chains on the GPU (fx8010_chain_*): every call is compared, bit for bit in the output and in every stage's whole final state,
with its definition — twin handles run one after another with fx8010_gpu_process_batch — and the fused calls also with the stages'
oracles on sampled instances.  Covers the fused kernel, the stage-by-stage path and the reason status gives for it, the mode-1
switch-over, invalidation of folded values, stream ordering, refused calls, and kernel sharing between chains."""
import importlib
import time

import numpy as np
import pytest

import chain_common as cc
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

    def definition(self, d_x, d_y, s, stream=None):
        t = [torch.empty_like(d_y) for _ in range(2)]
        cur = d_x
        for j, g in enumerate(self.twins):
            out = d_y if j + 1 == len(self.twins) else t[j & 1]
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


def run_and_compare(su, s, seed, what, d_x=None, expect_fused=None, tram=False):
    if d_x is None:
        d_x = input_block(su.ch, s, su.n, seed)
    d_y, d_r = torch.full_like(d_x, 7.0), torch.full_like(d_x, -7.0)
    su.chain.process_batch(d_x, d_y, s)
    su.definition(d_x, d_r, s)
    torch.cuda.synchronize()
    assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), what + " output")
    st = su.chain.status()
    if expect_fused is not None:
        assert st["fused_last"] == (1 if expect_fused else 0), (what, st)
    return d_x, d_y, st


def oracle_sampled(po, su, x, y, idx, what):
    """The stages' oracles, block after block (the definition), on the instances idx."""
    cur = np.ascontiguousarray(x[:, :, idx])
    for j, p in enumerate(su.progs):
        orc = po.Oracle(po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables()), len(idx), su.ch)
        for nm, v in su.ctl[j].items():
            orc.set_register(nm, v[idx])
        cur = orc.process(cur)
    assert_bits_equal(np.ascontiguousarray(y[:, :, idx]), cur, what + " against the oracle")


@pytest.mark.parametrize("s", [1024, 333])
@pytest.mark.parametrize("n", [4096, 65536])
@pytest.mark.parametrize("name", ["two", "three", "eight", "two_ch_two", "two_ch_eight"])
def test_fused_chain_matches_the_definition(po, name, n, s):
    texts, ch = cc.chain_texts(name)
    su = Setup(texts, ch, n)
    try:
        for b in range(2):
            d_x, d_y, st = run_and_compare(su, s, 100 + b, f"{name} N={n} S={s} block {b}", expect_fused=True)
            if b == 0:                                   # (the oracles start from a freshly loaded state)
                idx = np.random.default_rng(n + s).choice(n, 64, replace=False)
                oracle_sampled(po, su, d_x.cpu().numpy(), d_y.cpu().numpy(), idx, name)
        assert st["state"] == 2 and st["local_bytes"] == 0 and st["message"] == "", st
        assert st["launches"] == 2
        assert_same_state(su, name)
    finally:
        su.close()


@pytest.mark.parametrize("stateful", ["cfg4", "cfg3_1000", "cfg5"])
def test_stateful_stage_runs_stage_by_stage(stateful):
    text = {"cfg4": progs.CFG4_ONEPOLE, "cfg3_1000": progs.cfg3_delay(1000), "cfg5": progs.cfg5_allops()}[stateful]
    su = Setup([progs.CFG2_LOG_GAIN, text, cc.LIMIT], 1, 4096, relaxed=True)
    try:
        for b in range(3):
            _, _, st = run_and_compare(su, 256, b, f"{stateful} block {b}", expect_fused=False, tram=True)
        assert st["state"] == -1 and "stage 1 carries state across sample periods" in st["message"], st
        assert st["launches"] == 0
        assert_same_state(su, stateful, tram=True)
    finally:
        su.close()


@pytest.mark.parametrize("case", ["n_not_multiple_of_4", "unaligned", "mode_0"])
def test_unfusable_calls_run_stage_by_stage(case):
    n = 4094 if case == "n_not_multiple_of_4" else 4096
    texts, ch = cc.chain_texts("three")
    su = Setup(texts, ch, n, mode=0 if case == "mode_0" else 2)
    try:
        s = 200
        d_x = None
        if case == "unaligned":
            base = torch.zeros(s * n + 1, dtype=torch.float32, device="cuda")
            d_x = base[1:].view(1, s, n)
            d_x.copy_(input_block(1, s, n, 3))
        for b in range(2):
            _, _, st = run_and_compare(su, s, b, f"{case} block {b}", d_x=d_x, expect_fused=False)
        want = {"n_not_multiple_of_4": "multiple of 4", "unaligned": "16-byte aligned", "mode_0": "FX8010_OPT_TRANSLATE 0"}[case]
        assert want in st["message"], st
        assert_same_state(su, case)
    finally:
        su.close()


def test_mode_1_switches_over_with_identical_bits():
    texts = [progs.CFG2_LOG_GAIN, cc.LIMIT.replace("-0.5", "-0.4375")]        # (a source no other test compiles)
    su = Setup(texts, 1, 8192, mode=1)
    try:
        fused = []
        t0 = time.time()
        for b in range(400):
            _, _, st = run_and_compare(su, 128, b, f"mode 1 call {b}")
            fused.append(st["fused_last"])
            if st["fused_last"] and len(fused) > 2 and fused[-3:] == [1, 1, 1]:
                break
            if not st["fused_last"]:
                time.sleep(0.05)
            assert time.time() - t0 < 120, "the chain kernel never came"
        assert fused[0] == 0 and fused[-1] == 1 and fused == sorted(fused), fused
        assert_same_state(su, "mode 1")
    finally:
        su.close()


MIDDLE = "\n".join(["static k = 0.75", "input in_l 0", "output out_l 0", "macs out_l, 0, in_l, k", "end"])


def test_folded_register_and_reload_void_the_chain_kernel():
    su = Setup([progs.CFG2_LOG_GAIN, MIDDLE, cc.LIMIT], 1, 4096)
    try:
        run_and_compare(su, 64, 0, "before", expect_fused=True)
        assert "0x3f400000" in fx.translate_source_chain(su.progs)[0]           # k = 0.75 is an immediate
        c0 = fx.kernel_cache_stats()["nvrtc_compiles"]
        k = su.progs[1].reg_index("k")
        for g in (su.stages[1], su.twins[1]):
            g.set_controls(k, 0.3125, broadcast=True)
        run_and_compare(su, 64, 1, "after set_controls on a folded register", expect_fused=True)
        run_and_compare(su, 64, 2, "again", expect_fused=True)
        assert fx.kernel_cache_stats()["nvrtc_compiles"] == c0 + 1
        new = fx.Program(cc.LIMIT.replace("0.5", "0.375"))
        for g in (su.stages[2], su.twins[2]):
            g.load_program(new)
        su.progs[2] = new
        run_and_compare(su, 64, 3, "after load_program", expect_fused=True)
        assert fx.kernel_cache_stats()["nvrtc_compiles"] == c0 + 2
        su.stages[2].load_program(fx.Program(progs.CFG4_ONEPOLE)); su.twins[2].load_program(fx.Program(progs.CFG4_ONEPOLE))
        _, _, st = run_and_compare(su, 64, 4, "after loading a stateful program", expect_fused=False)
        assert "stage 2 carries state" in st["message"]
        assert_same_state(su, "invalidation")
    finally:
        su.close()


def test_stream_ordering():
    texts, ch = cc.chain_texts("three")
    n, s = 65536, 512
    su = Setup(texts, ch, n)
    other, other_twin = fx.Gpu(n, ch), fx.Gpu(n, ch)
    for g in (other, other_twin):
        g.load_program(fx.Program(progs.CFG2_LOG_GAIN)); g.set_option(fx.OPT_TRANSLATE, 0)
    s1, s2, s3 = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    try:
        d_a, d_x = input_block(ch, s, n, 1), input_block(ch, s, n, 2)
        junk = torch.empty_like(d_a)
        d_y, d_z, d_w = torch.empty_like(d_x), torch.empty_like(d_x), torch.empty_like(d_x)
        torch.cuda.synchronize()
        su.stages[0].process_device(d_a, junk, s, s1.cuda_stream)           # earlier work of stage 0 on another stream
        su.chain.process_batch(d_x, d_y, s, s2.cuda_stream)
        other.process_device(d_y, d_z, s, s2.cuda_stream)                   # the chain's output feeds another handle (same stream)
        su.stages[1].process_device(d_x, d_w, s, s3.cuda_stream)            # a plain call of a stage on a third stream
        torch.cuda.synchronize()
        assert su.chain.status()["fused_last"] == 1
        r_junk, r_y, r_z, r_w = (torch.empty_like(d_x) for _ in range(4))
        su.twins[0].process_device(d_a, r_junk, s)
        su.definition(d_x, r_y, s)
        other_twin.process_device(r_y, r_z, s)
        su.twins[1].process_device(d_x, r_w, s)
        torch.cuda.synchronize()
        for a, b, what in ((d_y, r_y, "chain output"), (d_z, r_z, "consumer output"), (d_w, r_w, "plain call after the chain")):
            assert_bits_equal(a.cpu().numpy(), b.cpu().numpy(), what)
        assert_same_state(su, "ordering")
    finally:
        su.close(); other.close(); other_twin.close()


def test_refused_calls_queue_nothing():
    texts, ch = cc.chain_texts("three")
    n = 4096
    su = Setup(texts, ch, n)
    empty = fx.Gpu(n, ch)
    try:
        d_x = input_block(ch, 16, n, 0)
        d_y = torch.empty_like(d_x)
        su.chain.process_batch(d_x, d_y, 16)
        torch.cuda.synchronize()
        before = [g.launch_info().kernel_launches for g in su.stages], su.chain.status()["launches"]
        for args, code in (((d_x, None, 16), 1), ((d_x, d_y, -1), 1), ((None, d_y, 16), 1)):
            with pytest.raises(fx.FxError) as e:
                su.chain.process_batch(*args)
            assert e.value.code == code
        c2 = fx.Chain([su.stages[0], empty])
        with pytest.raises(fx.FxError) as e:
            c2.process_batch(d_x, d_y, 16)
        assert e.value.code == 3
        c2.close()
        assert ([g.launch_info().kernel_launches for g in su.stages], su.chain.status()["launches"]) == before
        for bad in ([su.stages[0], su.stages[0]], [su.stages[0], fx.Gpu(n + 4, ch)], [su.stages[0], fx.Gpu(n, ch + 1)], [], su.stages * 3):
            with pytest.raises(fx.FxError) as e:
                fx.Chain(bad)
            assert e.value.code == 1
    finally:
        su.close(); empty.close()


def test_two_chains_share_one_compile():
    texts = [progs.CFG2_LOG_GAIN, cc.LIMIT.replace("-0.5", "-0.40625")]        # (a source no other test compiles)
    c0 = fx.kernel_cache_stats()["nvrtc_compiles"]
    a, b = Setup(texts, 1, 4096), Setup(texts, 1, 4096, seed=8)
    try:
        run_and_compare(a, 64, 0, "first chain", expect_fused=True)
        run_and_compare(b, 64, 1, "second chain", expect_fused=True)
        assert fx.kernel_cache_stats()["nvrtc_compiles"] == c0 + 1
    finally:
        a.close(); b.close()


def test_facade_chain():
    n, s = 4096, 128
    texts, ch = cc.chain_texts("three")
    objs = [fx.Program(t, channels=ch, instances=n) for t in texts]
    for o in objs:
        o.set_translation(2)
    pc = objs[0].chain(objs[1:])
    d_x = input_block(ch, s, n, 9)
    d_y, d_r = torch.empty_like(d_x), torch.empty_like(d_x)
    pc(d_x, d_y, s)
    twins = []
    cur = d_x
    for j, t in enumerate(texts):
        g = fx.Gpu(n, ch); g.load_program(objs[j]); g.set_option(fx.OPT_TRANSLATE, 0); twins.append(g)
        out = d_r if j + 1 == len(texts) else torch.empty_like(d_x)
        g.process_device(cur, out, s)
        cur = out
    torch.cuda.synchronize()
    assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), "facade chain")
    pc.close()
    for g in twins:
        g.close()
    if torch.cuda.device_count() >= 2:
        multi = fx.Program(texts[0], channels=ch, instances=n, devices=[0, 1])
        with pytest.raises(fx.FxError):
            multi.chain([objs[1]])
