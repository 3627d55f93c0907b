"""Program chains from host memory on the GPU (fx8010_chain_process_batch_host(_curves), fx8010_multi_chain_*, FX8010Chain::processBlock).
Every call is compared, bit for bit in the output and in every stage's whole final state, with its definition — twin stages running the
device chain call on device copies of the same buffers — and on sampled instances with the stages' oracles stepped per period.  Each case
asserts whether its sub-blocks ran fused (fx8010_chain_status).  Covers fused and stage-by-stage chains over N x S x FX8010_TUNE_SUB,
page-locked asynchronous calls in a row, in-place and slice calls, curves, refused lists, mode 0 and the mode-1 switch-over inside one call,
interleaving with the stages' own calls, executor chains (two shards on one ordinal, uneven shards, refusals, create checks, cfg4 at the
bench geometry, two GPUs) and the facade on one device and on several."""
import ctypes as C
import importlib

import numpy as np
import pytest

import chain_common as cc
import chain_curves_common as ccc
import progs
from conftest import assert_bits_equal

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

fx = importlib.import_module("fx8010-emulator-core_b200")


def chain_texts(name):
    """The chains of tests/chain_common.py plus the stage-by-stage ones: stage texts, channels, whether the chain runs fused."""
    if name == "cfg4_cfg2":
        return [progs.CFG4_ONEPOLE, progs.CFG2_LOG_GAIN], 1, False
    if name == "cfg2_cfg3":
        return [progs.CFG2_LOG_GAIN, progs.cfg3_delay(100)], 1, False
    if name == "cfg5":
        return [progs.CFG2_LOG_GAIN, progs.cfg5_allops(64), cc.LIMIT], 1, False
    texts, ch = cc.chain_texts(name)
    return texts, ch, True


class Setup:
    """Chain stages and their twins: the same programs and per-instance controls on separate handles, each set in a chain."""

    def __init__(self, texts, ch, n, mode=2, twin_mode=2, seed=7):
        self.n, self.ch = n, ch
        self.progs = [fx.Program(t, channels=ch) for t in texts]
        for p in self.progs:
            assert p.loaded, p.errors()
        rng = np.random.default_rng(seed)
        self.ctl = [cc.controls(p, n, rng) if j % 2 == 0 else {} for j, p in enumerate(self.progs)]
        self.stages = [self.handle(j, mode) for j in range(len(texts))]
        self.twins = [self.handle(j, twin_mode) for j in range(len(texts))]
        self.chain = fx.Chain(self.stages)
        self.twin_chain = fx.Chain(self.twins)

    def handle(self, j, mode):
        g = fx.Gpu(self.n, self.ch)
        g.load_program(self.progs[j])
        g.set_option(fx.OPT_TRANSLATE, mode)
        for nm, v in self.ctl[j].items():
            g.set_controls(self.progs[j].reg_index(nm), v)
        return g

    def definition(self, x, s, curves=(), vals=()):
        """The twins' device chain call on device copies of x and the curve values; returns the output on the host."""
        d_x = None if x is None else torch.from_numpy(np.ascontiguousarray(x)).cuda()
        d_y = torch.full((self.ch, s, self.n), -7.0, device="cuda")
        if curves:
            d_vals = [torch.from_numpy(np.ascontiguousarray(v)).cuda() for v in vals]
            self.twin_chain.process_batch_curves(d_x, d_y, s, [(st, reg, v, bc) for (st, reg, bc), v in zip(curves, d_vals)])
        else:
            self.twin_chain.process_batch(d_x, d_y, s)
        torch.cuda.synchronize()
        return d_y.cpu().numpy()

    def close(self):
        self.chain.close(); self.twin_chain.close()
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


def assert_same_state(su, what, tram=True):
    for j, (a, b) in enumerate(zip(su.stages, su.twins)):
        sa, sb = full_state(a, tram), full_state(b, tram)
        for k in sa:
            assert_bits_equal(sa[k], sb[k], f"{what}: stage {j} {k}")


def input_block(ch, s, n, seed):
    return (1.8 * np.random.default_rng(seed).random((ch, s, n)) - 0.9).astype(np.float32)


def oracle_sampled(po, su, x, y, what, curves=(), vals=(), n_idx=48, seed=0):
    """The stages' oracles stepped per period (with the curves), from a freshly loaded state, on sampled instances."""
    idx = np.sort(np.random.default_rng(seed).choice(su.n, min(n_idx, su.n), replace=False))
    orcs = []
    for j, p in enumerate(su.progs):
        orc = po.Oracle(po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables()), len(idx), su.ch)
        for nm, v in su.ctl[j].items():
            orc.set_register(nm, v[idx])
        orcs.append(orc)
    xs = None if x is None else np.ascontiguousarray(x[:, :, idx])
    s = y.shape[1]
    if curves:
        sub = [v if bc else np.ascontiguousarray(v[:, idx]) for (_, _, bc), v in zip(curves, vals)]
        want = ccc.oracle_chain_curves_stepped(orcs, xs, s, list(curves), sub, len(idx))
    else:
        want = cc.oracle_chain_stepped(orcs, xs, s)
    assert_bits_equal(np.ascontiguousarray(y[:, :, idx]), want, what + " against the oracle")


def n_sub_blocks(n, ch, s, sub=None, n_pi=0):
    """The sub-blocks of the host pipeline for a call (process_host_impl's sub-block length)."""
    if not sub:
        sub = (16 << 20) // (4 * n * (ch + n_pi))
    sub = min(max(8, sub // 8 * 8), s)
    return -(-s // sub)


def run_case(po, su, s, seed, what, fused, curves=(), sub=None, oracle=True):
    x = input_block(su.ch, s, su.n, seed)
    vals = ccc.curve_values(list(curves), s, su.n, np.random.default_rng(seed + 1000)) if curves else []
    want = su.definition(x, s, curves, vals)
    before = su.chain.status()["launches"]
    y = su.chain.process_host_curves(x, [(st, reg, v, bc) for (st, reg, bc), v in zip(curves, vals)])
    assert_bits_equal(y, want, what + " output")
    st = su.chain.status()
    n_pi = sum(1 for c in curves if not c[2])
    assert st["fused_last"] == (1 if fused else 0), (what, st)
    assert st["launches"] - before == (n_sub_blocks(su.n, su.ch, s, sub, n_pi) if fused else 0), (what, st)
    if not fused:
        assert st["message"], st
    if oracle:
        oracle_sampled(po, su, x, y, what, curves, vals)
    return x, y


@pytest.mark.parametrize("n,s", [(4096, 1024), (65536, 333), (300, 333)])
@pytest.mark.parametrize("name", ["three", "eight", "two_ch_three", "cfg4_cfg2", "cfg2_cfg3", "cfg5"])
def test_chains_over_sizes(po, name, n, s):
    texts, ch, fused = chain_texts(name)
    if name == "cfg5" and n == 65536:
        n = 4096
    su = Setup(texts, ch, n)
    try:
        for b in range(2):
            run_case(po, su, s, 10 * b + 1, f"{name} N={n} S={s} block {b}", fused, oracle=b == 0)
        assert_same_state(su, f"{name} N={n} S={s}")
    finally:
        su.close()


@pytest.mark.parametrize("sub", [8, 24, None])
@pytest.mark.parametrize("name", ["three", "cfg4_cfg2"])
def test_tune_sub(po, monkeypatch, name, sub):
    if sub:
        monkeypatch.setenv("FX8010_TUNE_SUB", str(sub))
    else:
        monkeypatch.delenv("FX8010_TUNE_SUB", raising=False)
    texts, ch, fused = chain_texts(name)
    su = Setup(texts, ch, 4096)
    try:
        run_case(po, su, 333, 3, f"{name} sub {sub}", fused, sub=sub)
        curves = ccc.curve_mix(su.progs, "several")
        run_case(po, su, 200, 4, f"{name} sub {sub} with curves", fused, curves=curves, sub=sub, oracle=fused)   # (the oracle starts fresh)
        assert_same_state(su, f"{name} sub {sub}")
    finally:
        su.close()


@pytest.mark.parametrize("name", ["three", "cfg4_cfg2"])
def test_pinned_async_calls_in_a_row(po, monkeypatch, name):
    """Three page-locked asynchronous calls queued back to back, then one synchronize, against pageable blocking calls on the twins."""
    monkeypatch.setenv("FX8010_TUNE_SUB", "64")
    texts, ch, fused = chain_texts(name)
    n, s = 4096, 300
    su = Setup(texts, ch, n)
    keep = []
    try:
        curves = ccc.curve_mix(su.progs, "several")
        xs, outs, vals = [], [], []
        for b in range(3):
            x, xo = fx.pinned_array((ch, s, n)); x[:] = input_block(ch, s, n, 40 + b)
            y, yo = fx.pinned_array((ch, s, n)); y[:] = 5.0
            keep += [xo, yo]
            v = ccc.curve_values(curves, s, n, np.random.default_rng(b))
            pv = []
            for a in v:
                p, po_ = fx.pinned_array(a.shape); p[:] = a; keep.append(po_); pv.append(p)
            xs.append(x); outs.append(y); vals.append(pv)
            if b == 1:
                su.chain.process_host_curves(x, [(st, reg, a, bc) for (st, reg, bc), a in zip(curves, pv)], out=y, wait=False)
            else:
                su.chain.process_host(x, out=y, wait=False)
        su.chain.synchronize()
        assert su.chain.status()["fused_last"] == (1 if fused else 0)
        for b in range(3):
            want = su.twin_chain.process_host_curves(np.array(xs[b]), [(st, reg, np.array(a), bc) for (st, reg, bc), a in zip(curves, vals[b])]
                                                     if b == 1 else [])
            assert_bits_equal(outs[b], want, f"{name} async call {b} against the pageable blocking call")
        assert_same_state(su, f"{name} async in a row")
    finally:
        su.close()
        del keep


@pytest.mark.parametrize("name", ["two_ch_three", "cfg2_cfg3"])
def test_in_place_and_slice(po, name):
    texts, ch, fused = chain_texts(name)
    n, s, lo, wide = 4096, 257, 12, 4096 + 40
    su = Setup(texts, ch, n)
    try:
        curves = ccc.curve_mix(su.progs, "several")
        x = input_block(ch, s, n, 5)
        vals = ccc.curve_values(curves, s, n, np.random.default_rng(6))
        want = su.definition(x, s, curves, vals)
        y = x.copy()
        su.chain.process_host_curves(y, [(st, reg, v, bc) for (st, reg, bc), v in zip(curves, vals)], out=y)
        assert_bits_equal(y, want, f"{name} in place")
        assert su.chain.status()["fused_last"] == (1 if fused else 0)
        # the slice form: columns lo .. lo + n of host blocks `wide` instances wide, curves included
        big_x = np.full((ch, s, wide), 9.0, np.float32); big_x[:, :, lo:lo + n] = x
        big_y = np.full((ch, s, wide), 3.0, np.float32)
        big_v = []
        for (_, _, bc), v in zip(curves, vals):
            if bc:
                big_v.append(v)
            else:
                b = np.full((s, wide), 2.0, np.float32); b[:, lo:lo + n] = v; big_v.append(b)
        want = su.definition(x, s, curves, vals)
        su.chain.process_host_curves(big_x[:, :, lo:lo + n], [(st, reg, v if bc else v[:, lo:lo + n], bc) for (st, reg, bc), v in zip(curves, big_v)],
                                     out=big_y[:, :, lo:lo + n], host_instances=wide)
        assert_bits_equal(big_y[:, :, lo:lo + n], want, f"{name} slice")
        assert bool((big_y[:, :, :lo] == 3.0).all() and (big_y[:, :, lo + n:] == 3.0).all()), "columns outside the slice were written"
        # no `out`: the bindings allocate a block `wide` instances wide and return its first n columns
        want = su.definition(x, s)
        y = su.chain.process_host(big_x[:, :, lo:lo + n], host_instances=wide)
        assert y.shape == (ch, s, n) and y.strides[1] == 4 * wide
        assert_bits_equal(y, want, f"{name} slice without out")
        assert_same_state(su, f"{name} in place and slice")
    finally:
        su.close()


@pytest.mark.parametrize("name,mix", [("eight", "eight"), ("three", "several"), ("two_ch_three", "eight"), ("cfg4_cfg2", "cutoff")])
def test_curves(po, name, mix):
    texts, ch, fused = chain_texts(name)
    su = Setup(texts, ch, 4096)
    try:
        curves = [(0, su.progs[0].reg_index("filter_cutoff"), False)] if mix == "cutoff" else ccc.curve_mix(su.progs, mix)
        if mix == "eight":
            assert len(curves) == 8 and any(c[2] for c in curves) and not all(c[2] for c in curves)
        for b in range(2):
            run_case(po, su, 333, 20 + b, f"{name} {mix} block {b}", fused, curves=curves, oracle=b == 0)
        assert_same_state(su, f"{name} {mix}")
    finally:
        su.close()


def test_refused_calls_change_nothing():
    texts, ch, _ = chain_texts("three")
    n, s = 4096, 16
    su = Setup(texts, ch, n)
    try:
        vol = su.progs[1].reg_index("volume")
        in_l = su.progs[1].reg_index("in_l")
        x = input_block(ch, s, n, 0)
        v = np.random.default_rng(1).random((s, n)).astype(np.float32)
        vb = v[0, :s].copy()
        su.chain.process_host(x)
        y = np.full((ch, s, n), 3.0, np.float32)
        before = ([g.launch_info().kernel_launches for g in su.stages], su.chain.status()["launches"], [full_state(g) for g in su.stages])
        bad = [[(3, vol, v, False)], [(-1, vol, v, False)], [(1, 999, v, False)], [(1, vol, v, False), (1, vol, vb, True)],
               [(1, in_l, v, False)], [(1, vol, v, False)] * 9, [(0, su.progs[0].reg_index("volume"), v, False), (2, 999, v, False)]]
        for curves in bad:
            with pytest.raises(fx.FxError) as e:
                su.chain.process_host_curves(x, curves, out=y)
            assert e.value.code == 1, curves
        L = fx.gpu_lib()
        h, px, py = su.chain.h, x.ctypes.data, y.ctypes.data
        arr = (fx.CChainHostCurve * 1)()
        arr[0].stage, arr[0].reg_index, arr[0].broadcast, arr[0].values = 1, vol, 0, None
        assert L.fx8010_chain_process_batch_host_curves(h, px, py, s, C.addressof(arr), 1, 0, 1) == 1         # NULL values
        assert L.fx8010_chain_process_batch_host_curves(h, px, py, s, None, 1, 0, 1) == 1
        assert L.fx8010_chain_process_batch_host_curves(h, px, py, s, None, -1, 0, 1) == 1
        assert L.fx8010_chain_process_batch_host(h, px, py, s, n - 1, 1) == 1                                  # host rows too short
        assert L.fx8010_chain_process_batch_host(h, None, py, s, 0, 1) == 1                                     # stage 0 reads an input
        assert L.fx8010_chain_process_batch_host(h, px, None, s, 0, 1) == 1
        assert L.fx8010_chain_process_batch_host(h, px, py, -1, 0, 1) == 1
        after = ([g.launch_info().kernel_launches for g in su.stages], su.chain.status()["launches"], [full_state(g) for g in su.stages])
        assert after[:2] == before[:2]
        for j, (a, b) in enumerate(zip(before[2], after[2])):
            for key in a:
                assert_bits_equal(a[key], b[key], f"stage {j} {key} after refused calls")
        assert bool((y == 3.0).all()), "the output buffer was written"
        bare = fx.Gpu(n, ch)
        ch2 = fx.Chain([su.stages[0], bare])
        assert L.fx8010_chain_process_batch_host(ch2.h, px, py, s, 0, 1) == 3                                  # a stage without a program
        ch2.close(); bare.close()
    finally:
        su.close()


def test_mode_0_runs_stage_by_stage(po):
    texts, ch, _ = chain_texts("three")
    su = Setup(texts, ch, 4096, mode=0, twin_mode=0)
    try:
        run_case(po, su, 333, 2, "mode 0", False)
        assert "translation is off" in su.chain.status()["message"]
        assert_same_state(su, "mode 0")
    finally:
        su.close()


def test_mode_1_switches_over_inside_one_call(po, monkeypatch):
    """Mode 1: the calls queue stage by stage until the background compile ends; the call during which it ends runs its first sub-blocks
    stage by stage and the rest fused, with the same bits.  A call here is 65 536 sub-blocks of 8 periods over pageable buffers, each one
    paced by its own copies (seconds per call), and the compile starts inside the first call: it ends inside a call, not in the
    microseconds between two."""
    monkeypatch.setenv("FX8010_TUNE_SUB", "8")
    texts = [progs.CFG2_LOG_GAIN, cc.LIMIT.replace("-0.5", "-0.421875")]          # (a source no other test compiles)
    n, s = 4, 8 * 65536
    su = Setup(texts, 1, n, mode=1, twin_mode=0)
    try:
        x = input_block(1, s, n, 0)
        want = su.definition(x, s)
        n_sub = n_sub_blocks(n, 1, s, 8)
        deltas, partial = [], []
        y = np.empty_like(x)
        for _ in range(30):
            before = su.chain.status()["launches"]
            su.chain.process_host(x, out=y)
            st = su.chain.status()
            deltas.append(st["launches"] - before)
            if 0 < deltas[-1] < n_sub:
                assert st["fused_last"] == 0 and "compiling" in st["message"], st
                partial.append(y.copy())
            if st["fused_last"]:
                assert deltas[-1] == n_sub and st["message"] == "", st
                break
        assert deltas[0] < n_sub and deltas[-1] == n_sub and deltas == sorted(deltas), deltas
        assert len(partial) == 1, f"no call saw the compile end (fused launches per call {deltas})"
        assert_bits_equal(partial[0], want, "mode 1 switch-over call")
        assert_bits_equal(y, want, "mode 1 fused call")
        for _ in range(len(deltas) - 1):
            su.definition(x, s)
        assert_same_state(su, "mode 1")
    finally:
        su.close()


def test_interleaving_with_the_stages_own_calls(po):
    """Stage 0's own asynchronous host call, an asynchronous host chain call, a device chain call on a torch stream and stage 1's state
    getters right after the asynchronous chain call, on the same handles; the twins run the same sequence blocking."""
    texts, ch, _ = chain_texts("three")
    n, s = 4096, 500
    su = Setup(texts, ch, n)
    keep = []
    try:
        x0, o0 = fx.pinned_array((ch, s, n)); x0[:] = input_block(ch, s, n, 1)
        y0, o1 = fx.pinned_array((ch, s, n))
        x1, o2 = fx.pinned_array((ch, s, n)); x1[:] = input_block(ch, s, n, 2)
        y1, o3 = fx.pinned_array((ch, s, n))
        keep += [o0, o1, o2, o3]
        su.stages[0].process_host_ptr(x0.ctypes.data, y0.ctypes.data, s, wait=False)
        su.chain.process_host(x1, out=y1, wait=False)
        regs1 = su.stages[1].registers()                     # (waits for the chain call's work)
        d_x = torch.from_numpy(input_block(ch, s, n, 3)).cuda()
        d_y = torch.empty_like(d_x)
        stream = torch.cuda.Stream()
        su.chain.process_batch(d_x, d_y, s, stream.cuda_stream)
        su.chain.synchronize()
        torch.cuda.synchronize()
        w0 = su.twins[0].process_host(np.array(x0))
        w1 = su.twin_chain.process_host(np.array(x1))
        assert_bits_equal(su.twins[1].registers(), regs1, "stage 1 registers right after the asynchronous chain call")
        d_r = torch.empty_like(d_x)
        su.twin_chain.process_batch(d_x, d_r, s)
        torch.cuda.synchronize()
        assert_bits_equal(y0, w0, "stage 0's own host call")
        assert_bits_equal(y1, w1, "host chain call")
        assert_bits_equal(d_y.cpu().numpy(), d_r.cpu().numpy(), "device chain call")
        assert_same_state(su, "interleaved")
    finally:
        su.close()
        del keep


# ---- executor chains ----

class ShardView(fx.Gpu):
    """The handle of shard k of an executor (fx8010_multi_shard), read through Gpu's state getters; the executor owns it."""

    def __init__(self, m, k):
        self.L = fx.gpu_lib()
        lo, hi = C.c_int(), C.c_int()
        self.h = self.L.fx8010_multi_shard(m.h, k, C.byref(lo), C.byref(hi))
        self.lo, self.n, self.c = lo.value, hi.value - lo.value, m.c

    def close(self):
        pass

    __del__ = close


class MultiSetup:
    """Executors (one per stage) over `devices` and twins: single-device handles over all N instances in a device chain."""

    def __init__(self, texts, ch, n, devices, mode=2, seed=3):
        self.n, self.ch = n, ch
        self.progs = [fx.Program(t, channels=ch) for t in texts]
        rng = np.random.default_rng(seed)
        self.ctl = [cc.controls(p, n, rng) if j % 2 == 0 else {} for j, p in enumerate(self.progs)]
        self.execs = []
        for j, p in enumerate(self.progs):
            m = fx.MultiGpu(devices, n, ch)
            m.load_program(p)
            m.set_option(fx.OPT_TRANSLATE, mode)
            for nm, v in self.ctl[j].items():
                m.set_controls(p.reg_index(nm), v)
            self.execs.append(m)
        self.twins = []
        for j, p in enumerate(self.progs):
            g = fx.Gpu(n, ch); g.load_program(p); g.set_option(fx.OPT_TRANSLATE, 0)
            for nm, v in self.ctl[j].items():
                g.set_controls(p.reg_index(nm), v)
            self.twins.append(g)
        self.chain = fx.MultiChain(self.execs)
        self.twin_chain = fx.Chain(self.twins)

    definition = Setup.definition

    def assert_same_state(self, what):
        """Every shard handle's whole state against the twin's columns of that shard; the flags OR-ed over the shards."""
        for j, (m, g) in enumerate(zip(self.execs, self.twins)):
            want = full_state(g)
            for k in range(len(m.shards())):
                sh = ShardView(m, k)
                got, lo, hi = full_state(sh), sh.lo, sh.lo + sh.n
                for key in ("registers", "lfsr", "latch", "ptrs"):
                    assert_bits_equal(got[key], want[key][:, lo:hi], f"{what}: stage {j} shard {k} {key}")
                for key in ("acc", "counts"):
                    assert_bits_equal(got[key], want[key][lo:hi], f"{what}: stage {j} shard {k} {key}")
                d = sh.dims()
                for which, size in ((0, d.itram_size), (1, d.xtram_size)):
                    for i in (0, sh.n // 2, sh.n - 1) if size else ():
                        assert_bits_equal(sh.tram(which, i), g.tram(which, lo + i), f"{what}: stage {j} shard {k} tram{which} {i}")
            assert m.flags() == g.flags(), f"{what}: stage {j} flags"

    def close(self):
        self.chain.close(); self.twin_chain.close()
        for o in self.execs + self.twins:
            o.close()


def run_multi(po, ms, s, seed, what, fused, curves=(), oracle=True):
    x = input_block(ms.ch, s, ms.n, seed)
    vals = ccc.curve_values(list(curves), s, ms.n, np.random.default_rng(seed + 1)) if curves else []
    want = ms.definition(x, s, curves, vals)
    y = ms.chain.process_host_curves(x, [(st, reg, v, bc) for (st, reg, bc), v in zip(curves, vals)])
    assert_bits_equal(y, want, what + " output")
    for g in range(len(ms.execs[0].shards())):
        assert ms.chain.shard_status(g)["fused_last"] == (1 if fused else 0), (what, g, ms.chain.shard_status(g))
    if oracle:
        oracle_sampled(po, ms, x, y, what, curves, vals)
    return y


@pytest.mark.parametrize("name,n", [("three", 4096), ("three", 6002), ("cfg2_cfg3", 4096)])
def test_executor_chain_two_shards_on_one_ordinal(po, name, n):
    """Two shards on GPU 0: N = 4096 gives 2048 instances a shard (fused when every stage is stateless); N = 6002 gives 3001 (not a
    multiple of 4: stage by stage).  cfg2 -> cfg3 carries a delay line: its TRAM and pointers are compared shard by shard."""
    texts, ch, stateless = chain_texts(name)
    fused = stateless and n % 8 == 0
    ms = MultiSetup(texts, ch, n, [0, 0])
    try:
        curves = ccc.curve_mix(ms.progs, "several")
        run_multi(po, ms, 333, 1, f"executor {name} N={n}", fused)
        run_multi(po, ms, 200, 2, f"executor {name} N={n} with curves", fused, curves=curves, oracle=stateless)   # (the oracle starts fresh)
        x = input_block(ch, 100, n, 3)
        y = ms.chain.process_host(x, wait=False)
        ms.chain.synchronize()
        assert_bits_equal(y, ms.definition(x, 100), f"executor {name} N={n} asynchronous")
        ms.assert_same_state(f"executor {name} N={n}")
    finally:
        ms.close()


def test_executor_chain_refusals_and_create_checks():
    texts, ch, _ = chain_texts("three")
    n, s = 1000, 16
    ms = MultiSetup(texts, ch, n, [0, 0, 0])
    others = []
    try:
        vol = ms.progs[1].reg_index("volume")
        x = input_block(ch, s, n, 0)
        ms.chain.process_host(x)
        regs = [m.registers() for m in ms.execs]
        counts = [m.count_total() for m in ms.execs]
        y = np.full((ch, s, n), 3.0, np.float32)
        v = np.zeros((s, n), np.float32)
        for curves in ([(1, 999, v, False)], [(3, vol, v, False)], [(0, ms.progs[0].reg_index("volume"), v, False), (2, 999, v[0, :s], True)]):
            with pytest.raises(fx.FxError) as e:
                ms.chain.process_host_curves(x, curves, out=y)
            assert e.value.code == 1
        assert bool((y == 3.0).all()), "a refused list wrote the output"
        L = fx.gpu_lib()
        assert L.fx8010_multi_chain_process_batch_host(ms.chain.h, x.ctypes.data, None, s, 1) == 1
        assert "out is NULL" in L.fx8010_multi_chain_last_error(ms.chain.h).decode()
        assert L.fx8010_multi_chain_process_batch_host_curves(ms.chain.h, x.ctypes.data, y.ctypes.data, s, None, 9, 1) == 1
        assert "curve count" in L.fx8010_multi_chain_last_error(ms.chain.h).decode()
        for j, m in enumerate(ms.execs):
            assert_bits_equal(m.registers(), regs[j], f"stage {j} registers after refused lists")
            assert m.count_total() == counts[j]
        # create: mismatched executors are refused
        for devs, nn, cc_ in (([0, 0], n, ch), ([0, 0, 0], n + 4, ch), ([0, 0, 0], n, ch + 1)):
            m = fx.MultiGpu(devs, nn, cc_)
            others.append(m)
            with pytest.raises(fx.FxError) as e:
                fx.MultiChain([ms.execs[0], m])
            assert e.value.code == 1
        with pytest.raises(fx.FxError):
            fx.MultiChain([ms.execs[0], ms.execs[0]])
    finally:
        ms.close()
        for m in others:
            m.close()


def test_executor_chain_cfg4_full_size(po):
    """cfg4 (a per-instance cutoff curve) then cfg2 at 65 536 instances x 1 024 periods over the shards."""
    devices = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    texts, ch, _ = chain_texts("cfg4_cfg2")
    ms = MultiSetup(texts, ch, 65536, devices)
    try:
        curves = [(0, ms.progs[0].reg_index("filter_cutoff"), False)]
        run_multi(po, ms, 1024, 4, "executor cfg4 65536 x 1024", False, curves=curves)
        ms.assert_same_state("executor cfg4 65536 x 1024")
    finally:
        ms.close()


def test_executor_chain_two_gpus(po):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    texts, ch, _ = chain_texts("three")
    ms = MultiSetup(texts, ch, 8192, [0, 1])
    try:
        run_multi(po, ms, 333, 5, "executor two GPUs", True, curves=ccc.curve_mix(ms.progs, "several"))
        ms.assert_same_state("executor two GPUs")
    finally:
        ms.close()


# ---- the facade ----

@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_facade_host_chain(po, devices):
    n, s = 4096, 300
    texts, ch, _ = chain_texts("three")
    objs = [fx.Program(t, channels=ch, instances=n, devices=devices) for t in texts]
    for o in objs:
        o.set_translation(2)
    pc = objs[0].chain(objs[1:])
    twins = []
    try:
        x = input_block(ch, s, n, 9)
        vals = ccc.curve_values([(0, 0, False), (2, 0, True)], s, n, np.random.default_rng(5))
        y0 = pc.process_block(x)
        y1 = pc.process_block_curves(x, [(0, "volume", vals[0], False), (2, "ceil", vals[1], True)])
        for j, o in enumerate(objs):
            g = fx.Gpu(n, ch); g.load_program(o); g.set_option(fx.OPT_TRANSLATE, 0); twins.append(g)
        tc = fx.Chain(twins)
        d_x = torch.from_numpy(x).cuda()
        d_r = torch.empty_like(d_x)
        tc.process_batch(d_x, d_r, s)
        torch.cuda.synchronize()
        assert_bits_equal(y0, d_r.cpu().numpy(), "facade processBlock")
        d_v = [torch.from_numpy(v).cuda() for v in vals]
        tc.process_batch_curves(d_x, d_r, s, [(0, objs[0].reg_index("volume"), d_v[0], False), (2, objs[2].reg_index("ceil"), d_v[1], True)])
        torch.cuda.synchronize()
        assert_bits_equal(y1, d_r.cpu().numpy(), "facade processBlockWithCurves")
        tc.close()
        for bad in ([(3, "volume", vals[0], False)], [(1, "no_such_register", vals[0], False)]):
            with pytest.raises(fx.FxError):
                pc.process_block_curves(x, bad)
        if devices:
            with pytest.raises(fx.FxError):
                pc(d_x, d_r, s)
            with pytest.raises(fx.FxError):
                pc.process_curves(d_x, d_r, s, [])
            single = fx.Program(texts[0], channels=ch, instances=n)
            with pytest.raises(fx.FxError):
                fx.ProgramChain([single, objs[1]])
            with pytest.raises(fx.FxError):
                fx.ProgramChain([objs[1], single])
            single.close()
    finally:
        pc.close()
        for g in twins:
            g.close()
        for o in objs:
            o.close()
