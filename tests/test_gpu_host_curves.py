"""Control curves from host memory (fx8010_gpu_process_batch_host_curves, fx8010_multi_process_batch_host_curves, the facade's
processBlockWithCurves) on the GPU: bit-identical, in outputs and in the whole final state, to the oracle stepped one sample period at a
time and to fx8010_gpu_process_batch_curves on device copies of the same buffers.  Covers blocks spanning several pipeline sub-blocks,
page-locked and pageable buffers, chained asynchronous calls, the slice form, the per-period fallback, refused lists on a handle and on
every executor shard, uneven executor shards on one GPU and on two, cfg4 at the bench geometry, the facade on one and several devices,
and interleaving with plain host calls and device-curve calls without a second compile."""
import ctypes as C
import time

import numpy as np
import pytest

import curves_common as cc
import progs
from conftest import assert_bits_equal

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def image_of(po, prog):
    return po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())


def setup(fx, po, name, n, mode=2):
    text, ch, cv = cc.programs()[name]
    prog = fx.Program(text, channels=ch)
    assert prog.loaded, prog.errors()
    orc = po.Oracle(image_of(po, prog), n, ch)
    gpu = fx.Gpu(n, ch, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, mode)
    return prog, orc, gpu, [prog.reg_index(r) for r, _ in cv], [b for _, b in cv], [r for r, _ in cv], ch


def curves_for(name, names, bcast, s, n, rng):
    return [cc.make_curve(name, r, b, s, n, rng) for r, b in zip(names, bcast)]


def run_device_curves(gpu, x, vals, regs, bcast):
    d_x = torch.from_numpy(x).cuda()
    d_y = torch.empty_like(d_x)
    d_v = [torch.from_numpy(v).cuda() for v in vals]
    torch.cuda.synchronize()
    gpu.process_device_curves(d_x, d_y, x.shape[1], list(zip(regs, d_v, bcast)))
    gpu.synchronize()
    return d_y.cpu().numpy()


def check_state(gpu, orc, prog, what, lo=0, hi=None):
    """The handle's whole state against the oracle's instances lo..hi (registers, accumulator, LFSR, latch, TRAM pointers and contents,
    counters; the runtime flags when the handle holds every instance)."""
    hi = orc.n if hi is None else hi
    acc, lfsr, latch, ptrs = gpu.scalars()
    assert_bits_equal(gpu.registers(), orc.registers[:, lo:hi], what + " registers")
    assert_bits_equal(acc, orc.acc[lo:hi], what + " accumulator")
    assert_bits_equal(lfsr, orc.lfsr[:, lo:hi], what + " lfsr")
    assert_bits_equal(latch, orc.out_latch[:, lo:hi], what + " latch")
    assert_bits_equal(ptrs, orc.tram_ptrs[:, lo:hi], what + " tram pointers")
    assert_bits_equal(gpu.counts(), orc.counts[lo:hi], what + " counters")
    if (lo, hi) == (0, orc.n):
        assert gpu.flags() == orc.flags, what + " runtime flags"
    if prog.itram_size:
        for i in sorted({lo, (lo + hi) // 2, hi - 1}):
            assert_bits_equal(gpu.tram(0, i - lo), orc.tram(0, i), f"{what} itram[{i}]")


def shard_views(fx, m):
    """fx.Gpu views of an executor's shard handles (state access only; the executor owns and destroys them)."""
    class Shard(fx.Gpu):
        def close(self):
            self.h = None
        __del__ = close
    out = []
    for g, (lo, hi) in enumerate(m.shards()):
        v = Shard.__new__(Shard)
        v.L, v.n, v.c, v._keep = m.L, hi - lo, m.c, None
        v.h = C.c_void_p(m.L.fx8010_multi_shard(m.h, g, None, None))
        out.append((v, lo, hi))
    return out


def host_call_blocks(name):
    return [64, 3, 1] if name == "cfg5" else ([260, 1, 99] if name in ("delay_fb", "delay_mod") else [100, 1, 37])


@pytest.mark.parametrize("n,sub", [(1, 0), (300, 0), (300, 8), (4096, 0), (4096, 24)])
@pytest.mark.parametrize("name", sorted(cc.programs()))
def test_host_curves_match_the_oracle_and_device_curves(fx, po, monkeypatch, name, n, sub):
    """Every curve program in mode 2: the host call equals the oracle and the device call on device copies; FX8010_TUNE_SUB cuts a
    block into sub-blocks of 8 or 24 periods, so the curves are staged in many pieces."""
    if sub:
        monkeypatch.setenv("FX8010_TUNE_SUB", str(sub))
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, name, n)
    monkeypatch.delenv("FX8010_TUNE_SUB", raising=False)
    dev = fx.Gpu(n, ch, 0)
    dev.load_program(prog)
    dev.set_option(fx.OPT_TRANSLATE, 2)
    rng = np.random.default_rng(sum(map(ord, name)) + n + sub)
    for b, s in enumerate(host_call_blocks(name)):
        x = (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)
        vals = curves_for(name, names, bcast, s, n, rng)
        y = gpu.process_host_curves(x, list(zip(regs, vals, bcast)))
        assert gpu.launch_info().kernel_variant & fx.VARIANT_CURVES, f"{name} n={n}: the automated kernel did not run ({gpu.translate_status_curves()})"
        what = f"{name} n={n} sub={sub} block {b}"
        assert_bits_equal(y, cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s), what + " vs oracle")
        assert_bits_equal(y, run_device_curves(dev, x, vals, regs, bcast), what + " vs device curves")
    check_state(gpu, orc, prog, f"{name} n={n} sub={sub} host")
    check_state(dev, orc, prog, f"{name} n={n} sub={sub} device")
    gpu.close(); dev.close()


@pytest.mark.parametrize("name", ["cfg4_cutoff", "delay_mod"])
def test_pinned_async_chain_equals_blocking_pageable_calls(fx, po, monkeypatch, name):
    """Three wait=False calls from page-locked buffers, one synchronize: the same bits as three blocking calls from pageable memory."""
    n, s = 4096, 96
    monkeypatch.setenv("FX8010_TUNE_SUB", "32")
    prog, orc, a, regs, bcast, names, ch = setup(fx, po, name, n)
    b = fx.Gpu(n, ch, 0)
    monkeypatch.delenv("FX8010_TUNE_SUB")
    b.load_program(prog)
    b.set_option(fx.OPT_TRANSLATE, 2)
    rng = np.random.default_rng(5)
    owners, pinned, want = [], [], []
    for k in range(3):
        x = (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)
        vals = curves_for(name, names, bcast, s, n, rng)
        px, o1 = fx.pinned_array(x.shape); px[...] = x
        py, o2 = fx.pinned_array(x.shape); py[...] = 0
        pv = []
        for v in vals:
            p, o = fx.pinned_array(v.shape); p[...] = v; pv.append(p); owners.append(o)
        owners += [o1, o2]
        pinned.append((px, py, pv))
        want.append(cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s))
        a.process_host_curves(px, list(zip(regs, pv, bcast)), out=py, wait=False)
    a.synchronize()
    for k, (px, py, pv) in enumerate(pinned):
        y_b = b.process_host_curves(np.array(px), list(zip(regs, [np.array(v) for v in pv], bcast)))
        assert_bits_equal(py, y_b, f"{name} call {k}: async pinned vs blocking pageable")
        assert_bits_equal(py, want[k], f"{name} call {k} vs oracle")
    check_state(a, orc, prog, name + " async")
    check_state(b, orc, prog, name + " blocking")
    a.close(); b.close()


def test_slice_with_a_column_offset(fx, po):
    """host_instances > N: the handle's columns start at column 20 of blocks 300 wide; nothing outside them is written."""
    n, wide, lo, s = 256, 300, 20, 72
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, "delay_mod", n)
    rng = np.random.default_rng(9)
    for rnd in range(2):
        big_x = (1.8 * rng.random((ch, s, wide)) - 0.9).astype(np.float32)
        big_y = np.full((ch, s, wide), 7.0, np.float32)
        vals = curves_for("delay_mod", names, bcast, s, wide, rng)
        host = [v if bc else v[:, lo:lo + n] for v, bc in zip(vals, bcast)]
        gpu.process_host_curves(big_x[:, :, lo:lo + n], list(zip(regs, host, bcast)), out=big_y[:, :, lo:lo + n], host_instances=wide)
        assert gpu.launch_info().kernel_variant & fx.VARIANT_CURVES
        want = cc.oracle_stepped(orc, np.ascontiguousarray(big_x[:, :, lo:lo + n]),
                                 [(r, v if bc else np.ascontiguousarray(v), bc) for r, v, bc in zip(regs, host, bcast)], s)
        assert_bits_equal(big_y[:, :, lo:lo + n], want, f"slice round {rnd}")
        assert (big_y[:, :, :lo] == 7.0).all() and (big_y[:, :, lo + n:] == 7.0).all(), "columns outside the slice were written"
    check_state(gpu, orc, prog, "slice")
    gpu.close()


@pytest.mark.parametrize("sub", [0, 24])
def test_mode_0_runs_period_by_period_and_stays_exact(fx, po, monkeypatch, sub):
    n, s = 256, 64
    if sub:
        monkeypatch.setenv("FX8010_TUNE_SUB", str(sub))
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, "cfg4_cutoff", n, mode=0)
    rng = np.random.default_rng(8)
    x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
    vals = curves_for("cfg4_cutoff", names, bcast, s, n, rng)
    before = gpu.launch_info().kernel_launches
    y = gpu.process_host_curves(x, list(zip(regs, vals, bcast)))
    info = gpu.launch_info()
    assert not info.kernel_variant & fx.VARIANT_CURVES and info.kernel_launches - before == 2 * s     # per period: one copy, one launch
    assert_bits_equal(y, cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s), f"mode 0 sub={sub}")
    check_state(gpu, orc, prog, f"mode 0 sub={sub}")
    gpu.close()


BAD_LISTS = [
    lambda reg, p, inp, out: [(reg, p, 0)] * 9,                                 # more than 8
    lambda reg, p, inp, out: [(reg, p, 0), (reg, p, 1)],                        # named twice
    lambda reg, p, inp, out: [(inp, p, 0)],                                     # an INPUT register
    lambda reg, p, inp, out: [(out, p, 0)],                                     # an OUTPUT register
    lambda reg, p, inp, out: [(10 ** 6, p, 0)],                                 # out of range
    lambda reg, p, inp, out: [(-1, p, 0)],
    lambda reg, p, inp, out: [(reg, None, 0)],                                  # NULL values
]


def curve_array(fx, curves):
    arr = (fx.CHostCurve * max(1, len(curves)))()
    for i, (r, p, b) in enumerate(curves):
        arr[i].reg_index, arr[i].broadcast, arr[i].values = r, b, p
    return arr


def test_rejected_lists_queue_nothing(fx, po):
    n, s = 64, 8
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, "cfg4_cutoff", n)
    L = fx.gpu_lib()
    x = np.zeros((1, s, n), np.float32); y = np.zeros_like(x); v = np.zeros((s, n), np.float32)
    inp, out, p = prog.reg_index("in_l"), prog.reg_index("out_l"), v.ctypes.data

    def call(curves, count=None, host_instances=0):
        return L.fx8010_gpu_process_batch_host_curves(gpu.h, x.ctypes.data, y.ctypes.data, s, C.addressof(curve_array(fx, curves)),
                                                      len(curves) if count is None else count, host_instances, 1)

    before = gpu.launch_info().kernel_launches
    for make in BAD_LISTS:
        assert call(make(regs[0], p, inp, out)) == 1
    assert call([(regs[0], p, 0)], count=-1) == 1
    assert call([(regs[0], p, 0)], host_instances=n - 1) == 1                   # host rows narrower than the handle
    assert L.fx8010_gpu_process_batch_host_curves(gpu.h, x.ctypes.data, y.ctypes.data, s, None, 1, 0, 1) == 1
    assert gpu.launch_info().kernel_launches == before
    assert call([(regs[0], p, 0)]) == 0 and gpu.launch_info().kernel_launches == before + 1
    gpu.close()

    m = fx.MultiGpu([0, 0, 0], 1000)
    m.load_program(prog)
    m.set_option(fx.OPT_TRANSLATE, 2)
    shards = shard_views(fx, m)
    x = np.zeros((1, s, 1000), np.float32); y = np.zeros_like(x); v = np.zeros((s, 1000), np.float32)
    p = v.ctypes.data
    launches = [sh.launch_info().kernel_launches for sh, _, _ in shards]

    def mcall(curves, count=None):
        return L.fx8010_multi_process_batch_host_curves(m.h, x.ctypes.data, y.ctypes.data, s, C.addressof(curve_array(fx, curves)),
                                                        len(curves) if count is None else count, 1)

    for make in BAD_LISTS:
        assert mcall(make(regs[0], p, inp, out)) == 1
    assert mcall([(regs[0], p, 0)], count=-1) == 1
    assert L.fx8010_multi_process_batch_host_curves(m.h, x.ctypes.data, y.ctypes.data, s, None, 1, 1) == 1
    assert [sh.launch_info().kernel_launches for sh, _, _ in shards] == launches, "a shard queued work for a refused list"
    assert mcall([(regs[0], p, 0)]) == 0
    assert [sh.launch_info().kernel_launches for sh, _, _ in shards] == [k + 1 for k in launches]
    m.close()


def run_executor(fx, po, name, devices, n, blocks, seed):
    text, ch, cv = cc.programs()[name]
    prog = fx.Program(text, channels=ch)
    orc = po.Oracle(image_of(po, prog), n, ch)
    regs, bcast, names = [prog.reg_index(r) for r, _ in cv], [b for _, b in cv], [r for r, _ in cv]
    m = fx.MultiGpu(devices, n, ch)
    m.load_program(prog)
    m.set_option(fx.OPT_TRANSLATE, 2)
    rng = np.random.default_rng(seed)
    for b, s in enumerate(blocks):
        x = (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)
        vals = curves_for(name, names, bcast, s, n, rng)
        y = m.process_host_curves(x, list(zip(regs, vals, bcast)))
        assert_bits_equal(y, cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s), f"{name} on {devices} block {b}")
    flags = 0
    for sh, lo, hi in shard_views(fx, m):
        assert sh.launch_info().kernel_variant & fx.VARIANT_CURVES
        check_state(sh, orc, prog, f"{name} shard {lo}..{hi}", lo, hi)
        flags |= sh.flags()
    assert flags == orc.flags
    m.close()


@pytest.mark.parametrize("name", ["cfg4_cutoff", "delay_mod", "cfg5"])
def test_executor_three_uneven_shards_on_one_gpu(fx, po, name):
    """1 000 instances over three shards of device 0 (333, 333, 334): each shard reads its own columns of every per-instance curve."""
    run_executor(fx, po, name, [0, 0, 0], 1000, [64, 1, 37] if name == "cfg5" else [260, 1, 99], 31)


def test_executor_two_gpus(fx, po):
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU on this machine")
    run_executor(fx, po, "cfg4_cutoff", [0, 1], 1002, [200, 1, 57], 32)
    run_executor(fx, po, "delay_mod", [0, 1], 1002, [260, 3], 33)


def test_executor_cfg4_full_size_sampled(fx, po):
    """cfg4 at the bench geometry (65 536 instances x 1 024 periods, a per-instance cutoff curve) across the shards, sampled instances
    against the oracle."""
    n, s = 65536, 1024
    devices = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0, 0]
    prog = fx.Program(progs.CFG4_ONEPOLE)
    m = fx.MultiGpu(devices, n)
    m.load_program(prog)
    m.set_option(fx.OPT_TRANSLATE, 2)
    rng = np.random.default_rng(46)
    x = progs.sine_bank(n, s, rng).reshape(1, s, n)
    cut = cc.make_curve("cfg4_cutoff", "filter_cutoff", False, s, n, rng)
    reg = prog.reg_index("filter_cutoff")
    pin_cut, owner = fx.pinned_array(cut.shape)
    pin_cut[...] = cut
    y = m.process_host_curves(x, [(reg, pin_cut, False)])
    regs = m.registers()
    bounds = [lo for lo, _ in m.shards()] + [n]
    pick = np.unique(np.concatenate([[0, n - 1], [b - 1 for b in bounds[1:]], bounds[:-1], rng.choice(n, 70, replace=False)]))
    assert len(pick) >= 64
    orc = po.Oracle(image_of(po, prog), len(pick), 1)
    want = cc.oracle_stepped(orc, np.ascontiguousarray(x[:, :, pick]), [(reg, np.ascontiguousarray(cut[:, pick]), False)], s)
    assert_bits_equal(y[:, :, pick], want, "cfg4 65536 x 1024 sampled outputs")
    assert_bits_equal(regs[:, pick], orc.registers, "cfg4 sampled registers")
    m.close()


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_facade_by_register_name(fx, po, devices):
    """FX8010::processBlockWithCurves through the C view, on one device and with the multi-device constructor."""
    n = 512
    prog = fx.Program(cc.DELAY_MOD, instances=n, devices=devices)
    prog.set_translation(2)
    orc = po.Oracle(image_of(po, prog), n, 1)
    rng = np.random.default_rng(6)
    cv = cc.programs()["delay_mod"][2]
    for s in (120, 1, 48):
        x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
        vals = [cc.make_curve("delay_mod", r, b, s, n, rng) for r, b in cv]
        y = prog.process_block_curves(x, [(r, v, b) for (r, b), v in zip(cv, vals)])
        want = cc.oracle_stepped(orc, x, [(prog.reg_index(r), v, b) for (r, b), v in zip(cv, vals)], s)
        assert_bits_equal(y, want, f"facade on {devices or 'one device'} s={s}")
    with pytest.raises(fx.FxError):
        prog.process_block_curves(x, [("no_such_register", vals[0], False)])
    prog.close()


def test_interleaving_compiles_each_translation_once(fx, po):
    """Host-curve, plain-host and device-curve calls on one handle: state carries across them, and after the first plain and the first
    automated call (a fresh program text, so the process-wide kernel cache cannot serve it) no call compiles anything."""
    n, s = 1024, 48
    gain = 0.5 + (time.time_ns() % 1000003) / 4e6
    text = progs.CFG2_LOG_GAIN.replace("macs out_l, 0, a, volume", f"macs a, 0, a, {gain:.6f}\nmacs out_l, 0, a, volume")
    prog = fx.Program(text)
    orc = po.Oracle(image_of(po, prog), n, 1)
    gpu = fx.Gpu(n, 1, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, 2)
    reg = prog.reg_index("volume")
    rng = np.random.default_rng(13)
    compiles = []
    for k in range(9):
        x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
        vals = [cc.make_curve("cfg2_instance", "volume", False, s, n, rng)]
        kind = k % 3
        if kind == 0:
            y = gpu.process_host_curves(x, [(reg, vals[0], False)])
            want = cc.oracle_stepped(orc, x, [(reg, vals[0], False)], s)
        elif kind == 1:
            y = gpu.process_host(x)
            want = orc.process(x)
        else:
            y = run_device_curves(gpu, x, vals, [reg], [False])
            want = cc.oracle_stepped(orc, x, [(reg, vals[0], False)], s)
        assert gpu.launch_info().kernel_variant & (128 if kind == 1 else fx.VARIANT_CURVES), f"call {k}"
        assert_bits_equal(y, want, f"call {k} kind {kind}")
        compiles.append(fx.kernel_cache_stats()["nvrtc_compiles"])
    assert compiles[2] == compiles[-1], f"a later call compiled again: {compiles}"
    assert compiles[1] - compiles[0] <= 1
    check_state(gpu, orc, prog, "interleaved")
    gpu.close()
