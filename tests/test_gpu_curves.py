"""fx8010_gpu_process_batch_curves on the GPU: bit-identical to the oracle stepped one sample period at a time (set_register before each
period) and to process_batch_events with one event per curve at every period — outputs and the whole final state.  Also: the fast path
really runs (kernel_variant bit 4) in mode 2 and not in mode 0, the mode-1 switch-over keeps the bits, plain and automated calls
interleave without recompiling, a folded STATIC that gets automated voids the plain translation once, a second CUDA stream is ordered,
every rejected argument list queues nothing, and the facade call by register name."""
import ctypes as C
import time

import numpy as np
import pytest

import curves_common as cc
import progs
from conftest import assert_bits_equal

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def setup(fx, po, name, n, mode=2):
    text, ch, cv = cc.programs()[name]
    prog = fx.Program(text, channels=ch)
    assert prog.loaded, prog.errors()
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, n, ch)
    gpu = fx.Gpu(n, ch, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, mode)
    regs = [prog.reg_index(r) for r, _ in cv]
    return prog, orc, gpu, regs, [b for _, b in cv], [r for r, _ in cv], ch


def curves_for(name, names, bcast, s, n, rng):
    return [cc.make_curve(name, r, b, s, n, rng) for r, b in zip(names, bcast)]


def run_curves(gpu, x, vals, regs, bcast, stream=None):
    d_x = torch.from_numpy(x).cuda()
    d_y = torch.empty_like(d_x)
    d_v = [torch.from_numpy(v).cuda() for v in vals]
    torch.cuda.synchronize()
    gpu.process_device_curves(d_x, d_y, x.shape[1], list(zip(regs, d_v, bcast)), stream)
    gpu.synchronize(stream)
    return d_y.cpu().numpy()


def run_events(gpu, x, vals, regs):
    s = x.shape[1]
    events = [(k, r, v[k]) for k in range(s) for r, v in zip(regs, vals)]
    d_x = torch.from_numpy(x).cuda()
    d_y = torch.empty_like(d_x)
    torch.cuda.synchronize()
    gpu.process_device_events(d_x, d_y, s, events)
    gpu.synchronize()
    return d_y.cpu().numpy()


def state(gpu):
    acc, lfsr, latch, ptrs = gpu.scalars()
    return {"registers": gpu.registers(), "acc": acc, "lfsr": lfsr, "latch": latch, "ptrs": ptrs, "counts": gpu.counts(), "flags": np.array(gpu.flags())}


def check_state(gpu, orc, prog, what, n):
    st = state(gpu)
    assert_bits_equal(st["registers"], orc.registers, what + " registers")
    assert_bits_equal(st["acc"], orc.acc, what + " accumulator")
    assert_bits_equal(st["lfsr"], orc.lfsr, what + " lfsr")
    assert_bits_equal(st["latch"], orc.out_latch, what + " latch")
    assert_bits_equal(st["ptrs"], orc.tram_ptrs, what + " tram pointers")
    assert_bits_equal(st["counts"], orc.counts, what + " counters")
    assert int(st["flags"]) == orc.flags, what + " runtime flags"
    if prog.itram_size:
        for i in sorted({0, n // 2, n - 1}):
            assert_bits_equal(gpu.tram(0, i), orc.tram(0, i), f"{what} itram[{i}]")


@pytest.mark.parametrize("n", [1, 300, 4096])
@pytest.mark.parametrize("name", sorted(cc.programs()))
def test_curves_match_the_oracle_and_per_period_events(fx, po, name, n):
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, name, n)
    ev_gpu = fx.Gpu(n, ch, 0)
    ev_gpu.load_program(prog)
    ev_gpu.set_option(fx.OPT_TRANSLATE, 0)
    rng = np.random.default_rng(sum(map(ord, name)) + n)
    blocks = [64, 3] if name == "cfg5" else ([260, 1, 99] if name in ("delay_fb", "delay_mod") else [100, 1, 37])
    for b, s in enumerate(blocks):
        x = (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)
        vals = curves_for(name, names, bcast, s, n, rng)
        y = run_curves(gpu, x, vals, regs, bcast)
        info = gpu.launch_info()
        assert info.kernel_variant & fx.VARIANT_CURVES, f"{name} n={n}: the automated kernel did not run ({gpu.translate_status()})"
        assert_bits_equal(y, cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s), f"{name} n={n} block {b} vs oracle")
        assert_bits_equal(y, run_events(ev_gpu, x, vals, regs), f"{name} n={n} block {b} vs events")
    check_state(gpu, orc, prog, f"{name} n={n}", n)
    gpu.close(); ev_gpu.close()


def test_cfg4_full_size_sampled(fx, po):
    """cfg4 at the bench geometry (65 536 instances x 1 024 periods, a per-instance cutoff curve), sampled instances against the oracle."""
    n, s = 65536, 1024
    prog = fx.Program(progs.CFG4_ONEPOLE)
    gpu = fx.Gpu(n, 1, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, 2)
    rng = np.random.default_rng(44)
    x = progs.sine_bank(n, s, rng).reshape(1, s, n)
    cut = cc.make_curve("cfg4_cutoff", "filter_cutoff", False, s, n, rng)
    reg = prog.reg_index("filter_cutoff")
    y = run_curves(gpu, x, [cut], [reg], [False])
    assert gpu.launch_info().kernel_variant & fx.VARIANT_CURVES
    regs = gpu.registers()
    counts = gpu.counts()
    pick = np.unique(np.concatenate([[0, 1, n - 1], rng.choice(n, 93, replace=False)]))
    text = progs.CFG4_ONEPOLE
    from oracle import pyoracle
    p2 = fx.Program(text)
    img = pyoracle.Image(p2.instructions(), p2.registers(), p2.itram_size, p2.xtram_size, p2.controls(), p2.tables())
    orc = pyoracle.Oracle(img, len(pick), 1)
    want = cc.oracle_stepped(orc, np.ascontiguousarray(x[:, :, pick]), [(reg, np.ascontiguousarray(cut[:, pick]), False)], s)
    assert_bits_equal(y[:, :, pick], want, "cfg4 65536 x 1024 sampled outputs")
    assert_bits_equal(regs[:, pick], orc.registers, "cfg4 sampled registers")
    assert_bits_equal(counts[pick], orc.counts, "cfg4 sampled counters")
    gpu.close()


@pytest.mark.parametrize("name", ["cfg2_instance", "delay_fb", "log_select"])
def test_instance_count_not_a_multiple_of_four(fx, po, name):
    """The streaming kernel needs N % 4 == 0: such programs take the serial kernel with curves instead."""
    n = 301
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, name, n)
    rng = np.random.default_rng(3)
    for s in (250, 7):
        x = (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)
        vals = curves_for(name, names, bcast, s, n, rng)
        y = run_curves(gpu, x, vals, regs, bcast)
        assert gpu.launch_info().kernel_variant & fx.VARIANT_CURVES
        assert_bits_equal(y, cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s), f"{name} n=301")
    check_state(gpu, orc, prog, f"{name} n=301", n)
    gpu.close()


@pytest.mark.parametrize("mode", [0, 2])
def test_fast_path_bit_in_mode_2_only(fx, po, mode):
    n, s = 256, 64
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, "cfg4_cutoff", n, mode)
    rng = np.random.default_rng(8)
    x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
    vals = curves_for("cfg4_cutoff", names, bcast, s, n, rng)
    before = gpu.launch_info().kernel_launches
    y = run_curves(gpu, x, vals, regs, bcast)
    info = gpu.launch_info()
    assert_bits_equal(y, cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s), f"mode {mode}")
    check_state(gpu, orc, prog, f"mode {mode}", n)
    if mode == 2:
        assert info.kernel_variant & fx.VARIANT_CURVES and info.kernel_launches - before == 1
    else:
        assert not info.kernel_variant & fx.VARIANT_CURVES and info.kernel_launches - before == 2 * s     # per period: one copy, one launch
    gpu.close()


def test_mode_1_switch_over_keeps_the_bits(fx, po):
    n, s = 512, 32
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, "skip_data", n, 1)
    rng = np.random.default_rng(10)
    switched, t0 = False, time.time()
    while time.time() - t0 < 90:
        x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
        vals = curves_for("skip_data", names, bcast, s, n, rng)
        y = run_curves(gpu, x, vals, regs, bcast)
        assert_bits_equal(y, cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s), "mode 1")
        if gpu.launch_info().kernel_variant & fx.VARIANT_CURVES:
            if switched:
                break
            switched = True
    assert switched, "the automated kernel never came into use"
    check_state(gpu, orc, prog, "mode 1", n)
    gpu.close()


@pytest.mark.parametrize("name", ["cfg2_instance", "cfg5"])
def test_plain_and_automated_calls_interleave(fx, po, name):
    """State continues across plain / automated / plain calls; the plain translation stays in use and nothing is recompiled."""
    n = 512
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, name, n)
    rng = np.random.default_rng(12)
    d_x = torch.empty((1, 16, n), dtype=torch.float32, device="cuda")
    for k in range(3):
        for automated in (False, True, False):
            s = 16
            x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
            if automated:
                vals = curves_for(name, names, bcast, s, n, rng)
                y = run_curves(gpu, x, vals, regs, bcast)
                want = cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s)
            else:
                d_x.copy_(torch.from_numpy(x)); d_y = torch.empty_like(d_x)
                gpu.process_device(d_x, d_y, s)
                gpu.synchronize()
                y = d_y.cpu().numpy()
                want = orc.process(x)
                assert gpu.launch_info().kernel_variant & 128, "the plain call left its translated kernel"
            assert_bits_equal(y, want, f"{name} round {k} automated={automated}")
    assert gpu.translate_status()["state"] == 2
    check_state(gpu, orc, prog, name + " interleaved", n)
    gpu.close()


def test_interleaving_compiles_each_translation_once(fx, po, monkeypatch):
    """A fresh program text per test run (so the process-wide kernel cache cannot serve it): the first plain and the first automated
    call compile (mode 2: synchronously, ~hundreds of ms); every later call of either kind must take no compiler time."""
    n = 1024
    gain = 0.5 + (time.time_ns() % 1000003) / 4e6
    text = progs.CFG2_LOG_GAIN.replace("macs out_l, 0, a, volume", f"macs a, 0, a, {gain:.6f}\nmacs out_l, 0, a, volume")
    prog = fx.Program(text)
    gpu = fx.Gpu(n, 1, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, 2)
    reg = prog.reg_index("volume")
    d_x = torch.rand((1, 64, n), device="cuda"); d_y = torch.empty_like(d_x); d_v = torch.rand((64, n), device="cuda")
    times = []
    for k in range(8):
        t0 = time.perf_counter()
        if k % 2:
            gpu.process_device_curves(d_x, d_y, 64, [(reg, d_v, False)])
        else:
            gpu.process_device(d_x, d_y, 64)
        gpu.synchronize()
        times.append(time.perf_counter() - t0)
        assert gpu.launch_info().kernel_variant & (fx.VARIANT_CURVES if k % 2 else 128)
    assert max(times[2:]) < 0.05, f"a later call took {max(times[2:]) * 1e3:.1f} ms: recompiled? {times}"
    gpu.close()


def test_folded_static_automated_voids_the_plain_translation_once(fx, po):
    """`static k` is an immediate of the plain translation (a stateless program: the streaming kernel); automating it voids that
    translation, so the next plain call retranslates without folding it.  Once: from then on neither kind of call compiles anything
    (mode 2 compiles synchronously, hundreds of ms; a literal unique to this run keeps the process-wide kernel cache from serving it)."""
    kv = 0.25 + (time.time_ns() % 999983) / 8e6
    text = "\n".join([f"static k = {kv:.7f}", "static a", "input in_l 0", "output out_l 0", "log a, in_l, 3, 0", "macs out_l, 0, a, k", "end"])
    n, s = 256, 32
    prog = fx.Program(text)
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, n, 1)
    gpu = fx.Gpu(n, 1, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, 2)
    k = prog.reg_index("k")
    rng = np.random.default_rng(2)
    d_x = torch.empty((1, s, n), dtype=torch.float32, device="cuda")
    times = []                              # plain 0, automated 0, plain 1 (retranslated once), automated 1, plain 2, ...
    for rnd in range(4):
        x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
        d_x.copy_(torch.from_numpy(x)); d_y = torch.empty_like(d_x)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gpu.process_device(d_x, d_y, s); gpu.synchronize()
        times.append(time.perf_counter() - t0)
        assert_bits_equal(d_y.cpu().numpy(), orc.process(x), f"plain {rnd}")
        assert gpu.launch_info().kernel_variant & 128
        vals = curves_for("k", ["k"], [False], s, n, rng)
        d_v = torch.from_numpy(vals[0]).cuda(); d_y = torch.empty_like(d_x)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gpu.process_device_curves(d_x, d_y, s, [(k, d_v, False)]); gpu.synchronize()
        times.append(time.perf_counter() - t0)
        assert gpu.launch_info().kernel_variant & fx.VARIANT_CURVES
        assert_bits_equal(d_y.cpu().numpy(), cc.oracle_stepped(orc, x, [(k, vals[0], False)], s), f"automated {rnd}")
    assert max(times[3:]) < 0.05, f"a call after the one retranslation took {max(times[3:]) * 1e3:.1f} ms: recompiled? {times}"
    check_state(gpu, orc, prog, "folded static", n)
    gpu.close()


def test_unaligned_buffers_take_the_serial_kernel(fx, po):
    """A launch the streaming kernel cannot take (buffers not 16-byte aligned) moves the curve set to the serial kernel, not to one
    launch per period."""
    n, s = 4096, 64
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, "cfg2_instance", n)
    rng = np.random.default_rng(21)
    for rnd in range(2):
        x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
        vals = curves_for("cfg2_instance", names, bcast, s, n, rng)
        base = torch.zeros(s * n + 1, dtype=torch.float32, device="cuda")
        d_x = base[1:].view(1, s, n); d_x.copy_(torch.from_numpy(x))
        d_y = torch.zeros(s * n + 1, dtype=torch.float32, device="cuda")[1:].view(1, s, n)
        d_v = torch.from_numpy(vals[0]).cuda()
        torch.cuda.synchronize()
        before = gpu.launch_info().kernel_launches
        gpu.process_device_curves(d_x, d_y, s, [(regs[0], d_v, False)])
        gpu.synchronize()
        info = gpu.launch_info()
        assert info.kernel_variant & fx.VARIANT_CURVES and info.kernel_launches - before == 1
        assert gpu.translate_status_curves()["kind"] == 0
        assert_bits_equal(d_y.cpu().numpy(), cc.oracle_stepped(orc, x, [(regs[0], vals[0], False)], s), f"unaligned {rnd}")
    check_state(gpu, orc, prog, "unaligned", n)
    gpu.close()


def test_serial_ring_beyond_48_kib(fx, po):
    """cfg4 with a per-instance curve at 655 360 instances: two ring rows x 2 lanes x 32 periods x 128 threads = 64 KiB of shared memory,
    above the default dynamic limit (the kernel opts in)."""
    n, s = 655360, 64
    prog = fx.Program(progs.CFG4_ONEPOLE)
    gpu = fx.Gpu(n, 1, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, 2)
    rng = np.random.default_rng(45)
    x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
    cut = cc.make_curve("cfg4_cutoff", "filter_cutoff", False, s, n, rng)
    reg = prog.reg_index("filter_cutoff")
    y = run_curves(gpu, x, [cut], [reg], [False])
    info = gpu.launch_info()
    assert info.kernel_variant & fx.VARIANT_CURVES and info.last_smem_bytes > 48 * 1024, (info.kernel_variant, info.last_smem_bytes)
    pick = np.unique(np.concatenate([[0, 1, n - 1], rng.choice(n, 61, replace=False)]))
    orc = oracle_of(po, progs.CFG4_ONEPOLE, len(pick))
    want = cc.oracle_stepped(orc, np.ascontiguousarray(x[:, :, pick]), [(reg, np.ascontiguousarray(cut[:, pick]), False)], s)
    assert_bits_equal(y[:, :, pick], want, "cfg4 655360 sampled outputs")
    assert_bits_equal(gpu.registers()[:, pick], orc.registers, "cfg4 655360 sampled registers")
    gpu.close()


def oracle_of(po, text, n):
    import importlib
    p = importlib.import_module("fx8010-emulator-core_b200").Program(text)
    img = po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables())
    return po.Oracle(img, n, 1)


def test_curve_translation_status(fx, po):
    """The curve set's own translation is reported: the kernel kind in use, or why there is none (calls then run one launch per period)."""
    for name, n, kind in (("cfg2_instance", 256, 1), ("delay_fb", 256, 2), ("cfg4_cutoff", 256, 0)):
        prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, name, n)
        assert gpu.translate_status_curves()["state"] == 0
        vals = curves_for(name, names, bcast, 8, n, np.random.default_rng(1))
        run_curves(gpu, np.zeros((ch, 8, n), np.float32), vals, regs, bcast)
        st = gpu.translate_status_curves()
        assert st["state"] == 2 and st["kind"] == kind, (name, st)
        gpu.close()
    prog = fx.Program(cc.SKIP_COUNT)
    gpu = fx.Gpu(64, 1, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, 2)
    d_x = torch.zeros((1, 4, 64), device="cuda"); d_y = torch.empty_like(d_x); d_v = torch.ones(4, device="cuda")
    gpu.process_device_curves(d_x, d_y, 4, [(prog.reg_index("n"), d_v, True)])
    gpu.synchronize()
    st = gpu.translate_status_curves()
    assert st["state"] == -1 and "SKIP" in st["message"] and st["kind"] == -1, st
    assert not gpu.launch_info().kernel_variant & fx.VARIANT_CURVES
    gpu.close()


def test_second_stream_is_ordered(fx, po):
    """A curve buffer produced on one stream and consumed by a call on another, after earlier work of the handle on the first."""
    n, s = 4096, 128
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, "cfg4_cutoff", n)
    rng = np.random.default_rng(4)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    x1 = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
    x2 = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
    vals = curves_for("cfg4_cutoff", names, bcast, s, n, rng)
    d_x1, d_x2 = torch.from_numpy(x1).cuda(), torch.from_numpy(x2).cuda()
    d_y1, d_y2 = torch.empty_like(d_x1), torch.empty_like(d_x2)
    h_v = torch.from_numpy(vals[0]).pin_memory()
    d_v = torch.empty((s, n), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        gpu.process_device(d_x1, d_y1, s, s1.cuda_stream)
        torch.cuda._sleep(20_000_000)                    # keep s1 busy: the call on s2 must still come after
        d_v.copy_(h_v, non_blocking=True)
    gpu.process_device_curves(d_x2, d_y2, s, [(regs[0], d_v, False)], s2.cuda_stream)
    torch.cuda.synchronize()
    assert_bits_equal(d_y1.cpu().numpy(), orc.process(x1), "first call")
    assert_bits_equal(d_y2.cpu().numpy(), cc.oracle_stepped(orc, x2, [(regs[0], vals[0], False)], s), "second call on another stream")
    gpu.close()


def test_rejected_argument_lists_queue_nothing(fx, po):
    n = 64
    prog, orc, gpu, regs, bcast, names, ch = setup(fx, po, "cfg4_cutoff", n)
    L = fx.gpu_lib()
    d_x = torch.zeros((1, 8, n), device="cuda"); d_y = torch.zeros_like(d_x); d_v = torch.zeros((8, n), device="cuda")
    inp, out = prog.reg_index("in_l"), prog.reg_index("out_l")

    def call(curves, count=None):
        arr = (fx.CControlCurve * max(1, len(curves)))()
        for i, (r, p, b) in enumerate(curves):
            arr[i].reg_index, arr[i].broadcast, arr[i].d_values = r, b, p
        return L.fx8010_gpu_process_batch_curves(gpu.h, d_x.data_ptr(), d_y.data_ptr(), 8, C.addressof(arr), len(curves) if count is None else count, None)

    before = gpu.launch_info().kernel_launches
    p = d_v.data_ptr()
    bad = [
        [(regs[0], p, 0)] * 9,                                     # more than 8
        [(regs[0], p, 0), (regs[0], p, 1)],                        # named twice
        [(inp, p, 0)],                                             # an INPUT register
        [(out, p, 0)],                                             # an OUTPUT register
        [(10 ** 6, p, 0)],                                         # out of range
        [(-1, p, 0)],
        [(regs[0], None, 0)],                                      # NULL values
    ]
    for curves in bad:
        assert call(curves) == 1, curves
    assert call([(regs[0], p, 0)], count=-1) == 1
    assert L.fx8010_gpu_process_batch_curves(gpu.h, d_x.data_ptr(), d_y.data_ptr(), 8, None, 1, None) == 1
    assert gpu.launch_info().kernel_launches == before
    assert call([(regs[0], p, 0)]) == 0 and gpu.launch_info().kernel_launches == before + 1
    gpu.close()


def test_facade_by_register_name(fx, po):
    n, s = 512, 48
    text = progs.CFG4_ONEPOLE
    prog = fx.Program(text, instances=n)
    prog.set_translation(2)
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, n, 1)
    rng = np.random.default_rng(6)
    x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
    cut = cc.make_curve("cfg4_cutoff", "filter_cutoff", False, s, n, rng)
    d_x = torch.from_numpy(x).cuda(); d_y = torch.empty_like(d_x); d_c = torch.from_numpy(cut).cuda()
    torch.cuda.synchronize()
    prog.process_block_device_curves(d_x, d_y, s, [("filter_cutoff", d_c, False)])
    torch.cuda.synchronize()
    assert_bits_equal(d_y.cpu().numpy(), cc.oracle_stepped(orc, x, [(prog.reg_index("filter_cutoff"), cut, False)], s), "facade")
    with pytest.raises(Exception):
        prog.process_block_device_curves(d_x, d_y, s, [("no_such_register", d_c, False)])
    prog.close()
