"""In-place calls (d_out == d_in, include/fx8010_gpu.h) on every launch path: each case runs on a handle in place and on a twin handle (same
program, controls and translation mode) with separate buffers, over several consecutive calls, and compares the outputs and the whole
final state (registers, accumulator, LFSR, latches, TRAM pointers, counters, flags and ring contents at three instances) bit for bit after
every call, so that wrong state left by one call shows in the next.  The first call is also compared with the oracle.  Every case asserts
the kernel that ran it (fx8010_launch_info.kernel_variant): every kernel is bit-exact, so a routing change would otherwise leave a case
testing some other kernel than the one it names."""
import importlib

import numpy as np
import pytest

import curves_common as ccv
import progs
from conftest import assert_bits_equal
from test_gpu_chain import full_state
from test_gpu_host_curves import shard_views
from test_gpu_parity import CARRIED_PROGS, _tram_prog, make_pair

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

fx = importlib.import_module("fx8010-emulator-core_b200")


def kernel_of(kv):
    """The kernel a launch_info.kernel_variant names."""
    if kv & 128:
        if (kv >> 8) & 0xff == 4 and kv & 4:
            return "tr_stream"
        if (kv >> 8) & 0xff == 4 and kv & 2:
            return "tr_cut"
        return "tr_serial"
    if kv & 8:
        return "im"
    if kv & 32:
        return "short"
    return "generic"


class Twins:
    """`a` runs in place, `b` on separate buffers; `orc` follows the first call."""

    def __init__(self, text, n, ch=1, mode=0, controls=None):
        from oracle import pyoracle as po
        self.n, self.ch = n, ch
        self.prog, self.img, self.orc, self.a = make_pair(fx, po, text, n, ch)
        self.b = fx.Gpu(n, ch)
        self.b.load_program(self.prog)
        for g in (self.a, self.b):
            g.set_option(fx.OPT_TRANSLATE, mode)
        for nm, v in (controls or {}).items():
            for g in (self.a, self.b):
                g.set_controls(self.prog.reg_index(nm), v)
            self.orc.set_register(nm, v)

    def same_state(self, what):
        sa, sb = full_state(self.a, True), full_state(self.b, True)
        for k in sa:
            assert_bits_equal(sa[k], sb[k], f"{what}: {k}")

    def close(self):
        self.a.close(); self.b.close()


def noise(rng, ch, s, n):
    return (1.8 * rng.random((ch, s, n)) - 0.9).astype(np.float32)


# name: (program, instances, channels, translation mode, environment, controls, blocks, kernel)
def _cases():
    rng = np.random.default_rng(77)
    cut = lambda n: {"filter_cutoff": (0.001 + 0.998 * rng.random(n)).astype(np.float32)}
    return {
        "generic": (CARRIED_PROGS["onepole"], 264, 1, 0, {"FX8010_NO_CARRY": "1", "FX8010_NO_SHORT": "1"}, cut(264), [37, 1, 100], "generic"),
        "short": (CARRIED_PROGS["onepole"], 264, 1, 0, {"FX8010_NO_CARRY": "1"}, cut(264), [37, 1, 100], "short"),
        "im_M1": (progs.CFG2_LOG_GAIN, 260, 1, 0, {"FX8010_TUNE_M": "1"}, {}, [37, 1, 100], "im"),
        "im_M8": (progs.CFG2_LOG_GAIN, 260, 1, 0, {"FX8010_TUNE_M": "8"}, {}, [37, 1, 100], "im"),
        "im_two_outputs": (("static a\ninput in_l 0\ninput in_r 1\noutput out_l 0\noutput out_r 1\nmacw a, in_l, 0.75, 0.5\n"
                            "limit out_r, in_r, a, 0.25\ntstneg out_l, in_l, a, 0\nmacintw out_l, out_l, a, 0.75\nend"),
                           260, 2, 0, {"FX8010_TUNE_M": "4"}, {}, [37, 1, 100], "im"),
        "im_carried": (CARRIED_PROGS["onepole"], 264, 1, 0, {}, cut(264), [37, 1, 100], "im"),
        "tram_im": (_tram_prog(size=100), 136, 1, 0, {"FX8010_NO_TSPLIT": "1"}, {}, [150, 1, 33], "im"),
        "tram_im_tsplit": (_tram_prog(size=700, two=(0, 150)), 136, 1, 0, {"FX8010_TUNE_K": "2", "FX8010_TUNE_M": "16"}, {}, [450, 1, 64], "im"),
        "tr_serial_cfg4": (progs.CFG4_ONEPOLE, 256, 1, 2, {"FX8010_TR_RECUR": "1"}, cut(256), [37, 1, 100], "tr_serial"),
        "tr_stream_4096": (progs.CFG2_LOG_GAIN, 4096, 1, 2, {}, {"volume": rng.random(4096).astype(np.float32)}, [64, 1, 37], "tr_stream"),
        "tr_stream_332": (progs.CFG2_LOG_GAIN, 332, 1, 2, {}, {"volume": rng.random(332).astype(np.float32)}, [64, 1, 37], "tr_stream"),
        "tr_cut_100": (progs.cfg3_delay(100), 256, 1, 2, {}, {}, [250, 1, 37], "tr_cut"),
        "tr_cut_8192": (progs.cfg3_delay(8192), 256, 1, 2, {}, {}, [8192 + 300, 1, 100], "tr_cut"),
    }


CASES = _cases()


@pytest.mark.parametrize("name", sorted(CASES))
def test_device_calls_in_place(name, monkeypatch):
    """process_batch with d_out == d_in, against a twin on separate buffers; three calls of ragged lengths."""
    text, n, ch, mode, env, ctl, blocks, kernel = CASES[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    t = Twins(text, n, ch, mode, ctl)
    rng = np.random.default_rng(5)
    try:
        for b, s in enumerate(blocks):
            x = noise(rng, ch, s, n)
            d_io = torch.from_numpy(x).cuda()
            d_x, d_y = d_io.clone(), torch.full_like(d_io, 7.0)
            torch.cuda.synchronize()
            t.a.process_device(d_io, d_io, s)
            kv = t.a.launch_info().kernel_variant
            t.b.process_device(d_x, d_y, s)
            torch.cuda.synchronize()
            assert kernel_of(kv) == kernel and kernel_of(t.b.launch_info().kernel_variant) == kernel, (name, hex(kv), t.a.translate_status())
            y = d_io.cpu().numpy()
            assert_bits_equal(y, d_y.cpu().numpy(), f"{name} call {b} outputs")
            if b == 0:
                assert_bits_equal(y, t.orc.process(x), f"{name} call {b} against the oracle")
            t.same_state(f"{name} after call {b}")
    finally:
        t.close()


@pytest.mark.parametrize("name,n,mode,kernel", [("cfg2_instance", 4096, 2, "tr_stream"), ("delay_fb", 256, 2, "tr_cut"),
                                                ("cfg4_cutoff", 256, 2, "tr_serial")])
def test_curve_calls_in_place(name, n, mode, kernel):
    """process_batch_curves (device values) and process_batch_host_curves (host values) in place."""
    text, ch, cv = ccv.programs()[name]
    t = Twins(text, n, ch, mode)
    regs, bcast = [t.prog.reg_index(r) for r, _ in cv], [b for _, b in cv]
    rng = np.random.default_rng(9)
    try:
        for b, s in enumerate([260, 1, 99]):
            x = noise(rng, ch, s, n)
            vals = [ccv.make_curve(name, r, bc, s, n, rng) for r, bc in cv]
            d_v = [torch.from_numpy(v).cuda() for v in vals]
            d_io = torch.from_numpy(x).cuda()
            d_x, d_y = d_io.clone(), torch.empty_like(d_io)
            torch.cuda.synchronize()
            if b % 2 == 0:             # device curves
                t.a.process_device_curves(d_io, d_io, s, list(zip(regs, d_v, bcast)))
                kv = t.a.launch_info().kernel_variant
                torch.cuda.synchronize()
                got = d_io.cpu().numpy()
            else:                      # host curves, out == in
                got = x.copy()
                t.a.process_host_curves(got, list(zip(regs, vals, bcast)), out=got)
                kv = t.a.launch_info().kernel_variant
            t.b.process_device_curves(d_x, d_y, s, list(zip(regs, d_v, bcast)))
            torch.cuda.synchronize()
            assert kv & fx.VARIANT_CURVES and kernel_of(kv) == kernel, (name, hex(kv), t.a.translate_status_curves())
            assert_bits_equal(got, d_y.cpu().numpy(), f"{name} call {b} outputs")
            if b == 0:
                assert_bits_equal(got, ccv.oracle_stepped(t.orc, x, list(zip(regs, vals, bcast)), s), f"{name} against the oracle")
            t.same_state(f"{name} curves after call {b}")
    finally:
        t.close()


@pytest.mark.parametrize("mode,kernel", [(2, "tr_stream"), (0, "im")])
def test_fused_blocks_in_place(mode, kernel):
    """process_blocks over 32 blocks, each d_out[b] == d_in[b]: one launch takes them all."""
    n, s, nb = 4096, 64, 32
    t = Twins(progs.CFG2_LOG_GAIN, n, 1, mode, {"volume": np.random.default_rng(3).random(n).astype(np.float32)})
    rng = np.random.default_rng(4)
    try:
        for call in range(2):
            xs = [noise(rng, 1, s, n) for _ in range(nb)]
            d_io = [torch.from_numpy(x).cuda() for x in xs]
            d_x = [d.clone() for d in d_io]
            d_y = [torch.empty_like(d) for d in d_io]
            torch.cuda.synchronize()
            before = t.a.launch_info().kernel_launches
            t.a.process_blocks(d_io, d_io, s)
            info = t.a.launch_info()
            t.b.process_blocks(d_x, d_y, s)
            torch.cuda.synchronize()
            assert kernel_of(info.kernel_variant) == kernel and info.last_fused_blocks == nb and info.kernel_launches - before == 1, \
                (hex(info.kernel_variant), info.last_fused_blocks, info.kernel_launches - before)
            for b in range(nb):
                y = d_io[b].cpu().numpy()
                assert_bits_equal(y, d_y[b].cpu().numpy(), f"call {call} block {b}")
                if call == 0:
                    assert_bits_equal(y, t.orc.process(xs[b]), f"block {b} against the oracle")
            t.same_state(f"fused blocks after call {call}")
    finally:
        t.close()


@pytest.mark.parametrize("how", ["pageable", "pinned_async", "slice8", "slice24"])
def test_host_buffers_in_place(how, monkeypatch):
    """process_batch_host with out == in: pageable, page-locked with the _async form, and the _slice form (columns 20.. of a block
    300 wide) with sub-blocks of 8 and 24 periods, so the pipeline copies many pieces in and out of one buffer."""
    n, wide, lo = 256, 300, 20
    if how.startswith("slice"):
        monkeypatch.setenv("FX8010_TUNE_SUB", how[5:])
    t = Twins(progs.CFG2_LOG_GAIN, n, 1, 2, {"volume": np.random.default_rng(6).random(n).astype(np.float32)})
    L = fx.gpu_lib()
    rng = np.random.default_rng(7)
    owners = []
    try:
        for b, s in enumerate([96, 1, 50]):
            x = noise(rng, 1, s, n)
            if how == "pageable":
                got = x.copy()
                t.a.process_host(got, out=got)
            elif how == "pinned_async":
                got, owner = fx.pinned_array(x.shape)
                owners.append(owner)
                got[...] = x
                t.a.process_host_ptr(got.ctypes.data, got.ctypes.data, s, wait=False)
                t.a.synchronize()
            else:
                big = np.full((1, s, wide), 7.0, np.float32)
                big[:, :, lo:lo + n] = x
                p = big.ctypes.data + 4 * lo
                assert L.fx8010_gpu_process_batch_host_slice(t.a.h, p, p, s, wide, 1) == 0
                assert (big[:, :, :lo] == 7.0).all() and (big[:, :, lo + n:] == 7.0).all(), "columns outside the slice were written"
                got = np.ascontiguousarray(big[:, :, lo:lo + n])
            assert kernel_of(t.a.launch_info().kernel_variant) == "tr_stream", hex(t.a.launch_info().kernel_variant)
            assert_bits_equal(got, t.b.process_host(x), f"{how} call {b}")
            if b == 0:
                assert_bits_equal(got, t.orc.process(x), f"{how} against the oracle")
            t.same_state(f"{how} after call {b}")
    finally:
        t.close()


def executor_in_place(devices, n, text, ctl_name=None):
    """fx8010_multi_process_batch_host with out == in against a twin executor; every shard's state against the twin's shard.  cfg2 takes
    the translated streaming kernel on a shard whose instance count is a multiple of 4 and an interpreter kernel elsewhere; cfg4 the
    instruction-major kernel."""
    prog = fx.Program(text)
    m, twin = fx.MultiGpu(devices, n), fx.MultiGpu(devices, n)
    rng = np.random.default_rng(12)
    try:
        for e in (m, twin):
            e.load_program(prog)
            e.set_option(fx.OPT_TRANSLATE, 2)
        if ctl_name:
            v = (0.001 + 0.998 * rng.random(n)).astype(np.float32)
            for e in (m, twin):
                e.set_controls(prog.reg_index(ctl_name), v)
        for b, s in enumerate([200, 1, 57]):
            x = noise(rng, 1, s, n)
            got = x.copy()
            m.process_host(got, out=got)
            assert_bits_equal(got, twin.process_host(x), f"executor on {devices} call {b}")
            for (sa, lo, hi), (sb, _, _) in zip(shard_views(fx, m), shard_views(fx, twin)):
                want = {"im"} if ctl_name else {"im", "short", "generic"} if (hi - lo) % 4 else {"tr_stream"}
                kv = sa.launch_info().kernel_variant
                assert kernel_of(kv) in want and kernel_of(kv) == kernel_of(sb.launch_info().kernel_variant), (devices, lo, hi, hex(kv))
                fa, fb = full_state(sa, True), full_state(sb, True)
                for k in fa:
                    assert_bits_equal(fa[k], fb[k], f"executor on {devices} call {b} shard {lo}..{hi} {k}")
    finally:
        m.close(); twin.close(); prog.close()


def test_executor_in_place_three_uneven_shards():
    """Three shards of device 0: 1 009 instances of cfg2 (336, 336, 337) and 1 000 of cfg4 (333, 333, 334)."""
    executor_in_place([0, 0, 0], 1009, progs.CFG2_LOG_GAIN)
    executor_in_place([0, 0, 0], 1000, progs.CFG4_ONEPOLE, "filter_cutoff")


def test_executor_in_place_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU on this machine")
    executor_in_place([0, 1], 1000, progs.CFG2_LOG_GAIN)
    executor_in_place([0, 1], 1002, progs.CFG4_ONEPOLE, "filter_cutoff")


def test_facade_in_place():
    """The facade's processBlock (host buffers) and FX8010Chain::processBlockDevice with out == in, against separate buffers."""
    n, s = 4096, 128
    H = fx.host_lib()
    objs = [fx.Program(progs.CFG2_LOG_GAIN, instances=n) for _ in range(2)]
    for o in objs:
        o.set_translation(2)
    rng = np.random.default_rng(13)
    x = noise(rng, 1, s, n)
    got = x.copy()
    assert H.fx8010_host_process_block(objs[0].h, got.ctypes.data, got.ctypes.data, s) == 0
    assert_bits_equal(got, objs[1].process_block(x), "processBlock in place")
    texts = [progs.CFG2_LOG_GAIN, progs.CFG1A_TESTCODE]
    chains = []
    for _ in range(2):
        cobj = [fx.Program(tx, instances=n) for tx in texts]
        for o in cobj:
            o.set_translation(2)
        chains.append((cobj, cobj[0].chain(cobj[1:])))
    try:
        for b in range(2):
            d_io = torch.from_numpy(noise(rng, 1, s, n)).cuda()
            d_x, d_y = d_io.clone(), torch.empty_like(d_io)
            chains[0][1](d_io, d_io, s)
            chains[1][1](d_x, d_y, s)
            torch.cuda.synchronize()
            assert_bits_equal(d_io.cpu().numpy(), d_y.cpu().numpy(), f"facade chain call {b}")
    finally:
        for cobj, pc in chains:
            pc.close()
            for o in cobj:
                o.close()
        for o in objs:
            o.close()
