"""Edge cases of test_gpu_parity.py on the translated kernels (FX8010_OPT_TRANSLATE = 2), and the host edits that the translated paths
keep knowledge about: folded registers, the TRAM offsets the time cut reads, the ring positions it derives from the periods launched.

Every call asserts which kernel ran it: the interpreter kernels are bit-exact as well, so a silent fallback would pass a parity check.
  * translated streaming: launch_info bit 7, 4 instances per thread (bits 8..15), bit 2 for a stateless program;
  * translated streaming cut along time: the same on a TRAM program, one launch per `span` periods of the call (ceil(ns / span));
  * translated serial: bit 7, bit 2 clear, one time segment;
  * interpreter: bit 7 clear.
Outputs and the whole state (ring contents at the first, middle and last instance) are compared with the oracle bit for bit.
"""
import itertools
import math

import numpy as np
import pytest

import progs
from conftest import assert_bits_equal
from test_gpu_parity import compare_state, make_pair

pytestmark = pytest.mark.gpu

STREAM, CUT, SERIAL, INTERP = "stream", "cut", "serial", "interp"
_salt = itertools.count(1)


def salted(text):
    """`text` plus an instruction that changes nothing the test looks at but the generated source: every handle of this file compiles
    kernels no other handle has loaded, so the NVRTC compile count shows each rebuild."""
    k = next(_salt)
    return text.replace("\nend", f"\nstatic salt{k}\nmacs salt{k}, 0, 0, {k / 8192:.10f}\nend")


def builds(fx):
    """Kernels the translator had to produce: NVRTC compiles, or loads from a disk kernel cache left by an earlier run."""
    s = fx.kernel_cache_stats()
    return s["nvrtc_compiles"] + s["disk_hits"]


class Pair:
    """A GPU handle in translate mode 2 and its oracle; `call` runs one API call and asserts the kernel that ran it."""

    def __init__(self, fx, po, text, n, channels=1, mode=2, span=None):
        self.fx, self.n, self.c, self.span = fx, n, channels, span
        self.prog, self.img, self.orc, self.gpu = make_pair(fx, po, text, n, channels)
        self.gpu.set_option(fx.OPT_TRANSLATE, mode)

    def close(self):
        self.gpu.close()

    def reg(self, name):
        r = self.prog.reg_index(name)
        assert r >= 0, name
        return r

    def call(self, path, fn, ns=None, launches=None, what="", curves=False):
        before = self.gpu.launch_info().kernel_launches
        out = fn()
        info = self.gpu.launch_info()
        kv, added = info.kernel_variant, info.kernel_launches - before
        st = self.gpu.translate_status_curves() if curves else self.gpu.translate_status()
        tag = f"{what}: expected {path}, kernel_variant {kv:#x}, {added} launches, translator {st}"
        if path == INTERP:
            assert not kv & 128, tag
        else:
            assert kv & 128 and st["state"] == 2, tag
            if path in (STREAM, CUT):
                assert (kv >> 8) & 0xff == 4, tag
            if path == STREAM and self.span is None:
                assert kv & 4, tag
            if path == CUT:
                assert kv & 2 and not kv & 4, tag
                if ns is not None and launches is None:
                    launches = math.ceil(ns / self.span)
            if path == SERIAL:
                assert not kv & 4 and info.last_time_split == 1, tag
        if launches is not None:
            assert added == launches, tag
        return out

    def host(self, path, x, what="", launches=None):
        """process_host on both sides (one internal sub-block for every size used here)."""
        yg = self.call(path, lambda: self.gpu.process_host(x), ns=x.shape[1], launches=launches, what=what)
        assert_bits_equal(yg, self.orc.process(x), what + " outputs")

    def check(self, what):
        compare_state(self.gpu, self.orc, self.img, what, sorted({0, self.n // 2, self.n - 1}))


def noise(rng, c, s, n, amp=0.9):
    return (2 * amp * rng.random((c, s, n)) - amp).astype(np.float32)


# ---- the programs, and which kernel each one reaches ------------------------------------------------------------------------

def _programs():
    rng = np.random.default_rng(4242)
    return {
        # name: (text, instances, path, span of the time cut, environment)
        "cfg2": (progs.CFG2_LOG_GAIN, 256, STREAM, None, {}),
        "skip": (progs.SNIPPETS["skip"], 128, SERIAL, None, {}),
        "cfg3_100": (progs.cfg3_delay(100), 256, CUT, 100, {}),
        "cfg3_1000": (progs.cfg3_delay(1000), 128, CUT, 1000, {}),
        "cfg4": (progs.CFG4_ONEPOLE, 256, SERIAL, None, {"FX8010_TR_RECUR": "1"}),
        "cfg5": (progs.cfg5_allops(n_instr=160), 128, SERIAL, None, {}),
        "random_xtram": (progs.random_program(rng, 40, xtram=True), 96, SERIAL, None, {}),
        # what the route keeps on the interpreter
        "cfg2_n333": (progs.CFG2_LOG_GAIN, 333, INTERP, None, {}),
        "cfg4_plain": (progs.CFG4_ONEPOLE, 256, INTERP, None, {}),
        "cfg3_n254": (progs.cfg3_delay(100), 254, INTERP, None, {}),
    }


PROGRAMS = _programs()


def open_pair(fx, po, name, monkeypatch, n=None):
    text, n0, path, span, env = PROGRAMS[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    p = Pair(fx, po, salted(text), n or n0, span=span)
    if name.startswith("cfg5"):
        rng = np.random.default_rng(3)
        for i in range(4):
            v = rng.random(p.n).astype(np.float32)
            p.gpu.set_controls(p.reg(f"k{i}"), v); p.orc.set_register(f"k{i}", v)
    if name.startswith("cfg4"):
        v = (0.001 + 0.998 * np.arange(p.n) / max(1, p.n - 1)).astype(np.float32)
        p.gpu.set_controls(p.reg("filter_cutoff"), v); p.orc.set_register("filter_cutoff", v)
    return p, path


@pytest.mark.parametrize("name", sorted(PROGRAMS))
def test_blocks_on_the_promised_kernel(fx, po, name, monkeypatch):
    """Ragged blocks (1, a stretch shorter than the span, several spans) through process_host."""
    p, path = open_pair(fx, po, name, monkeypatch)
    rng = np.random.default_rng(1)
    try:
        for s in (1, 37, 1024, 250):
            p.host(path, noise(rng, 1, s, p.n), f"{name} block of {s}")
        p.check(name)
    finally:
        p.close()


@pytest.mark.parametrize("name", ["cfg2", "cfg3_100", "cfg4", "random_xtram", "cfg2_n333"])
def test_null_input_block_is_silence(fx, po, name, monkeypatch):
    """d_in == NULL: INPUT operands read 0.0 — process_batch, and process_blocks with no input list."""
    import torch
    p, path = open_pair(fx, po, name, monkeypatch)
    rng = np.random.default_rng(61)
    try:
        s = 300
        p.host(path, noise(rng, 1, s, p.n), "warm-up block")
        d_out = torch.empty((1, s, p.n), dtype=torch.float32, device="cuda")
        p.call(path, lambda: (p.gpu.process_device(None, d_out, s, None), p.gpu.synchronize(None)), ns=s, what="NULL input")
        assert_bits_equal(d_out.cpu().numpy(), p.orc.process(None, s), "NULL input outputs")
        outs = [torch.empty((1, 64, p.n), dtype=torch.float32, device="cuda") for _ in range(3)]
        launches = 1 if path == STREAM else None      # a stateless program takes the three blocks in one launch
        p.call(path, lambda: (p.gpu.process_blocks(None, outs, 64, None), p.gpu.synchronize(None)), launches=launches, what="NULL block list")
        for b in range(3):
            assert_bits_equal(outs[b].cpu().numpy(), p.orc.process(None, 64), f"NULL block {b}")
        p.check("NULL input")
    finally:
        p.close()


@pytest.mark.parametrize("n", [1, 2, 3, 5, 8])
def test_tiny_instance_counts(fx, po, n, monkeypatch):
    """Fewer instances than a warp: the serial kernel masks its lanes; a stateless program takes the streaming kernel only at N % 4 == 0."""
    rng = np.random.default_rng(20 + n)
    for name in ("cfg2", "random_xtram"):
        p, path = open_pair(fx, po, name, monkeypatch, n=n)
        if name == "cfg2" and n % 4:
            path = INTERP
        try:
            v = rng.random(n).astype(np.float32)
            if name == "cfg2":
                p.gpu.set_controls(p.reg("volume"), v); p.orc.set_register("volume", v)
            for s in (9, 1, 30):
                p.host(path, noise(rng, 1, s, n), f"{name} n={n} block of {s}")
            p.check(f"{name} n={n}")
        finally:
            p.close()


def test_zero_samples_and_long_batch(fx, po, monkeypatch):
    """ns == 0 launches nothing; 5 000 periods run in one serial launch."""
    import torch
    p, path = open_pair(fx, po, "cfg4", monkeypatch, n=8)
    rng = np.random.default_rng(30)
    try:
        p.host(SERIAL, noise(rng, 1, 4, 8), "first block")
        d_out = torch.empty((1, 4, 8), dtype=torch.float32, device="cuda")
        p.call(SERIAL, lambda: p.gpu.process_device(None, d_out, 0, None), launches=0, what="zero periods")
        p.host(SERIAL, noise(rng, 1, 5000, 8), "5000-period block", launches=1)
        p.check("long batch")
    finally:
        p.close()


@pytest.mark.parametrize("name", ["testcode", "cfg2", "onepole", "delay", "dynsel", "folded_static"])
def test_control_events_inside_a_batch(fx, po, name, monkeypatch):
    """A control changes every 8 periods inside one process_batch_events call, broadcast and per instance.  `folded_static`: the
    register is a never-written STATIC the translation folded — the first event voids the kernel between two pieces of the call
    and it is rebuilt once; `dynsel`: the control is a LOG table selector."""
    import torch
    rng = np.random.default_rng(41)
    n = 300
    text, ctl, path, span = {
        "testcode": (progs.CFG1A_TESTCODE, "volume", STREAM, None),
        "cfg2": (progs.CFG2_LOG_GAIN, "volume", STREAM, None),
        "onepole": (progs.CFG4_ONEPOLE, "filter_cutoff", SERIAL, None),
        "delay": ("static a\nstatic rd\ncontrol fb = 0.5\ninput in_l 0\noutput out_l 0\nitramsize 150 \nidelay read, rd, at, 0\n"
                  "macs a, in_l, rd, fb\nidelay write, a, at, 0\nmacs out_l, in_l, rd, fb\nend", "fb", CUT, 150),
        "dynsel": ("static a\ninput in_l 0\ncontrol sel = 3\noutput out_l 0\nlog a, in_l, sel, 0\nmacs out_l, 0, a, 0.5\nend", "sel", STREAM, None),
        "folded_static": ("static g = 0.5\nstatic a\ninput in_l 0\noutput out_l 0\nmacs a, 0, in_l, g\nskip ccr, ccr, 6, 1\n"
                          "macsn a, a, g, g\nmacs out_l, a, g, 0.25\nend", "g", SERIAL, None),
    }[name]
    if name == "onepole":
        monkeypatch.setenv("FX8010_TR_RECUR", "1")
    p = Pair(fx, po, salted(text), n, span=span)
    try:
        reg = p.reg(ctl)
        s_total = 100
        p.host(path, noise(rng, 1, 50, n), "first block")
        x = noise(rng, 1, s_total, n)
        events = []
        for s0 in range(0, s_total, 8):
            if name == "dynsel":
                v = float(rng.integers(0, 32)) if (s0 // 8) % 2 else rng.integers(0, 32, n).astype(np.float32)
            else:
                v = float(rng.random()) if (s0 // 8) % 3 == 0 else rng.random(n).astype(np.float32)
            events.append((s0 + 3, reg, v))
        events.insert(3, (events[2][0], reg, 0.125))             # two changes at the same period: the later one wins
        yo = np.zeros_like(x)
        bounds = sorted({0} | {e[0] for e in events} | {s_total})
        for a, b in zip(bounds[:-1], bounds[1:]):
            for (s, r, v) in events:
                if s == a:
                    p.orc.set_register(r, np.full(n, v, np.float32) if np.isscalar(v) else v)
            yo[:, a:b] = p.orc.process(np.ascontiguousarray(x[:, a:b]))
        d_in = torch.from_numpy(x).cuda()
        d_out = torch.empty_like(d_in)
        st = torch.cuda.Stream()
        b0 = builds(fx)
        p.call(path, lambda: (p.gpu.process_device_events(d_in, d_out, s_total, events, st.cuda_stream), p.gpu.synchronize(st.cuda_stream)),
               what=f"{name} events")
        assert builds(fx) - b0 == (1 if name == "folded_static" else 0), "rebuilds during the events call"
        assert_bits_equal(d_out.cpu().numpy(), yo, f"{name} outputs with control events")
        p.host(path, noise(rng, 1, 40, n), "block after the events")
        p.check(f"{name} events")
    finally:
        p.close()


@pytest.mark.parametrize("n,s", [(300, 77), (64, 1024), (4, 5)])
def test_planar_buffers(fx, po, n, s):
    """[channel][instance][sample] device buffers: the transposes on the caller's stream feed the translated streaming launch."""
    import torch
    rng = np.random.default_rng(42)
    text = "static a\ninput in_l 0\ninput in_r 1\noutput out_l 0\noutput out_r 1\nmacs a, in_l, in_l, 0.5\nmacs out_l, a, 0.25, 0.5\nmacs out_r, in_r, a, 0.5\nend"
    p = Pair(fx, po, salted(text), n, channels=2)
    try:
        for k in range(2):
            x = noise(rng, 2, s, n)
            yo = p.orc.process(x)
            d_in = torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 1))).cuda()
            d_out = torch.empty_like(d_in)
            p.call(STREAM, lambda: (p.gpu.process_device_planar(d_in, d_out, s, None), p.gpu.synchronize(None)), launches=3, what=f"planar {k}")
            assert_bits_equal(d_out.cpu().numpy().transpose(0, 2, 1), yo, "planar outputs")
        p.check("planar")
    finally:
        p.close()


@pytest.mark.parametrize("name", ["cfg3_100", "random_xtram"])
def test_async_host_batches_chain_in_order(fx, po, name, monkeypatch):
    """Queued host batches on the internal streams keep their order and state; a device call afterwards waits for them."""
    import torch
    p, path = open_pair(fx, po, name, monkeypatch)
    rng = np.random.default_rng(40)
    try:
        s, calls = 300, 5
        ins = [fx.pinned_array((1, s, p.n)) for _ in range(calls)]
        outs = [fx.pinned_array((1, s, p.n)) for _ in range(calls)]
        for a, _ in ins:
            a[...] = noise(rng, 1, s, p.n)
        for (a, _), (b, _) in zip(ins, outs):
            p.call(path, lambda: p.gpu.process_host_ptr(a.ctypes.data, b.ctypes.data, s, wait=False), ns=s, what="async call")
        d_x = torch.from_numpy(ins[0][0].copy()).cuda(); d_y = torch.empty_like(d_x)
        torch.cuda.synchronize()
        p.call(path, lambda: (p.gpu.process_device(d_x, d_y, s, None), p.gpu.synchronize(None)), ns=s, what="device call after async")
        for k, ((a, _), (b, _)) in enumerate(zip(ins, outs)):
            assert_bits_equal(b, p.orc.process(a), f"async call {k}")
        assert_bits_equal(d_y.cpu().numpy(), p.orc.process(ins[0][0]), "device call after async")
        p.check("async")
    finally:
        p.close()


@pytest.mark.parametrize("name", ["cfg2", "cfg3_100"])
def test_broadcast_input(fx, po, name, monkeypatch):
    """One input signal for every instance, spread on the device before the translated launch."""
    p, path = open_pair(fx, po, name, monkeypatch)
    rng = np.random.default_rng(43)
    try:
        for s in (300, 64):
            x = (1.8 * rng.random((1, s)) - 0.9).astype(np.float32)
            y = p.call(path, lambda: p.gpu.process_host_broadcast(x), what="broadcast input")
            assert_bits_equal(y, p.orc.process(np.repeat(x[:, :, None], p.n, axis=2)), "broadcast input outputs")
        p.check("broadcast input")
    finally:
        p.close()


def test_state_roundtrip_checkpoint(fx, po, monkeypatch):
    """get_state -> new handle -> set_registers / set_scalars / set_tram: the translated serial kernel of the second handle continues."""
    p, path = open_pair(fx, po, "random_xtram", monkeypatch)
    rng = np.random.default_rng(5)
    gpu2 = fx.Gpu(p.n, 1)
    try:
        p.host(SERIAL, noise(rng, 1, 64, p.n), "first handle")
        gpu2.load_program(p.prog)
        gpu2.set_option(fx.OPT_TRANSLATE, 2)
        gpu2.set_registers(p.gpu.registers())
        gpu2.set_scalars(*p.gpu.scalars())
        d = p.gpu.dims()
        for i in range(p.n):
            if d.itram_size: gpu2.set_tram(0, i, p.gpu.tram(0, i))
            if d.xtram_size: gpu2.set_tram(1, i, p.gpu.tram(1, i))
        p.gpu.close()
        p.gpu = gpu2
        p.host(SERIAL, noise(rng, 1, 64, p.n), "resumed")
        assert_bits_equal(gpu2.registers(), p.orc.registers, "resumed registers")       # (instruction counters are not part of a checkpoint)
        assert_bits_equal(gpu2.scalars()[3], p.orc.tram_ptrs, "resumed pointers")
        assert_bits_equal(gpu2.tram(1, p.n - 1), p.orc.tram(1, p.n - 1), "resumed xTRAM")
    finally:
        p.close()


@pytest.mark.parametrize("order", ["rw", "wr"])
def test_host_written_pointers_turn_the_time_cut_off(fx, po, order):
    """TRAM pointers written through set_scalars (per instance, or all about to wrap): the ring positions are no longer the periods
    launched, so a delay line leaves the time-cut streaming kernel for the interpreter; before that it was cut along time."""
    from test_gpu_parity import _tram_prog
    rng = np.random.default_rng(51)
    n, size = 192, 400
    text = _tram_prog(size, order=order, roff="150" if order == "wr" else "0", woff="2" if order == "wr" else "150")
    span = 152 if order == "wr" else 150
    p = Pair(fx, po, salted(text), n, span=span)
    try:
        p.host(CUT, noise(rng, 1, 700, n), "before the pointers are written")
        ptrs = p.gpu.scalars()[3].copy()
        ptrs[0] = rng.integers(0, size, n)
        ptrs[1] = (ptrs[0] + rng.integers(0, size, n)) % size
        p.gpu.set_scalars(ptrs=ptrs); p.orc.tram_ptrs[...] = ptrs
        ring = (rng.random((n, size)) - 0.5).astype(np.float32)
        for i in range(n):
            p.gpu.set_tram(0, i, ring[i]); p.orc.set_tram(0, i, ring[i])
        for s in (1, 70, 700):
            p.host(INTERP, noise(rng, 1, s, n), f"per-instance pointers, {order}")
        p.check("per-instance pointers")
    finally:
        p.close()


def test_full_size_xtram(fx, po):
    """A 4 MiB ring per instance: cut along time while the pointers are pristine, then pointers about to wrap from the host."""
    rng = np.random.default_rng(32)
    text = ("static a\nstatic rd\ninput in_l 0\noutput out_l 0\nxtramsize 1048576 \nxdelay read, rd, at, 0\nmacs a, in_l, rd, 0.5\n"
            "xdelay write, a, at, 0\nxdelay read, rd, at, 5\nmacs out_l, in_l, rd, 0.5\nend")
    p = Pair(fx, po, salted(text), 8)
    try:
        p.host(SERIAL, noise(rng, 1, 40, 8), "pristine pointers", launches=1)
        ptr = p.gpu.scalars()[3].copy(); ptr[2] = 1048570; ptr[3] = 1048572
        p.gpu.set_scalars(ptrs=ptr); p.orc.tram_ptrs[:] = ptr
        p.host(SERIAL, noise(rng, 1, 40, 8), "pointers about to wrap")
        compare_state(p.gpu, p.orc, p.img, "xtram", tram_instances=(0, 7))
    finally:
        p.close()


def test_end_skipped_programs_stay_on_the_interpreter(fx, po):
    """A program whose END may be skipped repeats the period (rule U9, cap of 8 passes): the translator declines it, the interpreter
    runs it, and the cap flag is the oracle's."""
    forever = "static a\noutput out_l 0\nmacs a, 0, 0.5, 0.5\nmacs out_l, a, 0.1, 0.1\nskip ccr, ccr, 2, 1\nend"
    for text in (progs.END_SKIPPED_WRAP, forever):
        p = Pair(fx, po, text, 64)
        try:
            yg = p.call(INTERP, lambda: p.gpu.process_host(None, 40), what="END skipped")
            assert_bits_equal(yg, p.orc.process(None, 40), "END skipped outputs")
            st = p.gpu.translate_status()
            assert st["state"] == -1 and "END" in st["message"], st
            p.check("END skipped")
            assert (p.gpu.flags() & fx.RT_END_SKIPPED_CAP) == (p.orc.flags & fx.RT_END_SKIPPED_CAP)
        finally:
            p.close()


def test_literal_register_overwritten_through_api(fx, po):
    """The LOG selector '3' and the MACS addend '0' are immediates of the translated streaming kernel; per-instance values void it
    (one rebuild), and a later broadcast to the same register needs none (it is no longer folded)."""
    rng = np.random.default_rng(33)
    n = 128
    p = Pair(fx, po, salted(progs.CFG1B_LOGTUBE), n)
    try:
        x = noise(rng, 1, 20, n)
        p.host(STREAM, x, "before")
        b0 = builds(fx)
        sel = rng.integers(0, 32, n).astype(np.float32); add = (0.2 * rng.random(n)).astype(np.float32)
        for name, v in (("3", sel), ("0", add)):
            p.gpu.set_controls(p.reg(name), v); p.orc.set_register(name, v)
        p.host(STREAM, x, "per-instance literals")
        assert builds(fx) - b0 == 1
        p.gpu.set_controls(p.reg("3"), [7.0], broadcast=True); p.orc.set_register("3", np.full(n, 7.0, np.float32))
        p.host(STREAM, x, "broadcast literal")
        assert builds(fx) - b0 == 1
        p.check("literals")
    finally:
        p.close()


@pytest.mark.parametrize("which", ["write_only", "read_only", "both"])
def test_tram_written_only_or_read_only(fx, po, which):
    """A ring with only a WRITE constrains nothing but its size (cut along time, span = ring size); a ring nobody writes gives no span
    (the interpreter), and its contents come from the checkpoint API."""
    text, path, span = {
        "write_only": ("static a\ninput in_l 0\noutput out_l 0\nitramsize 150 \nmacs a, in_l, 0.5, 0.5\nidelay write, a, at, 3\n"
                       "macs out_l, a, in_l, 0.25\nend", INTERP, None),
        "read_only": ("static rd\ninput in_l 0\noutput out_l 0\nxtramsize 333 \nxdelay read, rd, at, 40\nmacs out_l, rd, in_l, 0.25\nend", INTERP, None),
        "both": ("static a\nstatic rd\ninput in_l 0\noutput out_l 0\nitramsize 150 \nxtramsize 333 \nxdelay read, rd, at, 40\nmacs a, in_l, rd, 0.5\n"
                 "idelay write, a, at, 3\nmacs out_l, a, in_l, 0.25\nend", CUT, 150),
    }[which]
    rng = np.random.default_rng(71)
    n = 100
    p = Pair(fx, po, salted(text), n, span=span)
    try:
        d = p.gpu.dims()
        if d.xtram_size:
            for i in range(n):
                ring = (rng.random(d.xtram_size) - 0.5).astype(np.float32)
                p.gpu.set_tram(1, i, ring); p.orc.set_tram(1, i, ring)
        for s in (1, 90, 64, 500):
            p.host(path, noise(rng, 1, s, n), f"{which} block of {s}")
        compare_state(p.gpu, p.orc, p.img, "one-sided TRAM", (0, 50, n - 1))
    finally:
        p.close()


@pytest.mark.parametrize("name", ["cfg2", "skip", "cfg3_100", "random_xtram"])
def test_trace_then_plain_call(fx, po, name, monkeypatch):
    """A trace runs on the interpreter; the plain call after it is translated again, and a delay line's ring positions (derived from the
    periods launched, the traced ones included) continue where the trace left them."""
    p, path = open_pair(fx, po, name, monkeypatch)
    rng = np.random.default_rng(50)
    try:
        p.host(path, noise(rng, 1, 130, p.n), "before the trace")
        x = noise(rng, 1, 9, p.n)
        out, _ = p.call(INTERP, lambda: p.gpu.trace(x, 5), what="trace")
        assert_bits_equal(out, p.orc.process(x), "trace outputs")
        for s in (250, 7):
            p.host(path, noise(rng, 1, s, p.n), f"after the trace, {s}")
        p.check("after trace")
    finally:
        p.close()


# ---- mixed NULL / non-NULL input lists ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["cfg2", "cfg3_100", "cfg4", "cfg4_plain"])
def test_mixed_null_input_list_is_refused(fx, po, name, monkeypatch):
    """process_blocks with 40 blocks whose inputs mix NULL (block 35, past the first fused group of 32) and device buffers: refused with
    FX8010_ERR_ARG on every path — fused streaming, time-cut split, translated serial, interpreter — with nothing launched and the
    registers, counters and pointers as they were."""
    import torch
    p, path = open_pair(fx, po, name, monkeypatch)
    rng = np.random.default_rng(77)
    try:
        s = 128 if name != "cfg3_100" else 256         # (cfg3: longer than its span, so the call would be split)
        p.host(path, noise(rng, 1, s, p.n), "first block")
        before = (p.gpu.registers(), p.gpu.counts(), p.gpu.scalars()[3], p.gpu.launch_info().kernel_launches)
        xs = [torch.from_numpy(noise(rng, 1, s, p.n)).cuda() for _ in range(40)]
        ys = [torch.zeros_like(v) for v in xs]
        ins = list(xs); ins[35] = None
        with pytest.raises(fx.FxError) as e:
            p.gpu.process_blocks(ins, ys, s, None)
        assert e.value.code == 1
        p.gpu.synchronize(None)
        assert p.gpu.launch_info().kernel_launches == before[3]
        assert_bits_equal(p.gpu.registers(), before[0], "registers after the refused call")
        assert_bits_equal(p.gpu.counts(), before[1], "counters after the refused call")
        assert_bits_equal(p.gpu.scalars()[3], before[2], "pointers after the refused call")
        assert all(float(y.abs().sum()) == 0 for y in ys)
        p.host(path, noise(rng, 1, s, p.n), "block after the refused call")
        p.check("after the refused call")
    finally:
        p.close()


# ---- host edits between two calls of a handle whose translated kernel is loaded ----------------------------------------------------

# A delay line cut along time that holds every kind of register the translation treats differently: a never-written STATIC (folded),
# a CONTROL (never folded), a literal, a LOG selector, and the read and write offsets of the ring (folded, and what the span is
# computed from: read-after-write distance 102, write-after-read 298).
EDIT_PROG = "\n".join(["static g = 0.5", "static a", "static rd", "static t", "control vol = 0.75", "input in_l 0", "output out_l 0",
                       "itramsize 400 ", "idelay read, rd, at, 100", "macs a, in_l, rd, g", "log t, a, 3, 0", "idelay write, a, at, 2",
                       "macs t, t, rd, 0.125", "macs out_l, 0, t, vol", "end"])
KINDS = {  # register: (name, a new broadcast value, per-instance values maker, folded by the translation, offset)
    "static": ("g", 0.25, lambda rng, n: (rng.random(n) - 0.5).astype(np.float32), True, None),
    "control": ("vol", 0.5, lambda rng, n: rng.random(n).astype(np.float32), False, None),
    "literal": ("0.125", 0.375, lambda rng, n: (0.5 * rng.random(n)).astype(np.float32), True, None),
    "selector": ("3", 7.0, lambda rng, n: rng.integers(0, 32, n).astype(np.float32), True, None),
    "read_offset": ("100", 150.0, lambda rng, n: rng.integers(60, 200, n).astype(np.float32), True, "read"),
    "write_offset": ("2", 5.0, lambda rng, n: rng.integers(0, 9, n).astype(np.float32), True, "write"),
}
EDITS = ["bcast_same", "bcast_new", "per_instance", "device", "registers_uniform", "registers_row", "events_bcast", "events_row", "curves"]


def edit_span(kind, value):
    """The span of EDIT_PROG after `kind` holds the one value `value` (None: not one value, no span)."""
    if value is None:
        return None
    r, w = (value if kind == "read_offset" else 100), (value if kind == "write_offset" else 2)
    d = int(r + w) % 400
    span = min(d, 400 - d)
    return span if span >= 64 else None


@pytest.mark.parametrize("kind", sorted(KINDS))
@pytest.mark.parametrize("edit", EDITS)
def test_host_edit_between_calls(fx, po, kind, edit):
    import torch
    name, new, per_inst, folded, offset = KINDS[kind]
    if edit == "curves" and kind not in ("static", "control"):
        pytest.skip("control curves drive CONTROL and STATIC registers only")
    rng = np.random.default_rng(hash((kind, edit)) % 2**32)
    n, s = 256, 1024
    p = Pair(fx, po, salted(EDIT_PROG), n, span=102)
    try:
        reg = p.reg(name)
        p.host(CUT, noise(rng, 1, s, n), "before the edit", launches=11)
        b0 = builds(fx)
        cur = np.float32(p.gpu.registers()[reg, 0])
        uniform = None                      # the one value the register holds after the edit (None: per instance)
        x = noise(rng, 1, s, n)
        d_in, d_out = torch.from_numpy(x).cuda(), torch.zeros((1, s, n), dtype=torch.float32, device="cuda")
        if edit == "bcast_same":
            p.gpu.set_controls(reg, [cur], broadcast=True); uniform = cur
        elif edit in ("bcast_new", "registers_uniform"):
            uniform = np.float32(new)
            if edit == "bcast_new":
                p.gpu.set_controls(reg, [uniform], broadcast=True)
            else:
                regs = p.gpu.registers(); regs[reg] = uniform; p.gpu.set_registers(regs)
            p.orc.set_register(reg, np.full(n, uniform, np.float32))
        elif edit in ("per_instance", "device", "registers_row"):
            v = per_inst(rng, n)
            if edit == "per_instance":
                p.gpu.set_controls(reg, v)
            elif edit == "device":
                p.gpu.set_controls_device(reg, torch.from_numpy(v).cuda(), None)
            else:
                regs = p.gpu.registers(); regs[reg] = v; p.gpu.set_registers(regs)
            p.orc.set_register(reg, v)
        if edit.startswith("events"):
            v = np.float32(new) if edit == "events_bcast" else per_inst(rng, n)
            uniform = v if edit == "events_bcast" else None
            at = 300
            yo = np.zeros_like(x)
            yo[:, :at] = p.orc.process(x[:, :at])
            p.orc.set_register(reg, np.full(n, v, np.float32) if np.isscalar(v) else v)
            yo[:, at:] = p.orc.process(x[:, at:])
            span = edit_span(kind, uniform) if offset else 102
            path = CUT if span else INTERP
            p.call(path, lambda: (p.gpu.process_device_events(d_in, d_out, s, [(at, reg, float(v) if np.isscalar(v) else v)], None),
                                  p.gpu.synchronize(None)), what="events call")
            assert_bits_equal(d_out.cpu().numpy(), yo, "events call outputs")
        elif edit == "curves":
            from curves_common import oracle_stepped
            cv = per_inst(rng, s * n).reshape(s, n)
            yo = oracle_stepped(p.orc, x, [(reg, cv, False)], s)
            d_cv = torch.from_numpy(cv).cuda()
            p.call(CUT, lambda: (p.gpu.process_device_curves(d_in, d_out, s, [(reg, d_cv, False)], None), p.gpu.synchronize(None)),
                   launches=11, what="curves call", curves=True)
            assert_bits_equal(d_out.cpu().numpy(), yo, "curves call outputs")
            assert builds(fx) - b0 == 1, "the curve set's kernel"
            b0 += 1
        else:
            span = edit_span(kind, uniform) if offset else 102
            p.span = span
            p.host(CUT if span else INTERP, x, f"after {edit} on {kind}")
        # the plain call after the edit: rebuilt once when a folded register changed its value, never when it kept it; a time-cut
        # program stays cut while its span is known and falls back to the interpreter when it is not
        changed = edit != "bcast_same" and folded
        span = edit_span(kind, uniform) if offset else 102
        p.span = span
        p.host(CUT if span else INTERP, noise(rng, 1, s, n), f"plain call after {edit} on {kind}")
        want = 1 if changed and (span or not offset) else 0
        assert builds(fx) - b0 == want, f"rebuilds after {edit} on {kind}"
        p.check(f"{edit} on {kind}")
    finally:
        p.close()


@pytest.mark.parametrize("edit", ["scalars_same", "scalars_moved", "tram", "trace"])
def test_host_edit_of_the_rings_between_calls(fx, po, edit):
    """Pointers written through set_scalars (even the values they held) leave the ring positions unknown: the time cut is off.  Ring
    contents written through set_tram, and a trace, keep it."""
    rng = np.random.default_rng(len(edit))
    n, s = 256, 1024
    p = Pair(fx, po, salted(EDIT_PROG), n, span=102)
    try:
        p.host(CUT, noise(rng, 1, s, n), "before the edit", launches=11)
        b0 = builds(fx)
        path = CUT
        if edit.startswith("scalars"):
            ptrs = p.gpu.scalars()[3].copy()
            if edit == "scalars_moved":
                ptrs[:2] = (ptrs[:2] + 3) % 400
            p.gpu.set_scalars(ptrs=ptrs); p.orc.tram_ptrs[...] = ptrs
            path = INTERP
        elif edit == "tram":
            for i in (0, 5, n - 1):
                ring = (rng.random(400) - 0.5).astype(np.float32)
                p.gpu.set_tram(0, i, ring); p.orc.set_tram(0, i, ring)
        else:
            x = noise(rng, 1, 33, n)
            out, _ = p.call(INTERP, lambda: p.gpu.trace(x, 3), what="trace")
            assert_bits_equal(out, p.orc.process(x), "trace outputs")
        for k in range(2):
            p.host(path, noise(rng, 1, s, n), f"plain call {k} after {edit}")
        assert builds(fx) == b0
        p.check(edit)
    finally:
        p.close()
