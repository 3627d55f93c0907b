"""Shared by tests/test_gpu_kernel_cache.py: the programs whose translated kernels go through the kernel cache, and one worker process that
runs them and reports, as one JSON line, what the first call ran on, whether the outputs and final state match the oracle, and the
process-wide cache counters.  The counters belong to the process, so every case runs in a fresh one:

    python tests/kernel_cache_common.py '{"programs": ["cfg2"], "mode": 1}'       (environment: FX8010_KERNEL_CACHE, FX8010_NVRTC, ...)
"""
from __future__ import annotations

import importlib
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [HERE, os.path.dirname(HERE)]
import curves_common as cc  # noqa: E402
import progs  # noqa: E402

VARIANT_TRANSLATED = 128


def programs():
    """name -> (text, instances, samples per call, [(curve register name, broadcast)]), one per kind of translated kernel."""
    return {
        "cfg2": (progs.CFG2_LOG_GAIN, 4096, 64, []),                                    # streaming kernel (kind 1)
        "cfg3_1000": (progs.cfg3_delay(1000), 1024, 256, []),                           # streaming kernel cut along time (kind 2)
        "cfg4_curve": (progs.CFG4_ONEPOLE, 1024, 128, [("filter_cutoff", False)]),      # serial kernel with a control curve
        "cfg5_512": (progs.cfg5_allops(), 1024, 64, []),                                # serial kernel, 512 instructions
    }


def _image(po, prog):
    return po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())


def run_program(fx, po, torch, name, mode, calls=2, rng=None):
    """Runs `calls` blocks of program `name` on a fresh handle in translation mode `mode`; returns what the first call ran on and
    whether every output and the final state are bit-identical to the oracle."""
    text, n, s, cv = programs()[name]
    rng = rng or np.random.default_rng(sum(map(ord, name)))
    prog = fx.Program(text)
    assert prog.loaded, prog.errors()
    orc = po.Oracle(_image(po, prog), n, 1)
    gpu = fx.Gpu(n, 1, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, mode)
    regs = [prog.reg_index(r) for r, _ in cv]
    bcast = [b for _, b in cv]
    first = None
    ok = True
    t0 = time.perf_counter()
    for k in range(calls):
        x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
        d_x = torch.from_numpy(x).cuda()
        d_y = torch.empty_like(d_x)
        if cv:
            vals = [cc.make_curve(name, r, b, s, n, rng) for (r, b) in cv]
            d_v = [torch.from_numpy(v).cuda() for v in vals]
            torch.cuda.synchronize()
            gpu.process_device_curves(d_x, d_y, s, list(zip(regs, d_v, bcast)))
            ref = cc.oracle_stepped(orc, x, list(zip(regs, vals, bcast)), s)
        else:
            torch.cuda.synchronize()
            gpu.process_device(d_x, d_y, s)
            ref = orc.process(x)
        gpu.synchronize()
        y = d_y.cpu().numpy()
        if first is None:
            status = gpu.translate_status_curves() if cv else gpu.translate_status()
            first = {"variant": int(gpu.launch_info().kernel_variant), "state": int(status["state"]), "ms": (time.perf_counter() - t0) * 1e3}
        ok = ok and np.array_equal(y.view(np.uint32), ref.view(np.uint32))
    ok = ok and np.array_equal(gpu.registers().view(np.uint32), orc.registers.view(np.uint32)) and np.array_equal(gpu.counts(), orc.counts)
    acc, lfsr, latch, ptrs = gpu.scalars()
    ok = ok and np.array_equal(acc.view(np.uint64), orc.acc.view(np.uint64)) and np.array_equal(ptrs, orc.tram_ptrs)
    gpu.close()
    prog.close()
    first["bit_exact"] = bool(ok)
    first["curves"] = bool(cv)
    return first


def unique_cfg2(tag: int) -> str:
    """cfg2 with one more literal that makes its source new to every cache (as tests/test_gpu_curves.py does)."""
    gain = 0.5 + (tag % 1000003) / 4e6
    return progs.CFG2_LOG_GAIN.replace("macs out_l, 0, a, volume", f"macs a, 0, a, {gain:.6f}\nmacs out_l, 0, a, volume")


def run_multi(fx, po, devices, mode, tag, n=3 * 4096, s=64):
    """The multi-GPU executor over `devices` (3 shards on one device: [0, 0, 0]) on a program text no cache has seen; calls until every
    shard runs translated (mode 1) and compares every output with the oracle."""
    prog = fx.Program(unique_cfg2(tag))
    assert prog.loaded, prog.errors()
    orc = po.Oracle(_image(po, prog), n, 1)
    m = fx.MultiGpu(devices, n, 1)
    m.load_program(prog)
    m.set_option(fx.OPT_TRANSLATE, mode)
    rng = np.random.default_rng(tag % 65536)
    ok, calls = True, 0
    t0 = time.perf_counter()
    t_translated = None
    while calls < 400:
        x = (1.8 * rng.random((1, s, n)) - 0.9).astype(np.float32)
        y = m.process_host(x)
        calls += 1
        ok = ok and np.array_equal(y.view(np.uint32), orc.process(x).view(np.uint32))
        if fx.kernel_cache_stats()["nvrtc_compiles"] and all_translated(fx, m):
            t_translated = (time.perf_counter() - t0) * 1e3
            break
        time.sleep(0.005)
    ok = ok and np.array_equal(m.registers().view(np.uint32), orc.registers.view(np.uint32))
    m.close()
    prog.close()
    return {"bit_exact": bool(ok), "calls": calls, "ms_to_translated": t_translated}


def all_translated(fx, m):
    import ctypes as C
    for g in range(m.L.fx8010_multi_num_shards(m.h)):
        h = m.L.fx8010_multi_shard(m.h, g, None, None)
        st = C.c_int()
        m.L.fx8010_gpu_translate_status(h, C.byref(st), None, None, None, 0)
        if st.value != 2:
            return False
    return True


def main():
    args = json.loads(sys.argv[1])
    import torch
    fx = importlib.import_module("fx8010-emulator-core_b200")
    from oracle import pyoracle as po
    if "cache_dir" in args:
        fx.set_kernel_cache_dir(args["cache_dir"])
    out = {"programs": {}}
    for name in args.get("programs", []):
        out["programs"][name] = run_program(fx, po, torch, name, args["mode"], args.get("calls", 2))
    if "multi" in args:
        out["multi"] = run_multi(fx, po, args["multi"], args["mode"], args["tag"])
    out["stats"] = fx.kernel_cache_stats()
    # whether this process can compile at all (probed last: a compile would count in the stats)
    _, cubin = fx.translate_source(fx.Program(progs.CFG2_LOG_GAIN), 1, compile_check=True)
    out["nvrtc_available"] = bool(cubin and cubin > 0)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
