"""Measures control curves from host memory (fx8010_gpu_process_batch_host_curves and the executor's
fx8010_multi_process_batch_host_curves) against the two ways a host-buffer caller has without them.

    python tests/host_curves_bench.py [--calls 10] [--warmup 2] [--out FILE]

Cases (1 024 periods per block, every buffer page-locked, translator in mode 2):
    cfg4 (one-pole low-pass, 65 536 instances, a per-instance filter_cutoff curve): blocking and asynchronous calls on one GPU, then
         through the executor over every GPU present;
    cfg2 (LOG waveshaper + gain, 4 096 instances, a broadcast volume ramp): blocking, one GPU.

One JSON line per case: milliseconds per block of the curve call (a host clock around `calls` back-to-back calls that ends in a
synchronize: every call blocks, or the asynchronous ones are synchronized once at the end), the PCIe bytes it moves per block,
4 x (inputs + outputs + per-instance curves) x periods x instances, the same block through process_batch_host without curves, and
the same block as the reference driver runs it: one blocking host call per 8 periods with set_controls in between.  Also a bit-exact
check of >= 64 sampled instances of the first curve call against the oracle stepped one period at a time, and the GPU's name and power
limit read in the same run.  Needs a GPU: without one it fails.
"""
import argparse
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
from curves_bench import gpu_identity, oracle_for  # noqa: E402

fx = importlib.import_module("fx8010-emulator-core_b200")
S = 1024
EVERY = 8


def pinned(a, owners):
    p, o = fx.pinned_array(a.shape, a.dtype)
    p[...] = a
    owners.append(o)
    return p


def timed_ms(fn, calls, warmup, sync):
    for _ in range(warmup):
        fn()
    sync()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    sync()
    return (time.perf_counter() - t0) * 1e3 / calls


def run_case(label, text, n, reg_name, bcast, devices, wait, calls, warmup):
    """devices None: one fx8010_gpu handle on device 0; else an executor over `devices`."""
    rng = np.random.default_rng(0x8010)
    owners = []
    prog = fx.Program(text)
    reg = prog.reg_index(reg_name)
    if devices is None:
        h = fx.Gpu(n, 1, 0)
    else:
        h = fx.MultiGpu(devices, n)
    h.load_program(prog)
    h.set_option(fx.OPT_TRANSLATE, 2)
    x = pinned(progs.sine_bank(n, S, rng).reshape(1, S, n), owners)
    y = pinned(np.zeros((1, S, n), np.float32), owners)
    if reg_name == "volume":
        vals = np.linspace(0.05, 1.0, S, dtype=np.float32)
    else:
        vals = cc.make_curve("cfg4", reg_name, bcast, S, n, rng)
    v = pinned(vals, owners)
    curves = [(reg, v, bcast)]

    # parity: the first call from the freshly loaded state, >= 64 sampled instances against the oracle stepped per period
    h.process_host_curves(x, curves, out=y)
    pick = np.unique(np.concatenate([[0, n - 1], rng.choice(n, 70, replace=False)]))
    orc = oracle_for(text, len(pick))
    want = cc.oracle_stepped(orc, np.ascontiguousarray(x[:, :, pick]), [(reg, vals if bcast else np.ascontiguousarray(vals[:, pick]), bcast)], S)
    parity = bool(np.array_equal(y[:, :, pick].view(np.uint32), want.view(np.uint32)))

    ms_curves = timed_ms(lambda: h.process_host_curves(x, curves, out=y, wait=wait), calls, warmup, h.synchronize)
    if devices is None:
        ms_plain = timed_ms(lambda: h.process_host_ptr(x.ctypes.data, y.ctypes.data, S), calls, warmup, h.synchronize)
    else:
        ms_plain = timed_ms(lambda: h.process_host(x, out=y), calls, warmup, h.synchronize)

    def per_8_periods():
        for k in range(0, S, EVERY):
            h.set_controls(reg, vals[k], broadcast=bcast)
            if devices is None:
                h.process_host_ptr(x.ctypes.data + 4 * k * n, y.ctypes.data + 4 * k * n, EVERY)
            else:
                h.process_host(x[:, k:k + EVERY, :], out=y[:, k:k + EVERY, :])
    ms_loop = timed_ms(per_8_periods, max(1, calls // 2), 1, h.synchronize)

    curve_rows = 0 if bcast else 1
    rec = {"case": label, "program": "cfg4" if reg_name == "filter_cutoff" else "cfg2", "instances": n, "periods": S,
           "curve": "broadcast" if bcast else "per-instance", "host_memory": "page-locked", "wait": wait,
           "path": "handle" if devices is None else f"executor over {len(devices)} GPU(s)", "devices": devices or [0],
           "calls_timed": calls, "warmup": warmup,
           "ms_per_block_curves": round(ms_curves, 3),
           "pcie_bytes_per_block": int(4 * (1 + 1 + curve_rows) * S * n) + (4 * S if bcast else 0),
           "ms_per_block_host_no_curves": round(ms_plain, 3),
           "pcie_bytes_per_block_no_curves": int(4 * 2 * S * n),
           "ms_per_block_host_call_per_8_periods": round(ms_loop, 3),
           "curves_over_no_curves": round(ms_curves / ms_plain, 3), "loop_over_curves": round(ms_loop / ms_curves, 2),
           "parity_instances": int(len(pick)), "parity_bit_exact": parity}
    h.close()
    prog.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("host_curves_bench.py needs a CUDA device (there is nothing to measure without one)")
    name, power = gpu_identity()
    every_gpu = list(range(torch.cuda.device_count()))
    cases = [
        ("cfg4_1gpu_blocking", progs.CFG4_ONEPOLE, 65536, "filter_cutoff", False, None, True),
        ("cfg4_1gpu_async", progs.CFG4_ONEPOLE, 65536, "filter_cutoff", False, None, False),
        ("cfg4_executor_blocking", progs.CFG4_ONEPOLE, 65536, "filter_cutoff", False, every_gpu, True),
        ("cfg4_executor_async", progs.CFG4_ONEPOLE, 65536, "filter_cutoff", False, every_gpu, False),
        ("cfg2_broadcast_1gpu_blocking", progs.CFG2_LOG_GAIN, 4096, "volume", True, None, True),
    ]
    failed = False
    for label, text, n, reg, bcast, devices, wait in cases:
        rec = run_case(label, text, n, reg, bcast, devices, wait, a.calls, a.warmup)
        rec["gpu"] = name
        rec["power_limit"] = power
        line = json.dumps(rec)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")
        failed = failed or not rec["parity_bit_exact"]
    if failed:
        raise SystemExit("parity check failed")


if __name__ == "__main__":
    main()
