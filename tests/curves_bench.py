"""Measures sample-accurate control curves (fx8010_gpu_process_batch_curves) against the ways a caller had before them.

    python tests/curves_bench.py [--calls 200] [--warmup 20] [--out FILE]

cfg4 (one-pole low-pass, 65 536 instances x 1 024 periods, a per-instance filter_cutoff curve):
    (a) curves   (b) process_batch_events every 8 periods (the reference driver's slider rate)   (c) events every period (fewer calls)
cfg2 (LOG waveshaper + gain, 4 096 instances x 1 024 periods):
    (d) plain, no curves   (e) a broadcast volume ramp   (f) a per-instance volume curve

One JSON line per case: microseconds per block (CUDA events around back-to-back calls on one stream, after a warm-up), kernel
launches per block and the last kernel_variant (launch_info), the share of the HBM roofline at 4 x (inputs + outputs + per-instance
curves) bytes per instance and period against bench.py's measured_peak() (with its label), a bit-exact parity check of >= 64 sampled
instances against the oracle stepped one period at a time, and the GPU's name and power limit read in the same run.  The translator runs
in mode 2 (kernels compiled before the first call).  Needs a GPU: without one it fails.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [HERE, ROOT]
import curves_common as cc  # noqa: E402
import progs  # noqa: E402
from bench import measured_peak  # noqa: E402

fx = importlib.import_module("fx8010-emulator-core_b200")


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip().split(",")[-1].strip() if q.returncode == 0 else "unknown"
    except Exception:
        power = "unknown"
    return name, power


def oracle_for(text, n):
    from oracle import pyoracle as po
    p = fx.Program(text)
    img = po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables())
    return po.Oracle(img, n, 1)


def held(vals, every):
    """The values a caller that changes the control every `every` periods sends (period k holds the value of period k - k % every)."""
    idx = np.arange(vals.shape[0]) // every * every
    return np.ascontiguousarray(vals[idx])


def run_case(label, text, n, s, reg_name, mode, every, bcast, calls, warmup, peak, torch):
    """mode: 'plain', 'curves' or 'events' (one event per curve every `every` periods)."""
    rng = np.random.default_rng(0x8010)
    prog = fx.Program(text)
    reg = prog.reg_index(reg_name)
    gpu = fx.Gpu(n, 1, 0)
    gpu.load_program(prog)
    gpu.set_option(fx.OPT_TRANSLATE, 2)
    x = progs.sine_bank(n, s, rng).reshape(1, s, n)
    if reg_name == "volume":
        vals = (np.linspace(0.05, 1.0, s, dtype=np.float32) if bcast else
                np.ascontiguousarray(np.linspace(0.05, 1.0, s, dtype=np.float32)[:, None] * np.linspace(0.2, 1.0, n, dtype=np.float32)[None, :]))
    else:
        vals = cc.make_curve("cfg4", reg_name, bcast, s, n, rng)
    d_x = torch.from_numpy(x).cuda()
    d_y = torch.empty_like(d_x)
    d_v = torch.from_numpy(vals).cuda()
    st = torch.cuda.Stream()
    if mode == "events":
        hv = held(vals, every)
        events = [(k, reg, hv[k]) for k in range(0, s, every)]

    def call():
        if mode == "plain":
            gpu.process_device(d_x, d_y, s, st.cuda_stream)
        elif mode == "curves":
            gpu.process_device_curves(d_x, d_y, s, [(reg, d_v, bcast)], st.cuda_stream)
        else:
            gpu.process_device_events(d_x, d_y, s, events, st.cuda_stream)

    # parity: the first call from the freshly loaded state, >= 64 sampled instances against the oracle stepped per period
    call()
    torch.cuda.synchronize()
    y = d_y.cpu().numpy()
    pick = np.unique(np.concatenate([[0, n - 1], rng.choice(n, 70, replace=False)]))
    orc = oracle_for(text, len(pick))
    if mode == "plain":
        want = orc.process(np.ascontiguousarray(x[:, :, pick]))
    else:
        v = held(vals, every) if mode == "events" else vals
        v = v if bcast else np.ascontiguousarray(v[:, pick])
        want = cc.oracle_stepped(orc, np.ascontiguousarray(x[:, :, pick]), [(reg, v, bcast)], s)
    parity = bool(np.array_equal(y[:, :, pick].view(np.uint32), want.view(np.uint32)))
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    l0 = gpu.launch_info().kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(calls):
        call()
    e1.record(st)
    torch.cuda.synchronize()
    info = gpu.launch_info()
    us = e0.elapsed_time(e1) * 1e3 / calls
    curve_rows = 1 if (mode != "plain" and not bcast) else 0
    bytes_per_block = 4.0 * (1 + 1 + curve_rows) * n * s
    rec = {"case": label, "program": "cfg4" if reg_name == "filter_cutoff" else "cfg2", "instances": n, "periods": s, "call": mode,
           "curve": None if mode == "plain" else ("broadcast" if bcast else "per-instance"), "event_every": every if mode == "events" else None,
           "calls_timed": calls, "warmup": warmup, "us_per_block": round(us, 2),
           "launches_per_block": (info.kernel_launches - l0) / calls, "kernel_variant": int(info.kernel_variant),
           "curves_in_kernel": bool(info.kernel_variant & fx.VARIANT_CURVES),
           "bytes_per_block": int(bytes_per_block), "hbm_roofline_fraction": round(bytes_per_block / (us * 1e-6) / (peak[0] * 1e9), 3),
           "hbm_peak_gbs": peak[0], "hbm_peak_source": peak[1], "parity_instances": int(len(pick)), "parity_bit_exact": parity}
    gpu.close()
    prog.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("curves_bench.py needs a CUDA device (there is nothing to measure without one)")
    name, power = gpu_identity()
    peak = measured_peak()
    S = 1024
    cases = [
        ("a", progs.CFG4_ONEPOLE, 65536, "filter_cutoff", "curves", 1, False, a.calls),
        ("b", progs.CFG4_ONEPOLE, 65536, "filter_cutoff", "events", 8, False, a.calls),
        ("c", progs.CFG4_ONEPOLE, 65536, "filter_cutoff", "events", 1, False, max(1, a.calls // 10)),
        ("d", progs.CFG2_LOG_GAIN, 4096, "volume", "plain", 1, False, a.calls),
        ("e", progs.CFG2_LOG_GAIN, 4096, "volume", "curves", 1, True, a.calls),
        ("f", progs.CFG2_LOG_GAIN, 4096, "volume", "curves", 1, False, a.calls),
    ]
    failed = False
    for label, text, n, reg, mode, every, bcast, calls in cases:
        rec = run_case(label, text, n, S, reg, mode, every, bcast, calls, min(a.warmup, calls), peak, torch)
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
