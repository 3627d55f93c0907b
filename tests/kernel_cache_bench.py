"""Measures what the translator's disk kernel cache saves a process that starts cold (empty directory) against one that starts warm (the
directory a previous process filled).

    python tests/kernel_cache_bench.py [--blocks 200] [--out FILE]

Cases, each in a fresh process (the cache counters and the process CUBIN store belong to the process), translation mode 1 (the default:
the compiler never blocks a call; until the kernel is ready a plain call runs on the interpreter kernels, a curve call one launch per
period):
    cfg2        4 096 instances x 1 024 periods, plain calls
    cfg4_curve  65 536 instances x 1 024 periods, a per-instance filter_cutoff curve (fx8010_gpu_process_batch_curves)
    cfg5        32 768 instances x 1 024 periods, plain calls
    multi3      the 3-shard executor on device 0, cfg2 at 3 x 4 096 instances x 1 024 periods, host buffers
For each, cold then warm: the time from load_program to the end of the first block that ran on the translated kernel, the wall time of
the first `--blocks` blocks (each block ends in a device synchronise, as a host that consumes every block does; blocks keep running past
them until the translated kernel is there), the number of those blocks that ran translated, the NVRTC compiles and disk hits of the process, and the NVRTC version it loaded (these processes import torch
first, and torch brings a libnvrtc of its own).  Two more lines time one NVRTC compile of cfg2 and of cfg5 (fx8010_translate_source
with compile_check), in a process that imported torch and in one that did not.  One JSON line per case and start, with the GPU's name
and power limit read in the same run.  Needs a GPU: without one it fails.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [HERE, ROOT]
import progs  # noqa: E402

CASES = {
    "cfg2": (progs.CFG2_LOG_GAIN, 4096, []),
    "cfg4_curve": (progs.CFG4_ONEPOLE, 65536, ["filter_cutoff"]),
    "cfg5": (progs.cfg5_allops(), 32768, []),
    "multi3": (progs.CFG2_LOG_GAIN, 3 * 4096, []),
}
S = 1024


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() if q.returncode == 0 else "unknown"
    except Exception:
        power = "unknown"
    return name, power


def nvrtc_loaded():
    """Version of the libnvrtc.so.12 this process has loaded (dlopen returns the one already mapped)."""
    import ctypes as C
    lib = C.CDLL("libnvrtc.so.12")
    major, minor = C.c_int(), C.c_int()
    lib.nvrtcVersion(C.byref(major), C.byref(minor))
    return f"{major.value}.{minor.value}"


def compile_times(with_torch):
    if with_torch:
        import torch  # noqa: F401
    fx = importlib.import_module("fx8010-emulator-core_b200")
    rec = {}
    for name, text in (("cfg2", progs.CFG2_LOG_GAIN), ("cfg5", progs.cfg5_allops())):
        prog = fx.Program(text)
        t0 = time.perf_counter()
        _, cubin = fx.translate_source(prog, 1, compile_check=True, instances=CASES[name][1])
        rec[name + "_compile_ms"] = round((time.perf_counter() - t0) * 1e3, 1) if cubin and cubin > 0 else None
    rec["nvrtc"] = nvrtc_loaded()
    return rec


def run_one(case, blocks):
    """One process, one case: what the parent prints as a JSON line."""
    if case.startswith("compile"):
        return compile_times(case == "compile_torch")
    import numpy as np
    import torch
    fx = importlib.import_module("fx8010-emulator-core_b200")
    text, n, curves = CASES[case]
    prog = fx.Program(text)
    assert prog.loaded, prog.errors()
    rng = np.random.default_rng(progs.SEED)
    if case == "multi3":
        x = (1.8 * rng.random((1, S, n)) - 0.9).astype(np.float32)
        out = np.empty_like(x)
        torch.cuda.init()
        t0 = time.perf_counter()
        h = fx.MultiGpu([0, 0, 0], n, 1)
        h.load_program(prog)
        h.set_option(fx.OPT_TRANSLATE, 1)
        import kernel_cache_common as kc
        first, done, b, total = None, 0, 0, None
        while b < blocks or (first is None and time.perf_counter() - t0 < 30):
            h.process_host(x, out=out)
            b += 1
            if kc.all_translated(fx, h):
                done += b <= blocks
                if first is None:
                    first = time.perf_counter() - t0
            if b == blocks:
                total = time.perf_counter() - t0
        h.close()
    else:
        d_x = torch.rand((1, S, n), device="cuda") * 1.8 - 0.9
        d_y = torch.empty_like(d_x)
        cv = [(prog.reg_index(r), torch.rand((S, n), device="cuda") * 0.998 + 0.001, False) for r in curves]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gpu = fx.Gpu(n, 1, 0)
        gpu.load_program(prog)
        gpu.set_option(fx.OPT_TRANSLATE, 1)
        bit = fx.VARIANT_CURVES if curves else 128
        first, done, b, total = None, 0, 0, None
        while b < blocks or (first is None and time.perf_counter() - t0 < 30):      # (past `blocks` until the kernel is there)
            if cv:
                gpu.process_device_curves(d_x, d_y, S, cv)
            else:
                gpu.process_device(d_x, d_y, S)
            gpu.synchronize()
            b += 1
            if gpu.launch_info().kernel_variant & bit:
                done += b <= blocks
                if first is None:
                    first = time.perf_counter() - t0
            if b == blocks:
                total = time.perf_counter() - t0
        gpu.close()
    st = fx.kernel_cache_stats()
    return {"first_translated_ms": None if first is None else round(first * 1e3, 2), "blocks": blocks, "wall_ms": round(total * 1e3, 2),
            "translated_blocks": done, "nvrtc_compiles": st["nvrtc_compiles"], "disk_hits": st["disk_hits"], "disk_writes": st["disk_writes"],
            "joined_compiles": st["joined_compiles"], "store_hits": st["store_hits"], "memory_hits": st["memory_hits"], "nvrtc": nvrtc_loaded()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--blocks", type=int, default=200)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.one:
        print(json.dumps(run_one(args.one, args.blocks)))
        return
    name, power = gpu_identity()
    lines = []
    for case in ("compile_torch", "compile_no_torch"):
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", case], capture_output=True, text=True, timeout=600)
        if r.returncode:
            raise SystemExit(f"{case}: {r.stderr[-3000:]}")
        rec = {"case": case, **json.loads(r.stdout.strip().splitlines()[-1]), "gpu": name, "power_limit": power}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    for case in CASES:
        with tempfile.TemporaryDirectory(prefix="fx8010-kcache-") as d:
            for start in ("cold", "warm"):
                env = dict(os.environ, FX8010_KERNEL_CACHE=d)
                env.pop("FX8010_TRANSLATE", None)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", case, "--blocks", str(args.blocks)], env=env,
                                   capture_output=True, text=True, timeout=1800)
                if r.returncode:
                    raise SystemExit(f"{case} {start}: {r.stderr[-3000:]}")
                rec = {"case": case, "start": start, "instances": CASES[case][1], "samples": S, **json.loads(r.stdout.strip().splitlines()[-1]),
                       "gpu": name, "power_limit": power}
                print(json.dumps(rec), flush=True)
                lines.append(rec)
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
