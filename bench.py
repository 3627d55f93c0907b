#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200: instance-samples/s (and DSP instructions/s)
of the batched FX8010 interpreter, next to the reference's own CPU interpreter.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2|cfg3|cfg4|cfg5] [--dump-outputs DIR]

One "step" = one fx8010_gpu_process_batch call = one block of 1 024 samples for every instance of
this rank (BASELINE.json configs[1]: MACS gain + LOG waveshaper, 4 096 instances per GPU).  Instances
shard across ranks with no collective on the data path (weak scaling: every rank runs the same
per-GPU workload).  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import faulthandler
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
PKG = "fx8010-emulator-core_b200"

import progs  # noqa: E402  (program texts + stimuli shared with the tests)

BLOCK = 1024          # samples per step (48 kHz blocks of 1 024 samples)
L2_BYTES = 126 << 20
DUMP_BYTES = 64 * 10**6       # --dump-outputs writes at most this much


def workload(name: str):
    """(program text, instances per GPU, algorithmic bytes per instance-sample, label)."""
    if name == "cfg2":
        return progs.CFG2_LOG_GAIN, 4096, 8, "configs[1]: MACS gain + LOG waveshaper, 4096 instances x 1024-sample blocks per GPU"
    if name == "cfg1":
        return progs.CFG1A_TESTCODE, 4096, 8, "configs[0] batched: shipped testcode.da (MACS gain), 4096 instances x 1024-sample blocks per GPU"
    if name == "cfg3":
        return progs.cfg3_delay(1000), 16384, 16, "configs[2]: idelay feedback delay line (itramsize 1000), 16384 instances x 1024-sample blocks per GPU"
    if name == "cfg4":
        return progs.CFG4_ONEPOLE, 65536, 8, "configs[3]: INTERP one-pole low-pass bank, 65536 instances in total (sharded across the GPUs) x 1024-sample blocks"
    if name == "cfg5":
        return progs.cfg5_allops(), 32768, 8, "configs[4]: 512-instruction all-opcode program, 32768 instances x 1024-sample blocks per GPU"
    raise SystemExit(f"unknown config {name}")


def controls_for(name: str, prog, n: int, rng):
    if name in ("cfg1", "cfg2"):
        return {"volume": rng.random(n).astype(np.float32)}
    if name == "cfg4":
        return {"filter_cutoff": (0.001 + 0.998 * np.arange(n) / max(1, n - 1)).astype(np.float32)}
    if name == "cfg5":
        return {f"k{i}": rng.random(n).astype(np.float32) for i in range(4)}
    return {}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons while the timed region runs (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [t.strip() for t in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# IEEE operations one executed DSP instruction needs (SURVEY.md §8d table): (FP32/INT-pipe ops, FP64-pipe ops).
# Dispatch, operand fetch and CCR are excluded — this is the arithmetic the semantics require.
OP_COST = {"macs": (4, 0), "macsn": (4, 0), "macints": (4, 0), "acc3": (4, 0), "macw": (5, 0), "macwn": (5, 0), "macintw": (5, 0),
           "macmv": (2, 1), "andxor": (10, 0), "tstneg": (7, 0), "limit": (2, 0), "limitn": (2, 0), "log": (2, 5), "exp": (2, 5),
           "interp": (6, 3), "skip": (4, 0), "idelay": (0, 0), "xdelay": (0, 0), "end": (0, 0)}


def pipe_peaks():
    """Measured issue rates (lane-ops per clock per SM) from profiles/pipe_peaks.json (tests/pipe_peaks.cu, run on
    a B200 of this pool); nominal 128 / 64 when the file is missing."""
    p = os.path.join(ROOT, "profiles", "pipe_peaks.json")
    try:
        d = json.load(open(p))["pipes"]
        return (min(d["fadd_f32"]["lane_ops_per_clk_per_sm"], d["fmul_f32"]["lane_ops_per_clk_per_sm"]),
                min(d["dadd_f64"]["lane_ops_per_clk_per_sm"], d["dmul_f64"]["lane_ops_per_clk_per_sm"]),
                "measured (profiles/pipe_peaks.json: FADD/FMUL and DADD/DMUL lane-ops per clock per SM)")
    except Exception:
        return 128.0, 64.0, "nominal (128 FP32 / 64 FP64 lane-ops per clock per SM)"


def compute_roofline(text: str, executed_per_step: float, n_inst: int, step_s: float, sm_mhz: float, bytes_per: int, hbm_gbs: float):
    """SURVEY.md §8d for compute-bound programs: t_roofline = max(bytes / BW_HBM, sum FP32 ops / P32, sum FP64 ops / P64)
    with the sums from the program's opcode histogram scaled by the executed fraction (skipped instructions do no
    arithmetic), P32 / P64 = the measured FP32 / FP64 issue rates per clock and SM at the SM clock seen during the run."""
    ops = [ln.split()[0] for ln in text.lower().splitlines() if ln.split() and ln.split()[0] in OP_COST]
    f32 = sum(OP_COST[o][0] for o in ops)
    f64 = sum(OP_COST[o][1] for o in ops)
    frac = executed_per_step / (len(ops) * float(n_inst) * BLOCK)          # executed / issued
    clk = (sm_mhz or 1965.0) * 1e6
    p32, p64, src = pipe_peaks()
    t32 = f32 * frac * n_inst * BLOCK / (148 * p32 * clk)
    t64 = f64 * frac * n_inst * BLOCK / (148 * p64 * clk)
    thbm = bytes_per * n_inst * BLOCK / (hbm_gbs * 1e9)
    t_roof = max(t32, t64, thbm)
    return {"bound": "fp32-pipe" if t_roof == t32 else ("fp64-pipe" if t_roof == t64 else "hbm"),
            "t_roofline_us": 1e6 * t_roof, "t_measured_us": 1e6 * step_s, "frac": t_roof / step_s,
            "fp32_ops_per_sample": f32 * frac, "fp64_ops_per_sample": f64 * frac, "executed_fraction": frac,
            "peaks": f"{src}: {p32:.1f} FP32 / {p64:.1f} FP64 lane-ops per clock per SM x 148 SMs at the SM clock sampled during the run"}


def ncu_traffic(cfg: str):
    """dram bytes per launch of the interpreter kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(cfg)
        except Exception:
            return None
    return None


def cpu_reference_rate(text: str, cfg: str, target_seconds: float, threads: int):
    """The reference's own interpreter (oracle/_ref, unmodified sources) — or the oracle port when
    that binary is absent — one instance per thread on all host cores.  Returns a dict."""
    from oracle import pyoracle as po
    rng = np.random.default_rng(progs.SEED)
    probe = 100_000
    if po.have_reference():
        ctl = controls_for(cfg, None, threads, rng)

        def run(ns):
            x = progs.sine_bank(threads, min(ns, 48000), rng).T.copy()            # [T][S]
            if ns > x.shape[1]:
                x = np.tile(x, (1, (ns + x.shape[1] - 1) // x.shape[1]))[:, :ns].copy()
            secs, instr, _ = po.reference_bench(text, 1, threads, ns, x.reshape(threads, ns, 1), ctl)
            return secs, instr
        secs, _ = run(probe)
        ns = int(max(probe, min(2_000_000_000 // max(1, threads), probe * target_seconds / max(secs, 1e-6))))
        secs, instr = run(ns)
        return {"value": threads * ns / secs, "unit": "instance-samples/s", "cores": threads, "kind": "reference",
                "dsp_instr_per_s": instr / secs,
                "sample": f"{threads} threads x 1 instance x {ns} samples, one process() call per sample (reference main.cpp loop), {secs:.2f} s"}
    prog_mod = importlib.import_module(PKG)
    prog = prog_mod.Program(text)
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    n = threads * 8
    orc = po.Oracle(img, n, 1)
    x = progs.sine_bank(n, 4096, rng).reshape(1, 4096, n)
    t0 = time.perf_counter(); orc.process(x, threads=threads); secs = time.perf_counter() - t0
    reps = max(1, int(target_seconds / max(secs, 1e-6)))
    t0 = time.perf_counter()
    for _ in range(reps):
        orc.process(x, threads=threads)
    secs = time.perf_counter() - t0
    return {"value": n * 4096 * reps / secs, "unit": "instance-samples/s", "cores": threads, "kind": "port",
            "dsp_instr_per_s": None, "sample": f"oracle port, {n} instances x {4096 * reps} samples on {threads} threads, {secs:.2f} s"}


def sample_instances(n: int, k: int, rng) -> np.ndarray:
    """Instances the oracle re-computes: first, last and middle of this rank's range, the rest random (BASELINE.md §3)."""
    pick = {i for i in (0, 1, n - 1, n - 2, n // 2, n // 2 - 1) if 0 <= i < n}
    while len(pick) < min(k, n):
        pick.add(int(rng.integers(0, n)))
    return np.array(sorted(pick))


def oracle_blocks(text: str, prog, idx, controls: dict, x_blocks: list):
    """The reference (oracle/_ref) — or the C restatement when that binary is absent — over the sampled instances:
    x_blocks[b] is [S][N]; returns (outputs per block [S][k], final registers [n_regs][k], counters [k], kind)."""
    from oracle import pyoracle as po
    k = len(idx)
    if po.have_reference():
        outs = [np.zeros((x.shape[0], k), np.float32) for x in x_blocks]
        regs = np.zeros((len(prog.registers()), k), np.float32)
        counts = np.zeros(k, np.uint64)
        for j, i in enumerate(idx):
            r = po.Reference(text)
            assert r.loaded
            for name, v in controls.items():
                r.set_register(name, float(v[i]))
            for b, x in enumerate(x_blocks):
                outs[b][:, j] = r.process(np.ascontiguousarray(x[:, i])).ravel()
            regs[:, j] = r.register_values()
            counts[j] = r.instruction_counter & 0xffffffff
        return outs, regs, counts, "reference"
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, k, 1)
    for name, v in controls.items():
        orc.set_register(prog.reg_index(name), np.ascontiguousarray(v[idx]))
    outs = [orc.process(np.ascontiguousarray(x[:, idx]).reshape(1, x.shape[0], k))[0] for x in x_blocks]
    return outs, orc.registers.copy(), orc.counts.copy(), "restatement"


class Workload:
    """One BASELINE config on this rank: handle, controls, rotating device buffers; times blocks of 1 024 samples."""

    def __init__(self, fx, torch, cfg: str, n_inst: int, local_rank: int, rank: int, itram: int = 1000, translate: int | None = None, share=None):
        self.fx, self.torch, self.cfg, self.n = fx, torch, cfg, n_inst
        # FX8010_OPT_TRANSLATE for this workload's handles: 2 = the translated kernel, compiled before the first launch (what a long-running
        # host gets from the default background mode after the first second); 0 = the interpreter kernels (FX8010_BENCH_TRANSLATE overrides)
        self.translate = int(os.environ.get("FX8010_BENCH_TRANSLATE", "2")) if translate is None else translate
        self.text, _, self.bytes_per, self.label = workload(cfg)
        if cfg == "cfg3":
            self.text = progs.cfg3_delay(itram)
        self.rank, self.local_rank = rank, local_rank
        self.prog = fx.Program(self.text)
        assert self.prog.loaded, self.prog.errors()
        self.controls = controls_for(cfg, self.prog, n_inst, np.random.default_rng(progs.SEED + rank))
        self.block_bytes = 4 * n_inst * BLOCK
        # inputs: rotate over enough buffer pairs that a step never finds its data in L2
        self.n_bufs = max(2, -(-2 * L2_BYTES // (2 * self.block_bytes)) + 1)
        rng = np.random.default_rng(progs.SEED + 17 * rank)
        amp = (0.9, 0.9) if cfg == "cfg5" else (0.05, 0.99)
        if cfg == "cfg3":
            self.host_in = [progs.impulse_noise(n_inst, BLOCK, rng) for _ in range(2)]
        else:
            self.host_in = [progs.sine_bank(n_inst, BLOCK, rng, start=b * BLOCK, amp_lo=amp[0], amp_hi=amp[1]) for b in range(2)]
        if share is not None:
            self.d_in, self.d_out = share.d_in, share.d_out
        else:
            self.d_in = [torch.from_numpy(self.host_in[b % 2]).cuda() for b in range(self.n_bufs)]
            self.d_out = [torch.empty_like(self.d_in[0]) for _ in range(self.n_bufs)]
        self.stream = torch.cuda.Stream()
        self.st = self.stream.cuda_stream
        self.gpu = self.new_handle()

    def new_handle(self):
        g = self.fx.Gpu(self.n, 1, self.local_rank)
        g.load_program(self.prog)
        g.set_option(self.fx.OPT_TRANSLATE, self.translate)
        for name, v in self.controls.items():
            g.set_controls(self.prog.reg_index(name), v)
        return g

    def pointers(self, g, steps: int, first: int = 0):
        return g.block_pointers([self.d_in[(first + i) % self.n_bufs] for i in range(steps)],
                                [self.d_out[(first + i) % self.n_bufs] for i in range(steps)])

    def timed(self, steps: int, warmup: int, repeats: int, barrier):
        """`repeats` timed regions of exactly `steps` blocks each through ONE fx8010_gpu_process_blocks call
        (CUDA events on the launching stream); returns the per-region milliseconds and the launches of one region."""
        torch, g = self.torch, self.gpu
        warm = g.block_pointers([self.d_in[i % self.n_bufs] for i in range(max(warmup, self.n_bufs))],
                                [self.d_out[i % self.n_bufs] for i in range(max(warmup, self.n_bufs))])
        g.process_blocks_raw(warm, BLOCK, self.st)            # touches every buffer of the rotation
        ptrs = self.pointers(g, steps)
        g.process_blocks_raw(ptrs, BLOCK, self.st)            # the timed call itself, once, untimed (plan + encoding cached)
        barrier()
        ms, launches = [], 0
        for _ in range(repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            l0 = g.launch_info().kernel_launches
            with torch.cuda.stream(self.stream):
                e0.record(self.stream)
                g.process_blocks_raw(ptrs, BLOCK, self.st)
                e1.record(self.stream)
            barrier()
            ms.append(e0.elapsed_time(e1))
            launches = g.launch_info().kernel_launches - l0
        return ms, int(launches)

    def per_call(self, steps: int, barrier, exclusive: bool):
        """One fx8010_gpu_process_batch call per step from this Python loop (what round 1 timed)."""
        torch, g = self.torch, self.gpu
        g.set_option(self.fx.OPT_STREAM_EXCLUSIVE, 1 if exclusive else 0)
        for i in range(self.n_bufs):
            g.process_device(self.d_in[i], self.d_out[i], BLOCK, self.st)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(self.stream):
            e0.record(self.stream)
            for i in range(steps):
                g.process_device(self.d_in[i % self.n_bufs], self.d_out[i % self.n_bufs], BLOCK, self.st)
            e1.record(self.stream)
        barrier()
        g.set_option(self.fx.OPT_STREAM_EXCLUSIVE, 0)
        return e0.elapsed_time(e1) / steps

    def isolated(self, reps: int = 10):
        """One block alone on an idle GPU (launch + kernel + drain), microseconds."""
        torch, g = self.torch, self.gpu
        us = []
        for i in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            with torch.cuda.stream(self.stream):
                e0.record(self.stream)
                g.process_device(self.d_in[i % self.n_bufs], self.d_out[i % self.n_bufs], BLOCK, self.st)
                e1.record(self.stream)
            torch.cuda.synchronize()
            us.append(1e3 * e0.elapsed_time(e1))
        return statistics.median(us)

    def parity(self, steps: int, n_check: int = 64):
        """The timed call again on a FRESH handle (same geometry: same instance count, block length, buffer rotation and
        fused-launch plan), against the reference on a sample of instances: outputs of every block whose buffer
        survives the rotation, final registers and executed-instruction counters, bit for bit."""
        torch = self.torch
        g = self.new_handle()
        try:
            rng = np.random.default_rng(progs.SEED + 1000 + self.rank)
            idx = sample_instances(self.n, n_check, rng)
            g.process_blocks_raw(self.pointers(g, steps), BLOCK, self.st)
            g.synchronize(self.st)
            outs, regs, counts, kind = oracle_blocks(self.text, self.prog, idx, self.controls, [self.host_in[(i % self.n_bufs) % 2] for i in range(steps)])
            bad = 0
            d_idx = torch.from_numpy(idx.astype(np.int64)).cuda()
            survivors = range(max(0, steps - self.n_bufs), steps)
            for i in survivors:
                y = self.d_out[i % self.n_bufs].index_select(1, d_idx).cpu().numpy()
                bad += int(np.count_nonzero(y.view(np.uint32) != outs[i].view(np.uint32)))
            gr = g.registers()[:, idx]
            bad += int(np.count_nonzero(gr.view(np.uint32) != regs.view(np.uint32)))
            gc = g.counts()[idx]
            bad += int(np.count_nonzero((gc & np.uint64(0xffffffff)) != (counts & np.uint64(0xffffffff))))
            return {"checked_instances": int(len(idx)), "checked_blocks": len(list(survivors)), "blocks_run": steps, "mismatches": bad, "oracle": kind,
                    "what": "outputs of the surviving blocks, final register file, executed-instruction counters; first/last/middle of the rank's range + random"}
        finally:
            g.close()

    def dump_last_step(self, steps: int, path: str):
        """The output block of the last of `steps` timed steps, [samples][instances] float32, as path/out.npy (call it before
        anything else runs on the rotating buffers).  A block larger than DUMP_BYTES is cut to a fixed seeded sample of the
        instances, in ascending order, so that runs with the same arguments write the same array."""
        y = self.d_out[(steps - 1) % self.n_bufs]
        k = (DUMP_BYTES - 4096) // (4 * BLOCK)
        if self.n > k:
            idx = np.sort(np.random.default_rng(progs.SEED).choice(self.n, k, replace=False))
            y = y.index_select(1, self.torch.from_numpy(idx).to(y.device))
        os.makedirs(path, exist_ok=True)
        np.save(os.path.join(path, "out.npy"), y.cpu().numpy())

    def executed_per_step(self):
        g = self.new_handle()
        g.process_device(self.d_in[0], self.d_out[0], BLOCK, self.st); g.synchronize(self.st)
        c = g.count_total()
        g.close()
        return c

    def close(self):
        self.gpu.close()


def main():
    faulthandler.enable()               # a native fault in any rank leaves a Python traceback on stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="blocks per timed region of the headline measurement (and of its per-call and "
                    "interpreter legs); the e2e leg runs max(10, min(K, 200)) steps and the sharded cfg3 / cfg4 / cfg5 records 10 / 20 / 3")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--instances", type=int, default=0, help="override instances per GPU")
    ap.add_argument("--itram", type=int, default=1000, help="cfg3: ring size")
    ap.add_argument("--repeats", type=int, default=5, help="timed regions of K steps each; the median is reported")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-interpreter-leg", action="store_true", help="skip timing the same steps on the interpreter kernels")
    ap.add_argument("--no-sharded", action="store_true", help="skip the cfg4 / cfg5 records of the scaling line")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the output block of the last one as DIR/out.npy "
                    "(float32 [samples][instances] of rank 0; a fixed sample of the instances when larger than 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed (--impl ours)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    text, n_inst, bytes_per, label = workload(args.config)
    if args.config == "cfg3":
        text = progs.cfg3_delay(args.itram)
        label = label.replace("itramsize 1000", f"itramsize {args.itram}")
    if args.config == "cfg4":
        n_inst = max(1, n_inst // world)                  # 65 536 in total, sharded
    if args.instances:
        n_inst = args.instances
    instr_per_sample = sum(progs.opcode_histogram(text).values())

    # ---------------------------------------------------------------- reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        threads = os.cpu_count() or 1
        per_step = max(0.2, min(1.0, 60.0 / max(1, args.steps + args.warmup)))
        base = cpu_reference_rate(text, args.config, per_step, threads)     # calibrates the step size
        from oracle import pyoracle as po
        # timed: K steps of the same bounded sample
        rng = np.random.default_rng(progs.SEED)
        ns = max(1024, int(base["value"] / threads * per_step))
        if po.have_reference():
            ctl = controls_for(args.config, None, threads, rng)
            x = progs.sine_bank(threads, min(ns, 48000), rng).T.copy()
            if ns > x.shape[1]:
                x = np.tile(x, (1, (ns + x.shape[1] - 1) // x.shape[1]))[:, :ns].copy()
            x = x.reshape(threads, ns, 1)
            total_s, total_instr = 0.0, 0
            for i in range(args.warmup + args.steps):
                secs, instr, _ = po.reference_bench(text, 1, threads, ns, x, ctl)
                if i >= args.warmup:
                    total_s += secs; total_instr += instr
            value = threads * ns * args.steps / total_s
            kind, ips = "reference", total_instr / total_s
        else:
            value, kind, ips, total_s = base["value"], "port", None, per_step * args.steps
        line = {"impl": "reference", "metric": "instance_samples_per_s", "value": value, "unit": "instance-samples/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_s / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
                "dsp_instr_per_s": ips,
                "config": {"workload": label, "instances_per_gpu": n_inst, "block_samples": BLOCK, "program_instructions_per_sample": instr_per_sample},
                "cpu_baseline": {"value": value, "unit": "instance-samples/s", "cores": threads, "kind": kind,
                                 "sample": f"per step: {threads} threads x 1 instance x {ns} samples, one process() per sample"},
                "e2e": {"value": value, "unit": "instance-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------- our arm (GPU)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    fx = importlib.import_module(PKG)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v: float) -> float:
        if world > 1:
            t = torch.tensor([v], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); return float(t.item())
        return v

    def sum_over_ranks(v: float) -> float:
        if world > 1:
            t = torch.tensor([v], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.SUM); return float(t.item())
        return v

    peak, peak_src = measured_peak()
    W = Workload(fx, torch, args.config, n_inst, local_rank, rank, args.itram)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    ms_all, launches = W.timed(args.steps, args.warmup, max(1, args.repeats), barrier)
    ms_all = [max_over_ranks(m) for m in ms_all]
    ms = statistics.median(ms_all)
    if args.dump_outputs and rank == 0:
        W.dump_last_step(args.steps, args.dump_outputs)
    # keep the clock sampler running over a longer window of the same work so it sees load
    if rank == 0:
        ptrs = W.pointers(W.gpu, min(32, max(args.steps, 8)))
        t_end = time.time() + 0.4
        while time.time() < t_end:
            for _ in range(4):
                W.gpu.process_blocks_raw(ptrs, BLOCK, W.st)
            W.gpu.synchronize(W.st)
    clocks = sampler.stop() if rank == 0 else None
    info = W.gpu.launch_info()
    translated = W.gpu.translate_status()
    # the same steps on the interpreter kernels (FX8010_OPT_TRANSLATE = 0): the number before translation, for comparison
    interp = None
    if W.translate and (info.kernel_variant & 128) and not args.no_interpreter_leg:
        Wi = Workload(fx, torch, args.config, n_inst, local_rank, rank, args.itram, translate=0, share=W)
        mi_all, li = Wi.timed(args.steps, args.warmup, 3, barrier)
        mi = statistics.median([max_over_ranks(v) for v in mi_all])
        ii = Wi.gpu.launch_info()
        interp = {"what": "the same timed call with FX8010_OPT_TRANSLATE = 0 (interpreter kernels only)", "ms_per_step": mi / args.steps,
                  "hbm_frac": bytes_per * n_inst * BLOCK * args.steps / (mi * 1e-3) / 1e9 / peak, "gpu_launches": li,
                  "kernel_variant": hex(ii.kernel_variant)}
        Wi.close()
    kernel_cfg = {"grid": info.last_grid, "block": info.last_block, "time_split": info.last_time_split, "blocks_per_launch": info.last_fused_blocks,
                  "smem_bytes": info.last_smem_bytes, "instances_per_thread": (info.kernel_variant >> 8) & 0xff, "samples_per_batch": info.kernel_variant >> 16,
                  "translated_kernel": bool(info.kernel_variant & 128)}
    value = float(n_inst) * BLOCK * args.steps * world / (ms * 1e-3)
    # the same steps as one C-ABI call per step from this Python loop, and one block alone on an idle GPU
    per_call_ms = max_over_ranks(W.per_call(args.steps, barrier, exclusive=False))
    per_call_excl_ms = max_over_ranks(W.per_call(args.steps, barrier, exclusive=True))
    isolated_us = W.isolated() if rank == 0 else None
    barrier()
    instr_per_step = sum_over_ranks(float(W.executed_per_step()))

    # ---- parity of the timed call (fresh state, same geometry) against the reference on a sample of instances
    parity = None
    if not args.no_parity:
        parity = W.parity(args.steps)
        parity["mismatches"] = int(sum_over_ranks(float(parity["mismatches"])))
        parity["checked_instances"] = int(sum_over_ranks(float(parity["checked_instances"])))

    # ---- end to end through the C ABI with HOST buffers (pinned), copies inside the timed region
    e2e = None
    if not args.no_e2e:
        gpu = W.gpu
        n_host = 4                                       # page-locked in/out pairs the steps rotate over
        pin = [fx.pinned_array((1, BLOCK, n_inst)) for _ in range(n_host)]
        pout = [fx.pinned_array((1, BLOCK, n_inst)) for _ in range(n_host)]
        for b in range(n_host):
            pin[b][0][...] = W.host_in[b % 2].reshape(1, BLOCK, n_inst)
        e2e_steps = max(10, min(args.steps, 200))

        def e2e_run(wait):
            for i in range(3):
                gpu.process_host_ptr(pin[i % n_host][0].ctypes.data, pout[i % n_host][0].ctypes.data, BLOCK)
            barrier()
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                gpu.process_host_ptr(pin[i % n_host][0].ctypes.data, pout[i % n_host][0].ctypes.data, BLOCK, wait=wait)
            gpu.synchronize(None)                        # every step's output has reached host memory
            barrier()
            return max_over_ranks(time.perf_counter() - t0)
        dt_sync = e2e_run(True)                          # one blocking call per step
        dt = statistics.median([e2e_run(False) for _ in range(3)])    # queued calls: copies of consecutive steps overlap
        e2e = {"value": float(n_inst) * BLOCK * e2e_steps * world / dt, "unit": "instance-samples/s",
               "h2d_bytes_per_step": W.block_bytes, "d2h_bytes_per_step": W.block_bytes, "steps": e2e_steps,
               "ms_per_step": 1e3 * dt / e2e_steps, "host_buffers": "pinned (fx8010_gpu_host_alloc)",
               "api": "fx8010_gpu_process_batch_host_async per step + one fx8010_gpu_synchronize (median of 3 runs)",
               "pcie_gbs_each_way_per_gpu": W.block_bytes * e2e_steps / dt / 1e9,
               "blocking_call_value": float(n_inst) * BLOCK * e2e_steps * world / dt_sync,
               "blocking_call_ms_per_step": 1e3 * dt_sync / e2e_steps}
        del pin, pout
    W.close()

    # ---- the other BASELINE.json configs at their per-GPU share (SURVEY.md §8e): cfg3 = 16 384 instances per GPU (ring of 1 000), cfg4 =
    # 65 536 instances in total, cfg5 = 32 768 per GPU; same timing rules, fewer steps
    sharded = None
    if not args.no_sharded and args.config == "cfg2":
        sharded = {}
        for cfg, n_cfg, k_steps in (("cfg3", 16384, 10), ("cfg4", max(1, 65536 // world), 20), ("cfg5", 32768, 3)):
            t_cfg, _, b_cfg, l_cfg = workload(cfg)
            Wc = Workload(fx, torch, cfg, n_cfg, local_rank, rank)
            m_all, l_n = Wc.timed(k_steps, 3, 3, barrier)
            m = statistics.median([max_over_ranks(v) for v in m_all])
            par = Wc.parity(2 if cfg == "cfg5" else k_steps, 32)
            par["mismatches"] = int(sum_over_ranks(float(par["mismatches"])))
            par["checked_instances"] = int(sum_over_ranks(float(par["checked_instances"])))
            ex = sum_over_ranks(float(Wc.executed_per_step()))
            step_s = 1e-3 * m / k_steps
            rec = {"workload": l_cfg, "instances_per_gpu": n_cfg, "instances_total": n_cfg * world, "steps": k_steps, "ms_per_step": 1e3 * step_s,
                   "value": float(n_cfg) * BLOCK * world / step_s, "unit": "instance-samples/s", "dsp_instr_per_s": ex / step_s,
                   "hbm_frac": b_cfg * n_cfg * BLOCK / step_s / 1e9 / peak, "gpu_launches": l_n, "parity": par}
            rec["translated_kernel"] = bool(Wc.gpu.launch_info().kernel_variant & 128)
            if cfg == "cfg5":
                rec["translated"] = Wc.gpu.translate_status()      # FX8010_OPT_TRANSLATE: state 2 = the NVRTC-compiled kernel ran
                rec["compute_roofline"] = compute_roofline(t_cfg, ex / world, n_cfg, step_s, (clocks or {}).get("sm_mhz") if clocks else None, b_cfg, peak)
            sharded[cfg] = rec
            Wc.close()

    def leave(code: int = 0):
        """Multi-rank runs end without tearing NCCL / CUDA down object by object (one run in six died with SIGSEGV in
        rank 0 somewhere after the last measurement on a 2-GPU box; the handles of this library are closed above)."""
        sys.stdout.flush(); sys.stderr.flush()
        if world > 1:
            os._exit(code)

    if world > 1:
        dist.barrier()
    if rank != 0:
        leave()
        return
    alg_bytes = bytes_per * n_inst * BLOCK * args.steps / max(1, launches)      # one launch covers steps / launches blocks
    launch_ms = ms / max(1, launches)
    achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    line = {"metric": "instance_samples_per_s", "value": value, "unit": "instance-samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.config == "cfg4" else "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
            "dsp_instr_per_s": instr_per_step * args.steps / (ms * 1e-3),
            "config": {"workload": label, "instances_per_gpu": n_inst, "block_samples": BLOCK,
                       "program_instructions_per_sample": instr_per_sample,
                       "l2": f"rotating {W.n_bufs} input/output buffer pairs ({2 * W.n_bufs * W.block_bytes >> 20} MiB > 126 MiB L2), every one touched during warm-up",
                       "timed_call": f"one fx8010_gpu_process_blocks call of {args.steps} blocks per timed region ({launches} kernel launches), median of {len(ms_all)} regions",
                       "kernel": kernel_cfg},
            "timed_regions_ms": ms_all,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (ncu_traffic(args.config) or 0) * args.steps / max(1, launches) or None, "peak_source": peak_src,
                         "traffic_source": "profiles/traffic.json: dram__bytes_read + dram__bytes_write per block from the committed ncu --set full capture, x blocks per launch",
                         "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_us": 1e3 * launch_ms,
                         "blocks_per_launch": args.steps / max(1, launches)},
            "per_call": {"what": "the same steps as one fx8010_gpu_process_batch call per step from the Python loop",
                         "ms_per_step": per_call_ms, "hbm_frac": bytes_per * n_inst * BLOCK / (per_call_ms * 1e-3) / 1e9 / peak,
                         "ms_per_step_stream_exclusive": per_call_excl_ms,
                         "hbm_frac_stream_exclusive": bytes_per * n_inst * BLOCK / (per_call_excl_ms * 1e-3) / 1e9 / peak,
                         "isolated_launch_us": isolated_us},
            "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e, "parity": parity,
            "translator": {"status": translated, "interpreter_kernels": interp,
                           "what": "FX8010_OPT_TRANSLATE: the loaded DSP program compiled (NVRTC, sm_100a) into one straight-line kernel built from the same "
                                   "hand-written arithmetic helpers as the interpreter kernels; bit-identical results (parity object above)"}}
    if sharded:
        line["sharded"] = sharded
    if args.config == "cfg5":        # compute-bound program: the arithmetic roofline of SURVEY.md §8d beside the HBM one
        line["compute_roofline"] = compute_roofline(text, instr_per_step / world, n_inst, 1e-3 * ms / args.steps,
                                                    (clocks or {}).get("sm_mhz"), bytes_per, peak)
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_reference_rate(text, args.config, 10.0, os.cpu_count() or 1)
    print(json.dumps(line))
    bad = (parity or {}).get("mismatches", 0) + sum(r["parity"]["mismatches"] for r in (sharded or {}).values())
    if bad:
        print(f"bench.py: GPU results differ from the reference ({bad} mismatching values)", file=sys.stderr)
        leave(1)
        raise SystemExit(1)
    leave()


if __name__ == "__main__":
    main()
