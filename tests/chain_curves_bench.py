"""Measures program chains with control curves (fx8010_chain_process_batch_curves) against the same stages called one after another
(fx8010_gpu_process_batch_curves on the automated stage, fx8010_gpu_process_batch on the others).

    python tests/chain_curves_bench.py [--calls 200] [--warmup 20] [--reps 5] [--out FILE]

Cases (1 024 periods per block, device buffers, translator in mode 2 on every stage):
    (a) cfg2 (LOG waveshaper + gain) -> the shipped testcode.da volume with a per-instance curve -> a limiter, 65 536 instances: every block
        buffer is 268 MB, beyond L2;
    (b) the same chain with a broadcast ramp on volume: the cost of a broadcast curve;
    (c) case (a) at 4 096 instances: the intermediate blocks fit in L2;
    (d) cfg2 -> cfg4 (one-pole low-pass) with a per-instance cutoff curve, 65 536 instances: a stage with state, so the chain runs stage by
        stage, the cfg4 stage on its translated serial curve kernel.

One JSON line per case: microseconds per block of the chain call and of the stage-by-stage form (CUDA events around `calls` back-to-back
calls after `warmup` calls, the median of `reps` repetitions, the two forms alternating on the same handles), the HBM share of each against
7.7 TB/s at 4 B per instance-sample for every input, output and per-instance curve pass (fused: 12 B with a per-instance curve, 8 B with a
broadcast one; stage by stage: 8 B per stage plus 4 B per per-instance curve), and a bit-exact check of >= 64 sampled instances of the first
and of the last timed chain call against the stages' oracles stepped per period.  The GPU's name and power limit are read in the same run.
Needs a GPU: without one it fails.
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [HERE, os.path.dirname(HERE)]
import chain_common as cc  # noqa: E402
import chain_curves_common as ccc  # noqa: E402
import progs  # noqa: E402
from curves_bench import gpu_identity  # noqa: E402

fx = importlib.import_module("fx8010-emulator-core_b200")
S = 1024
HBM_BYTES_PER_S = 7.7e12


def oracle_check(texts, ctl, x, y, curves, vals, idx):
    """True when y[:, :, idx] equals the stages' oracles stepped per period with the curves, from a freshly loaded state, on x[:, :, idx]."""
    from oracle import pyoracle as po
    orcs = []
    for text, c in zip(texts, ctl):
        p = fx.Program(text)
        orc = po.Oracle(po.Image(p.instructions(), p.registers(), p.itram_size, p.xtram_size, p.controls(), p.tables()), len(idx), 1)
        for nm, v in c.items():
            orc.set_register(nm, v[idx])
        orcs.append(orc)
    sub = [v if bc else np.ascontiguousarray(v[:, idx]) for (_, _, bc), v in zip(curves, vals)]
    want = ccc.oracle_chain_curves_stepped(orcs, np.ascontiguousarray(x[:, :, idx]), x.shape[1], curves, sub, len(idx))
    return bool(np.array_equal(np.ascontiguousarray(y[:, :, idx]).view(np.uint32), want.view(np.uint32)))


def run_case(torch, label, texts, n, curve_names, calls, warmup, reps):
    """curve_names: [(stage, register name, broadcast)]."""
    rng = np.random.default_rng(0x8010)
    stages, ctl, prog_list = [], [], []
    for j, text in enumerate(texts):
        p = fx.Program(text)
        g = fx.Gpu(n, 1)
        g.load_program(p)
        g.set_option(fx.OPT_TRANSLATE, 2)
        c = {nm: (0.05 + 0.95 * rng.random(n)).astype(np.float32) for nm in p.controls()}
        for nm, v in c.items():
            g.set_controls(p.reg_index(nm), v)
        stages.append(g); ctl.append(c); prog_list.append(p)
    chain = fx.Chain(stages)
    curves = [(j, prog_list[j].reg_index(nm), bc) for j, nm, bc in curve_names]
    vals = ccc.curve_values(curves, S, n, rng)
    d_vals = [torch.from_numpy(v).cuda() for v in vals]
    chain_list = [(j, r, d, bc) for (j, r, bc), d in zip(curves, d_vals)]
    x = (1.8 * rng.random((1, S, n)) - 0.9).astype(np.float32)
    d_x = torch.from_numpy(x).cuda()
    d_y, d_s = torch.empty_like(d_x), torch.empty_like(d_x)
    mid = [torch.empty_like(d_x) for _ in range(2)]
    idx = np.sort(rng.choice(n, 64, replace=False))

    def fused():
        chain.process_batch_curves(d_x, d_y, S, chain_list)

    def sequential():
        cur = d_x
        for j, g in enumerate(stages):
            out = d_s if j + 1 == len(stages) else mid[j & 1]
            mine = [(r, d, bc) for (st, r, d, bc) in chain_list if st == j]
            if mine:
                g.process_device_curves(cur, out, S, mine)
            else:
                g.process_device(cur, out, S)
            cur = out

    fused()
    torch.cuda.synchronize()
    st = chain.status()
    stateless = st["fused_last"] == 1
    first_ok = oracle_check(texts, ctl, x, d_y.cpu().numpy(), curves, vals, idx) if stateless else None
    cst = chain.status_curves()
    for _ in range(warmup):
        fused(); sequential()
    torch.cuda.synchronize()
    times = {"chain": [], "sequential": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(reps):
        for name, fn in (("chain", fused), ("sequential", sequential)):
            ev[0].record()
            for _ in range(calls):
                fn()
            ev[1].record()
            torch.cuda.synchronize()
            times[name].append(ev[0].elapsed_time(ev[1]) * 1e3 / calls)
    y_last, s_last = d_y.cpu().numpy(), d_s.cpu().numpy()
    # (stateless stages: the outputs of a call depend on its inputs and curves only, not on the state earlier calls left)
    last_ok = oracle_check(texts, ctl, x, y_last, curves, vals, idx) if stateless else None
    st = chain.status()
    us = {k: float(np.median(v)) for k, v in times.items()}
    k = len(texts)
    n_cvi = sum(0 if bc else 1 for _, _, bc in curves)
    bytes_fused = 4.0 * (2 + n_cvi) if st["fused_last"] else 8.0 * k + 4.0 * n_cvi
    bytes_seq = 8.0 * k + 4.0 * n_cvi
    row = {"case": label, "instances": n, "periods": S, "stages": k, "curves": [[j, nm, bool(bc)] for j, nm, bc in curve_names],
           "fused": st["fused_last"], "why_not_fused": st["message"],
           "chain_curve_kernel_state": cst["state"], "chain_regs_per_thread": cst["regs_per_thread"], "chain_local_bytes": cst["local_bytes"],
           "us_per_block_chain": round(us["chain"], 2), "us_per_block_sequential": round(us["sequential"], 2),
           "speedup": round(us["sequential"] / us["chain"], 3),
           "bytes_per_instance_sample_chain": bytes_fused, "bytes_per_instance_sample_sequential": bytes_seq,
           "hbm_share_chain": round(bytes_fused * n * S / (us["chain"] * 1e-6) / HBM_BYTES_PER_S, 3),
           "hbm_share_sequential": round(bytes_seq * n * S / (us["sequential"] * 1e-6) / HBM_BYTES_PER_S, 3),
           "reps_us_chain": [round(v, 2) for v in times["chain"]], "reps_us_sequential": [round(v, 2) for v in times["sequential"]],
           "chain_equals_sequential": bool(np.array_equal(y_last.view(np.uint32), s_last.view(np.uint32))),
           "oracle_first_call": first_ok, "oracle_last_timed_call": last_ok, "sampled_instances": len(idx)}
    chain.close()
    for g in stages:
        g.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(HERE), "profiles", "r08_chain_curves_bench.jsonl"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("chain_curves_bench needs a GPU")
    name, power = gpu_identity()
    three = [progs.CFG2_LOG_GAIN, progs.CFG1A_TESTCODE, cc.LIMIT]
    cases = [("a: cfg2 -> testcode volume (per-instance curve) -> limit", three, 65536, [(1, "volume", False)]),
             ("b: cfg2 -> testcode volume (broadcast ramp) -> limit", three, 65536, [(1, "volume", True)]),
             ("c: cfg2 -> testcode volume (per-instance curve) -> limit", three, 4096, [(1, "volume", False)]),
             ("d: cfg2 -> cfg4 (per-instance cutoff curve)", [progs.CFG2_LOG_GAIN, progs.CFG4_ONEPOLE], 65536, [(1, "filter_cutoff", False)])]
    with open(a.out, "w") as f:
        for label, texts, n, curve_names in cases:
            row = run_case(torch, label, texts, n, curve_names, a.calls, a.warmup, a.reps)
            row.update({"gpu": name, "power_limit": power})
            print(json.dumps(row), flush=True)
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
