"""Measures program chains over host buffers (fx8010_chain_process_batch_host(_curves), fx8010_multi_chain_*) against the two ways a caller
had without them: the stages' own process_batch_host calls through a host temporary, and the device chain call with hand-made copies.

    python tests/chain_host_bench.py [--calls 10] [--warmup 2] [--reps 3] [--out FILE]

Cases (1 024 periods per block, page-locked buffers, translator in mode 2 on every stage):
    (a) cfg2 (LOG waveshaper + gain) -> volume -> limiter, 65 536 instances: fused, 268 MB per block each way over PCIe;
    (b) the same with a per-instance volume curve: one more 268 MB host->device stream per block;
    (c) cfg4 (one-pole low-pass) -> cfg2, 65 536 instances: a stage with state, so every form runs stage by stage;
    (d) case (a) on an executor chain over every GPU (two shards on GPU 0 when there is one).

Per case and form, microseconds per block: a host clock around `calls` back-to-back blocking calls after `warmup` calls, the median of `reps`
repetitions, the forms alternating on the same handles.  Forms:
    host_chain      the host chain call (one PCIe round trip per sub-block, whatever the number of stages);
    per_stage_host  stage j's fx8010_gpu_process_batch_host (with its curves) from the previous stage's host output (k round trips);
    device_chain    one host->device copy of the block (and the curves), the device chain call, one device->host copy, on one stream
                    (unpipelined; not available on an executor chain).
The last call of every timed batch is compared bit for bit with twin handles that ran the same number of blocks stage by stage on device
copies.  The bytes each form moves over PCIe per instance-sample are reported, and the GPU's name and power limit are read in the same run.  Needs a GPU: without one it fails.
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
import chain_common as cc  # noqa: E402
import progs  # noqa: E402
from curves_bench import gpu_identity  # noqa: E402

fx = importlib.import_module("fx8010-emulator-core_b200")
S = 1024
VOLUME = "\n".join(["input in_l 0", "control volume = 0.5", "output out_l 0", "macs out_l, 0, in_l, volume", "end"])


def run_case(torch, label, texts, n, curve_names, devices, calls, warmup, reps):
    """curve_names: [(stage, register name)], per-instance curves; devices: None for one GPU, else the executor's ordinals."""
    rng = np.random.default_rng(0x8010)
    prog_list = [fx.Program(t) for t in texts]
    objs = []
    for p in prog_list:
        o = fx.Gpu(n, 1) if devices is None else fx.MultiGpu(devices, n, 1)
        o.load_program(p)
        o.set_option(fx.OPT_TRANSLATE, 2)
        for nm in p.controls():
            o.set_controls(p.reg_index(nm), (0.05 + 0.95 * rng.random(n)).astype(np.float32))
        objs.append(o)
    chain = fx.Chain(objs) if devices is None else fx.MultiChain(objs)
    keep = []

    def pinned(shape):
        a, owner = fx.pinned_array(shape)
        keep.append(owner)
        return a

    x, y, ref, tmp = pinned((1, S, n)), pinned((1, S, n)), pinned((1, S, n)), pinned((1, S, n))
    x[:] = (1.8 * rng.random((1, S, n)) - 0.9).astype(np.float32)
    curves = [(j, prog_list[j].reg_index(nm), False) for j, nm in curve_names]
    vals = []
    for _ in curves:
        v = pinned((S, n)); v[:] = (0.05 + 0.95 * rng.random((S, n))).astype(np.float32); vals.append(v)
    chain_list = [(j, r, v, bc) for (j, r, bc), v in zip(curves, vals)]

    def host_chain():
        chain.process_host_curves(x, chain_list, out=y)

    def per_stage_host():
        cur = x
        for j, o in enumerate(objs):
            out = ref if j + 1 == len(objs) else (tmp if cur is not tmp else y)
            mine = [(r, v, bc) for (st, r, v, bc) in chain_list if st == j]
            o.process_host_curves(cur, mine, out=out)
            cur = out

    forms = {"host_chain": host_chain, "per_stage_host": per_stage_host}
    if devices is None:
        d_x, d_y = torch.empty((1, S, n), device="cuda"), torch.empty((1, S, n), device="cuda")
        d_v = [torch.empty((S, n), device="cuda") for _ in vals]
        tx, ty, tv = torch.from_numpy(x), torch.from_numpy(y), [torch.from_numpy(v) for v in vals]

        def device_chain():
            d_x.copy_(tx, non_blocking=True)
            for d, t in zip(d_v, tv):
                d.copy_(t, non_blocking=True)
            chain.process_batch_curves(d_x, d_y, S, [(j, r, d, bc) for (j, r, bc), d in zip(curves, d_v)],
                                       torch.cuda.current_stream().cuda_stream)
            ty.copy_(d_y, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        forms["device_chain"] = device_chain
    # The reference: twin handles on one GPU running the stage-by-stage form on device copies, as many blocks as the timed handles ran
    # (the input is the same every block, so after m blocks every form has left the same state; a stage with state makes that matter).
    twins = []
    for p, o in zip(prog_list, objs):
        g = fx.Gpu(n, 1); g.load_program(p); g.set_option(fx.OPT_TRANSLATE, 2)
        for nm in p.controls():
            g.set_controls(p.reg_index(nm), o.get_register(p.reg_index(nm)))
        twins.append(g)
    t_x = torch.from_numpy(x).cuda()
    t_v = [torch.from_numpy(v).cuda() for v in vals]
    t_mid = [torch.empty_like(t_x) for _ in range(2)]
    t_out = torch.empty_like(t_x)

    def twins_run(m):
        for _ in range(m):
            cur = t_x
            for j, g in enumerate(twins):
                out = t_out if j + 1 == len(twins) else t_mid[j & 1]
                mine = [(r, d, bc) for (st, r, bc), d in zip(curves, t_v) if st == j]
                if mine:
                    g.process_device_curves(cur, out, S, mine)
                else:
                    g.process_device(cur, out, S)
                cur = out
        torch.cuda.synchronize()
        return t_out.cpu().numpy()

    for _ in range(warmup):
        for fn in forms.values():
            fn()
    twins_run(warmup * len(forms))
    times = {k: [] for k in forms}
    exact = True
    for _ in range(reps):
        for name, fn in forms.items():
            t0 = time.perf_counter()
            for _ in range(calls):
                fn()
            times[name].append((time.perf_counter() - t0) * 1e6 / calls)
            got = ref if name == "per_stage_host" else y
            exact = exact and bool(np.array_equal(got.view(np.uint32), twins_run(calls).view(np.uint32)))
    st = chain.status() if devices is None else chain.shard_status(0)
    us = {k: float(np.median(v)) for k, v in times.items()}
    k = len(texts)
    n_cv = len(curves)
    row = {"case": label, "instances": n, "periods": S, "stages": k, "devices": devices or [0], "per_instance_curves": n_cv,
           "fused": st["fused_last"], "why_not_fused": st["message"],
           **{f"us_per_block_{name}": round(v, 1) for name, v in us.items()},
           "pcie_bytes_per_instance_sample_host_chain": 4.0 * (2 + n_cv),
           "pcie_bytes_per_instance_sample_per_stage_host": 8.0 * k + 4.0 * n_cv,
           **{f"reps_us_{name}": [round(v, 1) for v in t] for name, t in times.items()},
           "every_batch_equals_stage_by_stage": exact}
    chain.close()
    for o in objs + twins:
        o.close()
    del keep
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(HERE), "profiles", "r09_chain_host_bench.jsonl"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("chain_host_bench needs a GPU")
    name, power = gpu_identity()
    three = [progs.CFG2_LOG_GAIN, VOLUME, cc.LIMIT]
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    cases = [("a: cfg2 -> volume -> limit", three, 65536, [], None),
             ("b: cfg2 -> volume (per-instance curve) -> limit", three, 65536, [(1, "volume")], None),
             ("c: cfg4 -> cfg2", [progs.CFG4_ONEPOLE, progs.CFG2_LOG_GAIN], 65536, [], None),
             ("d: cfg2 -> volume -> limit on an executor chain", three, 65536, [], devs)]
    with open(a.out, "w") as f:
        for label, texts, n, curve_names, devices in cases:
            row = run_case(torch, label, texts, n, curve_names, devices, a.calls, a.warmup, a.reps)
            row.update({"gpu": name, "power_limit": power})
            print(json.dumps(row), flush=True)
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
