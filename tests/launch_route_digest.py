"""One-off check that a change to the launch path leaves every routing decision untouched.

Runs a fixed matrix of programs, instance counts, translation modes, call kinds and developer switches on the GPU and prints one
line per call: the return code, the launches the call added, every launch_info field, the translator's state (plain, and state and
kind for control curves), the process's NVRTC compile count, and SHA-256 digests of the outputs, registers, instruction counters and
scalars.  Inputs come from fixed seeds.  Run it on two builds and diff the outputs:

    python tests/launch_route_digest.py --root parent > before.txt     # a checkout of the parent commit, built
    python tests/launch_route_digest.py > after.txt                     # this tree
    diff before.txt after.txt                                           # empty: same kernels, geometry, outputs and compiles

--digest prints one line per handle instead: the number of its call lines and the SHA-256 of their text (the form kept in profiles/;
rerun without it to see which call differs).  Needs a GPU.
"""
import argparse
import hashlib
import importlib
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(HERE), help="checkout whose package is imported")
ap.add_argument("--digest", action="store_true", help="one SHA-256 per handle instead of one line per call")
args = ap.parse_args()
sys.path[:0] = [HERE, os.path.abspath(args.root)]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import progs  # noqa: E402

fx = importlib.import_module("fx8010-emulator-core_b200")
SWITCHES = ["FX8010_NO_STATELESS", "FX8010_NO_TSPLIT", "FX8010_NO_SHORT", "FX8010_NO_PDL", "FX8010_TR_RECUR", "FX8010_USE_TMA"]
LINES = []                                                        # the current handle's call lines
SHORT = "static a\ninput in_l 0\noutput out_l 0\nmacs a, 0, in_l, 0.5\nmacs out_l, 0, a, 0.25\nend"


def programs():
    yield "cfg1", progs.CFG1A_TESTCODE, 1
    yield "cfg2", progs.CFG2_LOG_GAIN, 1
    for size in (100, 1000, 8192, 65536):
        yield f"cfg3_{size}", progs.cfg3_delay(size), 1
    yield "cfg4", progs.CFG4_ONEPOLE, 1
    yield "cfg5", progs.cfg5_allops(), 1
    yield "short", SHORT, 1
    yield "skip", progs.SNIPPETS["skip"], 1
    for seed in range(4):
        rng = np.random.default_rng(9100 + seed)
        yield f"random_{seed}", progs.random_program(rng, 24 + 8 * seed, xtram=seed % 2 == 1, skip=seed >= 2), 1


def h(*arrays):
    d = hashlib.sha256()
    for a in arrays:
        d.update(np.ascontiguousarray(a.cpu().numpy() if torch.is_tensor(a) else a).tobytes())
    return d.hexdigest()[:16]


def report(case, g, rc, before):
    i = g.launch_info()
    t, tc = g.translate_status(), g.translate_status_curves()
    torch.cuda.synchronize()
    acc, lfsr, latch, ptrs = g.scalars()
    fields = " ".join(f"{n}={getattr(i, n)}" for n, _ in i._fields_ if n not in ("kernel_launches", "reserved"))
    return (f"{case} rc={rc} launches={i.kernel_launches - before} {fields} tr={t['state']} trc={tc['state']}/{tc['kind']} "
            f"compiles={fx.kernel_cache_stats()['nvrtc_compiles']} regs={h(g.registers())} counts={h(g.counts())} "
            f"scalars={h(acc, lfsr, latch, ptrs)}")


def call(case, g, fn, outs):
    before = g.launch_info().kernel_launches
    try:
        fn()
        rc = 0
    except fx.FxError as e:
        rc = e.code
    LINES.append(report(case, g, rc, before) + f" out={h(*outs)}")


def flush(tag):
    text = "\n".join(LINES)
    print(f"{tag} calls={len(LINES)} sha256={hashlib.sha256(text.encode()).hexdigest()[:16]}" if args.digest else text, flush=True)
    LINES.clear()


def control_reg(prog):
    for k, r in enumerate(prog.registers()):
        if r[0] in (0, 2) and not r[3].startswith(("ccr", "noise")):
            return k
    return None


def run_handle(name, text, ch, n, mode, env, calls="all"):
    for k in SWITCHES:
        os.environ.pop(k, None)
    os.environ.update(env)
    prog = fx.Program(text, channels=ch, instances=n)
    g = fx.Gpu(n, ch)
    g.load_program(prog)
    g.set_option(fx.OPT_TRANSLATE, mode)
    tag = f"{name} n={n} mode={mode} env={','.join(f'{k}={v}' for k, v in env.items()) or '-'}"
    gen = torch.Generator(device="cuda").manual_seed(n + mode)
    S = 1024
    x = torch.rand((ch, S, n), generator=gen, device="cuda") * 2 - 1
    y = torch.zeros_like(x)
    call(f"{tag} device", g, lambda: g.process_device(x, y, S), [y])
    if calls == "all":
        xb = torch.rand(ch * S * n + 1, generator=gen, device="cuda")
        yb = torch.zeros_like(xb)
        call(f"{tag} device_offset", g, lambda: g.process_device(xb[1:], yb[1:], S), [yb])
    for nb in ((3, 40) if calls == "all" else (3,)):
        xs = [torch.rand((ch, 128, n), generator=gen, device="cuda") for _ in range(nb)]
        ys = [torch.zeros_like(v) for v in xs]
        call(f"{tag} blocks{nb}", g, lambda: g.process_blocks(xs, ys, 128), ys)
    if calls != "all":
        return flush(tag)
    xs = [torch.rand((ch, 128, n), generator=gen, device="cuda") for _ in range(3)]
    ys = [torch.zeros_like(v) for v in xs]
    call(f"{tag} blocks_null", g, lambda: g.process_blocks([xs[0], None, xs[2]], ys, 128), ys)
    for s in (1, 7):
        call(f"{tag} periods{s}", g, lambda: g.process_device(x[:, :s].contiguous(), y[:, :s], s), [y])
    reg = control_reg(prog)
    if reg is not None:
        ev = [(0, reg, 0.25), (100, reg, np.linspace(0, 1, n, dtype=np.float32)), (700, reg, -0.5)]
        call(f"{tag} events", g, lambda: g.process_device_events(x, y, S, ev), [y])
        cv = torch.rand((S, n), generator=gen, device="cuda") * 0.5
        call(f"{tag} curves", g, lambda: g.process_device_curves(x, y, S, [(reg, cv, False)]), [y])
        cvu = torch.rand(S * n + 1, generator=gen, device="cuda") * 0.5
        call(f"{tag} curves_unaligned", g, lambda: g.process_device_curves(x, y, S, [(reg, cvu[1:], False)]), [y])
        cb = torch.rand(S, generator=gen, device="cuda") * 0.5
        call(f"{tag} curves_bcast", g, lambda: g.process_device_curves(x, y, S, [(reg, cb, True)]), [y])
    xp = x.reshape(ch, S, n).permute(0, 2, 1).contiguous()
    yp = torch.zeros_like(xp)
    call(f"{tag} planar", g, lambda: g.process_device_planar(xp, yp, S), [yp])
    xh = x.cpu().numpy()
    res = {}
    call(f"{tag} host", g, lambda: res.setdefault("y", g.process_host(xh)), [np.zeros(1)])
    LINES.append(f"{tag} host_out={h(res.get('y', np.zeros(1)))}")
    d = g.dims()
    if d.itram_size > 0 or d.xtram_size > 0:                     # rows 0, 1: iTRAM write / read pointer; rows 2, 3: xTRAM
        ptrs = g.scalars()[3]
        for j, size in enumerate((d.itram_size, d.itram_size, d.xtram_size, d.xtram_size)):
            if size > 0:
                ptrs[j] = (ptrs[j] + 3) % size
        g.set_scalars(ptrs=ptrs)
        call(f"{tag} moved_ptrs", g, lambda: g.process_device(x, y, S), [y])
    flush(tag)
    g.close()
    prog.close()


def counter_split(mode):
    """A stateless program long enough that one call of 600 000 periods exceeds the 32-bit counter limit (536 870 periods)."""
    for k in SWITCHES:
        os.environ.pop(k, None)
    prog = fx.Program(progs.CFG2_LOG_GAIN, channels=1, instances=1)
    ins, regs = prog.instructions(), prog.registers()
    instrs = [ins[0]] * (1000 - len(ins)) + list(ins)
    n, S = 64, 600_000
    g = fx.Gpu(n, 1)
    g.load(instrs, regs, tables=prog.tables())
    g.set_option(fx.OPT_TRANSLATE, mode)
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = torch.rand((1, S, n), generator=gen, device="cuda")
    y = torch.zeros_like(x)
    call(f"counter_split mode={mode} n_instrs={len(instrs)}", g, lambda: g.process_device(x, y, S), [y])
    flush(f"counter_split mode={mode}")
    g.close()
    prog.close()


for mode in (0, 2):
    for name, text, ch in programs():
        for n in (4096, 4094, 64):
            run_handle(name, text, ch, n, mode, {})
    for name, text, ch in programs():
        if name not in ("cfg2", "cfg3_100", "cfg3_8192", "cfg4", "cfg5"):
            continue
        for env in ({"FX8010_NO_STATELESS": "1"}, {"FX8010_NO_TSPLIT": "1"}, {"FX8010_NO_SHORT": "1"}, {"FX8010_NO_PDL": "1"},
                    {"FX8010_TR_RECUR": "3"}, {"FX8010_USE_TMA": "2"}):
            run_handle(name, text, ch, 4096, mode, env, calls="some")
    counter_split(mode)
