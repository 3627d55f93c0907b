"""Shared by tests/test_curves_translate.py, tests/test_gpu_curves.py and tests/curves_bench.py: the programs whose controls get
automated, curve generation, and the reference for a call with control curves — the oracle stepped one sample period at a time with
set_register before each period (what fx8010_gpu_process_batch_curves is defined to equal)."""
from __future__ import annotations

import numpy as np

import progs

# a delay line whose feedback is a control (a ring of 200: periods closer than 200 are independent)
DELAY_FB = "\n".join(["static a", "static rd", "control fb = 0.5", "input in_l 0", "output out_l 0", "itramsize 200 ",
                      "idelay read, rd, at, 0", "macs a, in_l, rd, fb", "idelay write, a, at, 0", "macs out_l, in_l, rd, 0.5", "end"])
# a modulated delay (chorus / flanger): read and write offsets are controls, so a curve moves the delay time every period
DELAY_MOD = "\n".join(["static a", "static rd", "control roff = 30", "control woff = 4", "input in_l 0", "output out_l 0", "itramsize 200 ",
                       "idelay read, rd, at, roff", "macs a, in_l, rd, 0.5", "idelay write, a, at, woff", "macs out_l, in_l, rd, 0.5", "end"])
# LOG with the table selector in a control: integer values pick the table per period (stateless)
LOG_SELECT = "\n".join(["static a", "control sel = 3", "input in_l 0", "output out_l 0", "log a, in_l, sel, 0", "macs out_l, 0, a, 0.75", "end"])
# SKIP with a constant count and an automated data control
SKIP_DATA = "\n".join(["static a", "control g = 0.5", "input in_l 0", "output out_l 0", "macs a, in_l, g, 0.5", "skip ccr, ccr, 2, 1",
                       "macs a, a, g, 0.5", "macs out_l, a, g, 1.0", "end"])
# SKIP whose count is a STATIC register (a translation-time constant until it is automated)
SKIP_COUNT = "\n".join(["static n = 1", "static a", "input in_l 0", "output out_l 0", "macs a, in_l, 0.5, 0.5", "skip ccr, ccr, 2, n",
                        "macs a, a, 0.5, 0.5", "macs out_l, a, 0.25, 1.0", "end"])
# two channels, one control per channel path
TWO_CH = "\n".join(["input in_l 0", "input in_r 1", "output out_l 0", "output out_r 1", "static t", "control gl = 0.5", "control gr = 0.25",
                    "macs t, in_l, in_r, gl", "interp out_l, out_l, gl, t", "macs out_r, in_r, in_l, gr", "end"])


def programs():
    """name -> (text, channels, [(register name, broadcast)])"""
    return {
        "cfg2_instance": (progs.CFG2_LOG_GAIN, 1, [("volume", False)]),
        "cfg2_broadcast": (progs.CFG2_LOG_GAIN, 1, [("volume", True)]),
        "cfg4_cutoff": (progs.CFG4_ONEPOLE, 1, [("filter_cutoff", False)]),
        "delay_fb": (DELAY_FB, 1, [("fb", False)]),
        "delay_mod": (DELAY_MOD, 1, [("roff", False), ("woff", True)]),
        "log_select": (LOG_SELECT, 1, [("sel", True)]),
        "skip_data": (SKIP_DATA, 1, [("g", False)]),
        "cfg5": (progs.cfg5_allops(), 1, [("k0", False), ("k1", True), ("k2", False), ("k3", True)]),
        "two_channels": (TWO_CH, 2, [("gl", False), ("gr", True)]),
    }


def make_curve(name: str, reg_name: str, broadcast: bool, s: int, n: int, rng: np.random.Generator) -> np.ndarray:
    """[S][N] (or [S] when broadcast) float32 values a user would send: ramps, an LFO, integer table selectors."""
    t = np.arange(s, dtype=np.float64)[:, None]
    i = np.arange(1 if broadcast else n, dtype=np.float64)[None, :]
    if reg_name == "sel":
        v = np.floor((t * 7 + i * 3) % 34) - 1                   # -1..32: the out-of-range selectors raise the table flag
    elif reg_name in ("roff", "woff"):                           # delay offsets in periods (integers; the ring is 200 long)
        v = np.floor(60 + 45 * np.sin(2 * np.pi * (t / 53.0 + i / 7.0))) if reg_name == "roff" else np.floor(6 + 5 * np.sin(2 * np.pi * t / 31.0)) + 0 * i
    elif reg_name == "filter_cutoff":
        v = 0.001 + 0.998 * (0.5 + 0.5 * np.sin(2 * np.pi * (t / 97.0 + i / 13.0)))
    else:
        v = rng.uniform(-1.0, 1.0, size=(s, i.shape[1]))
        v[: s // 2] = np.linspace(0.0, 1.0, s // 2 + 2)[1:-1, None] * (1 + i[:, :] % 3) / 3.0
    v = v.astype(np.float32)
    return v[:, 0].copy() if broadcast else np.ascontiguousarray(v)


def oracle_stepped(orc, x, curves, s: int):
    """curves: [(register index, values, broadcast)].  Runs the oracle period by period with set_register before each one."""
    outs = []
    for k in range(s):
        for reg, vals, bc in curves:
            orc.set_register(reg, np.full(orc.n, vals[k], np.float32) if bc else vals[k])
        outs.append(orc.process(None if x is None else x[:, k:k + 1, :], 1))
    return np.concatenate(outs, axis=1)
