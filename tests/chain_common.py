"""Shared by tests/test_chain_translate.py, tests/test_gpu_chain.py and tests/chain_bench.py: the stateless stages chains are built from,
the chains themselves, and the reference for a chain call — the oracles of the stages stepped one sample period at a time, stage after
stage (what fx8010_chain_process_batch is defined to equal)."""
from __future__ import annotations

import numpy as np

import progs

# a two-sided limiter: min(in, ceil), then max(that, -0.5)
LIMIT = "\n".join(["static a", "input in_l 0", "control ceil = 0.5", "output out_l 0",
                   "limitn a, in_l, in_l, ceil", "limit out_l, a, a, -0.5", "end"])
# two channels: a cross-mix and a LOG shaper on the right channel
TWO_CH_MIX = "\n".join(["static t", "static u", "input in_l 0", "input in_r 1", "control g = 0.5", "output out_l 0", "output out_r 1",
                        "macs t, in_l, in_r, g", "log u, in_r, 5, 0", "macs out_l, 0, t, 0.75", "macsn out_r, u, in_l, 0.25", "end"])
# two channels: a pan-like gain pair
TWO_CH_GAIN = "\n".join(["input in_l 0", "input in_r 1", "control gl = 0.5", "control gr = 0.25", "output out_l 0", "output out_r 1",
                         "macs out_l, 0, in_l, gl", "macs out_r, in_r, in_l, gr", "end"])


def random_stateless(seed: int, channels: int = 1) -> str:
    """A seeded random program (progs.random_program) the product's analysis calls stateless: the first of a seeded series of short
    SKIP-, TRAM- and noise-free ones; a fixed LOG / LIMIT / EXP program with seed-dependent tables when none of them is."""
    import importlib
    fx = importlib.import_module("fx8010-emulator-core_b200")
    for k in range(200):
        rng = np.random.default_rng(9100 + 997 * seed + k)
        text = progs.random_program(rng, 5 + k % 4, channels=channels, n_static=3, n_controls=1, skip=False, tram=False, noise=False,
                                    ops=progs.SAT_OPS + progs.TABLE_OPS + ["limit", "tstneg", "andxor"])
        prog = fx.Program(text, channels=channels)
        src, _ = fx.translate_source(prog, channels)
        prog.close()
        if src is not None and "fx_translated_sl" in src and "#define FXT_NTR 0" in src:
            return text
    lines = ["static a", "static b", "control g = 0.5", "input in_l 0", "output out_l 0", "macs a, 0, in_l, g", f"log b, a, {seed % 32}, 0",
             "limit a, b, a, 0.25", f"exp b, a, {(7 * seed + 3) % 32}, 0", "macsn out_l, b, a, g"]
    if channels == 2:
        lines[4:4] = ["input in_r 1", "output out_r 1"]
        lines.append("macs out_r, in_l, in_r, g")
    return "\n".join(lines + ["end"])


def chain_texts(name: str):
    """name -> (stage texts, channels)."""
    one = [progs.CFG1A_TESTCODE, progs.CFG1B_LOGTUBE, progs.CFG2_LOG_GAIN, LIMIT]
    if name == "two":
        return [progs.CFG2_LOG_GAIN, progs.CFG1A_TESTCODE], 1
    if name == "three":
        return [progs.CFG2_LOG_GAIN, progs.CFG1A_TESTCODE, LIMIT], 1
    if name == "eight":
        return one + [random_stateless(0), progs.CFG2_LOG_GAIN, random_stateless(1), LIMIT], 1
    if name == "two_ch_two":
        return [TWO_CH_MIX, TWO_CH_GAIN], 2
    if name == "two_ch_three":
        return [TWO_CH_GAIN, random_stateless(2, channels=2), TWO_CH_MIX], 2
    if name == "two_ch_eight":
        return [TWO_CH_MIX, TWO_CH_GAIN, progs.CFG2_LOG_GAIN, random_stateless(3, channels=2), TWO_CH_MIX, LIMIT, TWO_CH_GAIN,
                random_stateless(4, channels=2)], 2
    raise KeyError(name)


CHAINS = ["two", "three", "eight", "two_ch_two", "two_ch_three", "two_ch_eight"]


def controls(prog, n: int, rng: np.random.Generator) -> dict:
    """Per-instance values for every control of a stage (kept out of the immediates), in [0.05, 1)."""
    return {nm: (0.05 + 0.95 * rng.random(n)).astype(np.float32) for nm in prog.controls()}


def oracle_chain_stepped(orcs, x, s: int):
    """Runs the stages' oracles one sample period at a time, stage after stage; x [C][S][N] or None.  Returns [C][S][N]."""
    outs = []
    for k in range(s):
        y = None if x is None else np.ascontiguousarray(x[:, k:k + 1, :])
        for orc in orcs:
            y = orc.process(y, 1)
        outs.append(y)
    return np.concatenate(outs, axis=1)
