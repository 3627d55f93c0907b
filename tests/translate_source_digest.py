"""One-off check that a change to the translator leaves the generated source of plain (curve-free) calls untouched.

Prints one line per program of the corpus (tests/progs.py: the cfg1-cfg5 programs, the feature snippets, seeded random programs)
and instance count: the SHA-256 of what fx8010_translate_source returns, or "declined".  Run it on two builds and diff the outputs:

    python tests/translate_source_digest.py > before.txt      # on the parent commit's build
    python tests/translate_source_digest.py > after.txt       # on this one
    diff before.txt after.txt                                  # empty: byte-identical sources

(FX8010_TR_* developer switches change the source on purpose: leave them unset.)  Needs no GPU.
"""
import hashlib
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [HERE, os.path.dirname(HERE)]
import progs  # noqa: E402

fx = importlib.import_module("fx8010-emulator-core_b200")


def corpus():
    yield "cfg1a", progs.CFG1A_TESTCODE, 1
    yield "cfg1b", progs.CFG1B_LOGTUBE, 1
    yield "cfg2", progs.CFG2_LOG_GAIN, 1
    for size in (100, 200, 1000, 8192):
        yield f"cfg3_{size}", progs.cfg3_delay(size), 1
    yield "cfg4", progs.CFG4_ONEPOLE, 1
    yield "cfg5", progs.cfg5_allops(), 1
    yield "end_skipped_wrap", progs.END_SKIPPED_WRAP, 1
    for name, text in progs.SNIPPETS.items():
        yield "snippet_" + name, text, 1
    for seed in range(24):
        rng = np.random.default_rng(7000 + seed)
        ch = 1 + seed % 2
        yield f"random_{seed}", progs.random_program(rng, 20 + 5 * seed, channels=ch, xtram=bool(seed % 3 == 0), skip=bool(seed % 4)), ch


def main():
    for name, text, ch in corpus():
        prog = fx.Program(text, channels=ch, relaxed=True)
        assert prog.loaded, (name, prog.errors())
        for n in (1, 300, 4096, 65536):
            src, _ = fx.translate_source(prog, ch, instances=n)
            digest = "declined" if src is None else hashlib.sha256(src.encode()).hexdigest()
            print(f"{name} n={n} {digest}")
        prog.close()


if __name__ == "__main__":
    main()
