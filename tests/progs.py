"""Program texts and stimuli shared by tests/, bench.py and tests/golden/make_golden.py.

The named configurations follow SURVEY.md §8(d) / BASELINE.json `configs`; the random generator
produces `.da` sources in the reference's dialect (reference source/testcode.da shows one snippet
per feature, source/FX8010.cpp:365-741 is the grammar).
"""
from __future__ import annotations

import numpy as np

SEED = 0x8010

# ---- BASELINE.json configs ----------------------------------------------------------------------

# config 1(a): the shipped program, verbatim semantics (reference source/testcode.da:24) without the
# comment lines; declarations kept in file order so the register indices match the shipped file.
CFG1A_TESTCODE = """name "testcode"
copyright "2023, klangraum"
static a
itramsize 1000 
xtramsize 48000 
input in_l 0
control volume = 1.0
control pan = 0.5
control filter_cutoff = 0.1
output out_l 0
static rd
static wr
static noise
macs out_l, 0, in_l, volume
end"""

# config 1(b): README variant, LOG tube + MACS output (reference README.md:33-35)
CFG1B_LOGTUBE = """static a
input in_l 0
control volume = 0.5
output out_l 0
log a, in_l, 3, 0
macs out_l, 0, a, 1.0
end"""

# config 2: MACS gain + LOG waveshaper (BASELINE.json configs[1]; the bench workload)
CFG2_LOG_GAIN = """static a
input in_l 0
control volume = 1.0
output out_l 0
log a, in_l, 3, 0
macs out_l, 0, a, volume
end"""


def cfg3_delay(size: int) -> str:
    """config 3: idelay feedback delay line, read-before-write => delay = itramsize, no UB.
    (`itramsize N` needs one trailing blank to pass the reference's regex, source/FX8010.cpp:377.)"""
    return f"""static a
static rd
input in_l 0
output out_l 0
itramsize {size} 
idelay read, rd, at, 0
macs a, in_l, rd, 0.5
idelay write, a, at, 0
macs out_l, in_l, rd, 0.5
end"""


# config 4: INTERP one-pole low-pass (reference source/testcode.da:44)
CFG4_ONEPOLE = """input in_l 0
control filter_cutoff = 0.1
output out_l 0
interp out_l, out_l, filter_cutoff, in_l
end"""

# END is skipped while `a` is in (0,1); `a` advances by a wrapping 0.3 per pass, so every sample period
# ends after at most 4 passes (a program that always skips END hangs the reference, SURVEY U9).
END_SKIPPED_WRAP = "static a\noutput out_l 0\nmacintw a, a, 0.3, 1.0\nmacs out_l, 0, a, 1.0\nskip ccr, ccr, 2, 1\nend"

SNIPPETS = {
    # one per commented feature snippet of reference source/testcode.da:26-57
    "exp": "static a\ninput in_l 0\noutput out_l 0\nexp a, in_l, 7, 0\nmacs out_l, 0, a, 1.0\nend",
    "interp_const": "control pan = 0.5\noutput out_l 0\ninterp out_l, -0.25, pan, 0.25\nend",
    "highpass": "static a\ninput in_l 0\ncontrol filter_cutoff = 0.1\noutput out_l 0\n"
                "interp a, a, filter_cutoff, in_l\nmacsn out_l, in_l, a, 1\nend",
    "skip": "static a\ninput in_l 0\noutput out_l 0\nmacs a, 0, in_l, 1.0\nskip ccr, ccr, 2, 1\n"
            "macs a, 0, a, 0.5\nmacs out_l, 0, a, 1.0\nend",
    "andxor": "static a\noutput out_l 0\nandxor a, 5, 3, -4\nmacs out_l, 0, a, 0.1\nend",
    "noise": "static noise\noutput out_l 0\nmacs out_l, 0, noise, 1.0\nend",
    "delay_fb_testcode": "static a\nstatic rd\ninput in_l 0\noutput out_l 0\nitramsize 1000 \n"
                         "macs a, in_l, rd, 0.1\nidelay write, a, at, 0\nidelay read, rd, at, 0\n"
                         "macs out_l, in_l, rd, 0.5\nend",
}


# ---- stimuli -------------------------------------------------------------------------------------

def sine_bank(n_instances: int, n_samples: int, rng: np.random.Generator, start: int = 0,
              amp_lo: float = 0.05, amp_hi: float = 0.99) -> np.ndarray:
    """Per-instance sines f_i = 55*2^((i mod 96)/12) Hz at 48 kHz, amplitude in [amp_lo, amp_hi);
    returns [S][N] float32 (double sin, then round) — SURVEY.md §8(d) config 2/4/5 stimulus."""
    i = np.arange(n_instances)
    f = 55.0 * 2.0 ** ((i % 96) / 12.0)
    amp = amp_lo + (amp_hi - amp_lo) * rng.random(n_instances)
    n = np.arange(start, start + n_samples)[:, None]
    return (amp[None, :] * np.sin(2.0 * np.pi * f[None, :] * n / 48000.0)).astype(np.float32)


def impulse_noise(n_instances: int, n_samples: int, rng: np.random.Generator) -> np.ndarray:
    """config 3 stimulus: unit impulse at n=0 plus 0.25-amplitude noise; [S][N] float32."""
    x = (0.25 * (2.0 * rng.random((n_samples, n_instances)) - 1.0)).astype(np.float32)
    x[0, :] = 1.0
    return x


# LOG / EXP input values outside the tables' domain, where rule U6 defines the result (index clamped, FX8010_RT_TABLE_RANGE set):
# |A| > 1 up to the largest finite value, signed zeros, subnormals, and a NaN.  The NaN is quiet, positive and carries every payload
# bit: the one NaN an IEEE operation produces on the GPU and propagates unchanged on the CPU.  (Infinities are left out: where a table
# row is flat, its zero slope times an infinite distance is an invalid operation, whose NaN is 0xffc00000 on x86 and 0x7fffffff on
# the GPU.)
TABLE_EDGE_BITS = [0x3f800001, 0xbf800001, 0x3fc00000, 0xbfc00000, 0x40000000, 0xc0000000, 0x7149f2ca, 0xf149f2ca, 0x7f7fffff, 0xff7fffff,
                   0x00000000, 0x80000000, 0x00000001, 0x80000001, 0x007fffff, 0x807fffff, 0x00400000, 0x80012345,
                   0x7fffffff]


def table_sweep_grid(n: int, rng: np.random.Generator) -> np.ndarray:
    """n float32 LOG / EXP inputs: every table boundary of [-1, 1] and both of its float32 neighbours, the U6 edge values above,
    then uniform values in [-1, 1)."""
    k = np.arange(64)
    bounds = (-1.0 + k * (2.0 / 63)).astype(np.float32)
    near = np.concatenate([np.nextafter(bounds, np.float32(-2)), bounds, np.nextafter(bounds, np.float32(2))]).astype(np.float32)
    edge = np.array(TABLE_EDGE_BITS, dtype=np.uint32).view(np.float32)
    head = np.concatenate([near, edge]).astype(np.float32)
    return np.concatenate([head, (2 * rng.random(n - head.size) - 1).astype(np.float32)]).astype(np.float32)


# ---- random programs -----------------------------------------------------------------------------

SAT_OPS = ["macs", "macsn", "macints", "acc3", "interp"]
WRAP_OPS = ["macw", "macwn", "macintw"]
WIDE_OPS = ["andxor", "tstneg", "limit", "limitn", "macmv"]
TABLE_OPS = ["log", "exp"]
CCR_VALUES = [0, 2, 6, 8, 16, 20]
LITERALS = ["0", "1", "0.5", "-0.5", "0.25", "-0.25", "0.75", "1.0", "-1", "0.125", "0.999", "-0.875",
            "0.0", "0.3", "-0.7", "0.01"]
INT_LITERALS = ["0", "1", "2", "3", "5", "-4", "-1", "7", "16777215", "-2"]


def random_program(rng: np.random.Generator, n_instr: int, *, channels: int = 1, n_static: int = 8,
                   n_controls: int = 2, skip: bool = True, tram: bool = True, noise: bool = True,
                   xtram: bool = False, itram_size: int = 64, xtram_size: int = 128, safe: bool = True,
                   ops: list | None = None, read_offsets: bool = False, wild_tables: bool = False) -> str:
    """Emit a random `.da` program with `n_instr` instructions + END.

    safe=True keeps the program inside the reference's DEFINED behaviour (SURVEY.md §8a UB ledger):
    LOG/EXP see |A|<=1 and a literal selector 0..31, wrap-family operands are bounded, TRAM reads
    use offset 0 (unless read_offsets), SKIP can never reach END, values cannot blow up to inf/NaN.
    safe=False adds `ccr` operands and unbounded operands for the wrap family (still defined in the
    reference); wild_tables=True also lets LOG/EXP see out-of-range input (defined only by rule U6).
    """
    lines = []
    narrow = []                     # registers guaranteed in [-1, 1]
    wide = []                       # registers that may leave [-1, 1] (bounded)
    for i in range(n_static):
        v = rng.random()
        if rng.random() < 0.5:
            lines.append(f"static s{i} = {v:.6f}")
        else:
            lines.append(f"static s{i}")
        narrow.append(f"s{i}")
    for i in range(max(2, n_static // 3)):
        lines.append(f"static w{i}")
        wide.append(f"w{i}")
    ins = []
    for c in range(channels):
        lines.append(f"input in{c} {c}")
        ins.append(f"in{c}")
    outs = []
    for c in range(channels):
        lines.append(f"output out{c} {c}")
        outs.append(f"out{c}")
    ctl = []
    for i in range(n_controls):
        lines.append(f"control c{i} = {rng.random():.4f}")
        ctl.append(f"c{i}")
    if noise:
        lines.append("static noise")
    if tram:
        lines.append(f"itramsize {itram_size} ")
        lines.append("static trd")
    if xtram:
        lines.append(f"xtramsize {xtram_size} ")
        lines.append("static xrd")

    pool_ops = list(ops) if ops else (SAT_OPS * 3 + WRAP_OPS + WIDE_OPS + TABLE_OPS * 2)
    if skip and not ops:
        pool_ops += ["skip"] * 2
    if tram and not ops:
        pool_ops += ["idelay"] * 3
    if xtram and not ops:
        pool_ops += ["xdelay"] * 3

    def src_narrow():
        k = rng.random()
        if k < 0.40: return str(rng.choice(narrow))
        if k < 0.60: return str(rng.choice(ins))
        if k < 0.72 and ctl: return str(rng.choice(ctl))
        if k < 0.80 and noise: return "noise"
        if k < 0.86 and tram: return "trd"
        if k < 0.90: return str(rng.choice(outs))
        return str(rng.choice(LITERALS))

    def src_any():
        if not safe and rng.random() < 0.1: return "ccr"
        if rng.random() < 0.25: return str(rng.choice(wide))
        return src_narrow()

    def dst_narrow():
        return str(rng.choice(outs)) if rng.random() < 0.2 else str(rng.choice(narrow))

    body = []
    for k in range(n_instr):
        op = str(rng.choice(pool_ops))
        remaining = n_instr - 1 - k          # instructions after this one, before END
        if op in SAT_OPS:
            body.append(f"{op} {dst_narrow()}, {src_any()}, {src_any()}, {src_any()}")
        elif op in WRAP_OPS:
            s = src_narrow if safe else src_any
            body.append(f"{op} {rng.choice(wide)}, {s()}, {s()}, {s()}")
        elif op in TABLE_OPS:
            a = src_any() if wild_tables else src_narrow()     # |A| > 1 is undefined in the reference (U6)
            sel = int(rng.integers(0, 32))
            body.append(f"{op} {dst_narrow()}, {a}, {sel}, {rng.choice(['0', '1'])}")
        elif op == "andxor":
            pick = lambda: str(rng.choice(INT_LITERALS)) if rng.random() < 0.6 else src_any()
            body.append(f"andxor {rng.choice(wide)}, {pick()}, {pick()}, {pick()}")
        elif op in ("tstneg", "limit", "limitn", "macmv"):
            body.append(f"{op} {rng.choice(wide)}, {src_any()}, {src_any()}, {src_any()}")
        elif op == "skip":
            kmax = min(3, remaining)      # never reaches END: a reference object would spin forever
            body.append(f"skip ccr, ccr, {rng.choice(CCR_VALUES)}, {int(rng.integers(0, kmax + 1))}")
        elif op in ("idelay", "xdelay"):
            rd = "trd" if op == "idelay" else "xrd"
            size = itram_size if op == "idelay" else xtram_size
            if rng.random() < 0.5:
                off = int(rng.integers(0, size)) if read_offsets and rng.random() < 0.5 else 0
                body.append(f"{op} read, {rd}, at, {off}")
            else:
                off = int(rng.integers(0, min(size, 8))) if rng.random() < 0.3 else 0
                body.append(f"{op} write, {src_narrow()}, at, {off}")
    # make sure every output is driven by something saturating at the end
    for c, o in enumerate(outs):
        body.append(f"macs {o}, 0, {rng.choice(narrow)}, 1.0")
    return "\n".join(lines + body + ["end"])


def cfg5_allops(n_instr: int = 511, seed: int = SEED) -> str:
    """config 5: max-length synthetic program mixing all 16 hardware opcodes round-robin, every 16th
    instruction a data-dependent SKIP that can never reach END (SURVEY.md §8(d) config 5)."""
    rng = np.random.default_rng(seed)
    lines = [f"static r{i} = {rng.random():.6f}" for i in range(32)]
    lines += [f"static w{i}" for i in range(4)]
    lines += ["input in_l 0", "output out_l 0"]
    lines += [f"control k{i} = {rng.random():.4f}" for i in range(4)]
    narrow = [f"r{i}" for i in range(32)]
    wide = [f"w{i}" for i in range(4)]
    lits = ["0", "1.0", "0.5", "-0.5", "0.25", "0.75", "-0.25", "0.125"]

    def sn():
        k = rng.random()
        if k < 0.6: return str(rng.choice(narrow))
        if k < 0.75: return "in_l"
        if k < 0.88: return f"k{int(rng.integers(0, 4))}"
        return str(rng.choice(lits))

    def sa():
        return str(rng.choice(wide)) if rng.random() < 0.2 else sn()

    order = ["macs", "macsn", "macw", "macwn", "macints", "macintw", "acc3", "macmv", "andxor", "tstneg",
             "limit", "limitn", "log", "exp", "interp", "skip"]
    body = []
    n_body = n_instr - 1                      # the last real instruction drives the output
    for k in range(n_body):
        op = order[k % 16]
        if op in ("macs", "macsn", "macints", "acc3", "interp"):
            body.append(f"{op} {rng.choice(narrow)}, {sa()}, {sa()}, {sa()}")
        elif op in ("macw", "macwn", "macintw"):
            body.append(f"{op} {rng.choice(wide)}, {sn()}, {sn()}, {sn()}")
        elif op in ("log", "exp"):
            body.append(f"{op} {rng.choice(narrow)}, {sn()}, {int(rng.integers(1, 32))}, 0")
        elif op == "andxor":
            body.append(f"andxor {rng.choice(wide)}, {sa()}, {rng.choice(['1', '3', '-1', '16777215'])}, {rng.choice(['0', '1', '-4'])}")
        elif op in ("tstneg", "limit", "limitn", "macmv"):
            body.append(f"{op} {rng.choice(wide)}, {sa()}, {sa()}, {sa()}")
        else:
            kmax = min(3, n_body - 1 - k)
            body.append(f"skip ccr, ccr, {rng.choice([2, 6, 8, 16, 20])}, {int(rng.integers(1, 4)) if kmax >= 3 else kmax}")
    body.append("macs out_l, 0, r0, 1.0")
    return "\n".join(lines + body + ["end"])


def opcode_histogram(text: str) -> dict:
    h = {}
    for line in text.splitlines():
        w = line.strip().split()
        if w and w[0] in ("macs", "macsn", "macw", "macwn", "macints", "macintw", "acc3", "macmv", "andxor",
                          "tstneg", "limit", "limitn", "log", "exp", "interp", "skip", "idelay", "xdelay", "end"):
            h[w[0]] = h.get(w[0], 0) + 1
    return h


# ---- front-end corpus: valid, odd and malformed sources ---------------------------------------------

FRONTEND_CASES = {
    "decl_forms": "static a\nstatic b = 0.5\nstatic c=0.25\nstatic d, 0.75\nstatic e 1\ntemp t\nconst k = 2\ncontrol v = 0.1\ninput i0 0\noutput o0 0\nmacs o0, a, b, c\nend",
    "decl_backtrack_name": "static a1.5\nstatic b12\nstatic 7\noutput o 0\nmacs o, a, b12, 7\nend",
    "decl_negative_value": "static x = -0.5\nend",
    "decl_two_per_line": "static a,b\nend",
    "decl_duplicate": "static a\ncontrol a = 1\nstatic ccr\nend",
    "decl_bad_number": "static a 0.\nstatic b .5\nstatic c 1.2.3\nend",
    "io_out_of_range": "input in_r 1\noutput out_r 2\nend",
    "io_fraction_index": "input in_l 0.9\noutput out_l 0\nmacs out_l, 0, in_l, 1\nend",
    "uppercase": "STATIC A\nINPUT IN_L 0\nOUTPUT OUT_L 0\nMACS OUT_L, 0, IN_L, 0.5\nEND",
    "comments_and_blanks": "; header\n\nstatic a ; trailing\n   \noutput o 0\nmacs o, 0, a, 1 ; c\n;\nend",
    "tram_ok": "itramsize 100 \nxtramsize 48000 \nstatic rd\nidelay read, rd, at, 0\nidelay write, rd, at, 0\nend",
    "tram_no_trailing_blank": "itramsize 100\nend",
    "tram_two_blanks": "itramsize 100  \nend",
    "tram_tab": "itramsize 64\t\nend",
    "tram_oversize_then_second": "itramsize 65536 \nitramsize 10 \nend",
    "tram_x_oversize": "xtramsize 2000000 \nxtramsize 5 \nend",
    "instr_undeclared": "output o 0\nmacs o, 0, nope, 1\nend",
    "instr_partial_literals": "output o 0\nmacs 0.5, 0.25, nope, 1\nmacs o, 0.5, 0.25, 1\nend",
    "instr_input_as_r": "input i 0\nmacs i, 0, 0, 0\nend",
    "instr_spacing": "output o 0\nmacs   o ,0,  0.5 ,   -0.5   \nmacs\to,\t1,\t1,\t1\nend",
    "instr_missing_operand": "output o 0\nmacs o, 0, 1\nmacs o, 0, 1, 1, 1\nmacs o 0 1 1\nend",
    "instr_unknown_op": "output o 0\nmacx o, 0, 1, 1\nmacs, o, 0, 1, 1\nend",
    "instr_number_forms": "output o 0\nmacs o, 1e5, 0, 0\nmacs o, 5., 0, 0\nmacs o, --1, 0, 0\nmacs o, -, 0, 0\nmacs o, -3, 0.50, 00.5\nend",
    "noise_and_flags": "static noise\ninput i 0\noutput o 0\nmacs o, noise, i, noise\nmacs o, i, noise, 0\nend",
    "metadata": 'name "Test Prog"\ncopyright "2023, x"\ncreated "2023/08/01"\nengine "e"\ncomment "c c"\nguid "0-0"\nname "second"\nend',
    "metadata_bad": 'name "x" \nname ""\nname x\ncomment "a;b"\nend',
    "end_trailing_blank": "static a\nend ",
    "end_leading_blank": "static a\n end",
    "end_missing": "static a\nmacs a, 0, 0, 0",
    "end_crlf": "static a\r\nend\r\n",
    "end_twice": "static a\nend\nmacs a, 0, 0, 0\nend",
    "end_blank_after": "static a\nend\n\n",
    "no_final_newline": "static a\nend",
    "keywords_as_names": "static end\nstatic macs\noutput o 0\nmacs o, end, macs, 0\nend",
    "special_registers": "output o 0\nmacs o, ccr, read, write\nmacs ccr, at, 0, 0\nend",
    "literal_spellings": "output o 0\nmacs o, 0, 0.0, 1\nmacs o, 1.0, 1, 0.00\nend",
    "garbage": "hello world\n= 5\nstatic\ncontrol\nmacs\n,,,\nend",
}

_FUZZ_ATOMS = ["static", "temp", "control", "input", "output", "const", "itramsize", "xtramsize", "macs", "macsn", "skip",
               "log", "idelay", "end", "name", "comment", "a", "b", "in_l", "out_l", "ccr", "read", "write", "at", "noise",
               "0", "1", "0.5", "-0.5", "12", "1.", ".5", "1.2.3", "-", "=", ",", " ", "  ", "\t", "\"", "x y", ".", "_"]


def fuzz_source(rng: np.random.Generator) -> str:
    """A small random source: mostly valid lines with random token-level damage (never the two
    inputs that abort the reference: an empty number after itramsize/xtramsize, 10+ digit numbers)."""
    head = ["static a", "static b = 0.5", "input in_l 0", "output out_l 0", "control c = 0.25", "itramsize 64 "]
    body = ["macs out_l, 0, in_l, c", "macsn a, b, 0.5, -0.5", "log a, in_l, 3, 0", "skip ccr, ccr, 2, 1",
            "idelay write, a, at, 0", "idelay read, b, at, 0", "name \"n\""]
    lines = list(head) + [str(rng.choice(body)) for _ in range(int(rng.integers(1, 5)))]
    for _ in range(int(rng.integers(1, 4))):
        k = int(rng.integers(0, len(lines)))
        toks = lines[k].replace(",", " , ").split(" ")
        op = rng.random()
        j = int(rng.integers(0, len(toks)))
        if op < 0.35:
            toks[j] = str(rng.choice(_FUZZ_ATOMS))
        elif op < 0.6:
            toks.insert(j, str(rng.choice(_FUZZ_ATOMS)))
        elif op < 0.8 and len(toks) > 1:
            del toks[j]
        else:
            toks[j] = toks[j].upper() + str(rng.choice(["", " ", "\t", ";x"]))
        lines[k] = " ".join(toks).replace(" , ", ", ")
    tail = str(rng.choice(["end", "end", "end", "end ", "END", "", "end\n"]))
    text = "\n".join(lines + [tail])
    import re
    if re.search(r"(?mi)^\s*[ix]tramsize\s\s+$", text) or re.search(r"\d{10,}", text) or re.search(r"(?mi)^\s*[ix]tramsize\s+;", text):
        return fuzz_source(rng)
    if not text.strip("\n"):
        return fuzz_source(rng)
    return text


def random_flow_program(rng: np.random.Generator, n_instr: int, *, channels: int = 1, tram: str = "", size: int = 200,
                        cross: bool = False) -> str:
    """A random SKIP-free program whose only loop-carried values are SELF recurrences (the data-flow class the
    instruction-major kernel takes): every operand is an input, a control / literal, a register defined earlier in the
    same sample period, or the instruction's own result register.  tram = "i" / "x" / "ix" adds one READ and one WRITE
    per TRAM at random places with literal offsets.  cross=True plants one value carried from a later instruction to an
    earlier one (such a program must NOT take that kernel).  All values stay inside the reference's defined behaviour."""
    lines, statics = [], [f"s{i}" for i in range(n_instr + 4)]
    for r in statics:
        lines.append(f"static {r} = {rng.random():.5f}" if rng.random() < 0.6 else f"static {r}")
    ins = [f"in{c}" for c in range(channels)]
    outs = [f"out{c}" for c in range(channels)]
    lines += [f"input {r} {c}" for c, r in enumerate(ins)] + [f"output {r} {c}" for c, r in enumerate(outs)]
    ctl = ["c0", "c1"]
    lines += [f"control {r} = {rng.random():.4f}" for r in ctl]
    rd = {}
    for t in tram:
        lines.append(f"{t}tramsize {size} ")
        lines.append(f"static rd{t}")
        rd[t] = f"rd{t}"
    free = list(statics)
    rng.shuffle(free)
    defined_narrow, defined_wide = [], []          # produced earlier in this period: in [-1, 1] / possibly wider
    body = []

    def lit():
        return f"{rng.choice([0.0, 0.125, 0.25, 0.5, 0.75, 1.0, -0.5, -0.25]):g}"

    def src(narrow_only, own=None):
        pool = list(ins) * 2 + ctl + [lit(), lit()] + defined_narrow * 2
        if not narrow_only:
            pool += defined_wide * 2
        if own is not None:
            pool += [own] * 3
        return str(rng.choice(pool))

    tram_ops = []
    for t in tram:
        d = "idelay" if t == "i" else "xdelay"
        roff, woff = int(rng.integers(0, size // 2)), int(rng.integers(0, 4))
        tram_ops += [("rd", t, f"{d} read, {rd[t]}, at, {roff}"), ("wr", t, d, woff)]
    slots = sorted(rng.choice(n_instr + 1, size=len(tram_ops), replace=True).tolist()) if tram_ops else []
    order = list(rng.permutation(len(tram_ops))) if tram_ops else []
    planted = None
    for i in range(n_instr + 1):
        for k, sl in enumerate(slots):
            if sl == i:
                op = tram_ops[order[k]]
                if op[0] == "rd":
                    body.append(op[2]); defined_narrow.append(rd[op[1]])
                else:
                    body.append(f"{op[2]} write, {src(True)}, at, {op[3]}")
        if i == n_instr:
            break
        last = (i >= n_instr - channels)
        r = outs[i - (n_instr - channels)] if last else free.pop()
        own = r if rng.random() < 0.45 else None       # self recurrence on this instruction's result register
        kind = rng.choice(["sat", "sat", "sat", "interp", "wrap", "limit", "tstneg", "table", "andxor"])
        if kind == "sat":
            body.append(f"{rng.choice(['macs', 'macsn', 'acc3', 'macints'])} {r}, {src(False, own)}, {src(True, own)}, {src(True, own)}")
            defined_narrow.append(r)
        elif kind == "interp":
            body.append(f"interp {r}, {src(True, own)}, {rng.choice(ctl + [lit()])}, {src(True)}")
            defined_narrow.append(r)
        elif kind == "wrap":
            body.append(f"{rng.choice(['macw', 'macwn', 'macintw'])} {r}, {src(True, own)}, {src(True)}, {src(True)}")
            defined_wide.append(r)
        elif kind == "limit":
            body.append(f"{rng.choice(['limit', 'limitn'])} {r}, {src(False, own)}, {src(True, own)}, {src(True)}")
            defined_narrow.append(r)
        elif kind == "tstneg":
            body.append(f"tstneg {r}, {src(False)}, {src(True, own)}, {src(True)}")
            defined_narrow.append(r)
        elif kind == "table":
            body.append(f"{rng.choice(['log', 'exp'])} {r}, {src(True, own)}, {int(rng.integers(0, 32))}, 0")
            defined_narrow.append(r)
        else:
            body.append(f"andxor {r}, {src(False)}, {src(True)}, {src(True)}")
            defined_wide.append(r)
        if cross and planted is None and i >= 1 and not last:
            planted = r
    if cross and planted is not None:
        # the first instruction now reads what a later one leaves behind: carried across instructions
        first = body[0].split(",")
        if not body[0].startswith(("idelay", "xdelay")):
            first[-1] = " " + planted
            body[0] = ",".join(first)
    return "\n".join(lines + body + ["end"])
