"""Operand edge values shared by tests/test_operand_edges_translate.py (CPU) and tests/test_gpu_operand_edges.py (B200).

DESIGN.md §2 keeps the 0 ULP promise on the device with four rules: no flush-to-zero, saturation that lets NaN through, signed zeros
preserved, and x86 `cvttss2si` semantics for every float -> int32 cast.  The values below are where those rules decide the result:
signed zeros, subnormals, the neighbours of +-1 and +-2, the CCR codes and table selectors, the ANDXOR 0xFFFFFF rules, the int32
conversion limits, the largest finite values, the infinities and one NaN.

NaN is compared as a class (DESIGN.md ledger U11): where the oracle holds a NaN the device must hold a NaN, whatever its pattern,
because x86 and the GPU produce and propagate different NaN bit patterns.  Everything else is compared bit for bit.
"""
import numpy as np

from conftest import assert_bits_equal

EDGE_BITS = [
    0x00000000, 0x80000000,                                  # +-0
    0x00000001, 0x80000001, 0x007fffff, 0x00800000,          # +-min subnormal, max subnormal, min normal
    0x3f7fffff, 0xbf7fffff, 0x3f800000, 0xbf800000,          # +-(1 - ulp), +-1
    0x3f800001, 0xbf800001, 0x40000000, 0xc0000000,          # +-(1 + ulp), +-2
    0x3f000000, 0x41a00000, 0x41f80000, 0x41ffffff, 0x42000000,   # 0.5, 20 (CCR codes), 31, 31.999998, 32 (table selectors)
    0x4b7fffff, 0x4b800000,                                  # 16777215, 16777216 (ANDXOR's 0xFFFFFF rules)
    0x4effffff, 0x4f000000, 0xcf000000, 0xcf000001,          # 2147483520, 2^31, -2^31, -2^31 - 256 (cvt_x86 limits)
    0x7f7fffff, 0xff7fffff, 0x7f800000, 0xff800000,          # +-FLT_MAX, +-inf
    0x7fffffff,                                              # the one NaN both sides propagate alike (progs.TABLE_EDGE_BITS)
]
EDGE = np.array(EDGE_BITS, dtype=np.uint32).view(np.float32)
E = len(EDGE)                                                # 30: 30^3 = 27 000 instances, a multiple of 4 and 8

# A decimal spelling the front-end (`-?\d+(\.\d+)?` through strtof) reads as exactly these bits; every edge value but the NaN.
LITERAL_SPELLING = {
    0x00000000: "0", 0x80000000: "-0",
    0x00000001: "0." + "0" * 44 + "14", 0x80000001: "-0." + "0" * 44 + "14",
    0x007fffff: "0." + "0" * 37 + "11754942", 0x00800000: "0." + "0" * 37 + "11754944",
    0x3f7fffff: "0.99999994", 0xbf7fffff: "-0.99999994", 0x3f800000: "1", 0xbf800000: "-1",
    0x3f800001: "1.00000012", 0xbf800001: "-1.00000012", 0x40000000: "2", 0xc0000000: "-2",
    0x3f000000: "0.5", 0x41a00000: "20", 0x41f80000: "31", 0x41ffffff: "31.999998", 0x42000000: "32",
    0x4b7fffff: "16777215", 0x4b800000: "16777216",
    0x4effffff: "2147483520", 0x4f000000: "2147483648", 0xcf000000: "-2147483648", 0xcf000001: "-2147483904",
    0x7f7fffff: "340282346638528859811704183484516925440", 0xff7fffff: "-340282346638528859811704183484516925440",
    0x7f800000: "9" * 40, 0xff800000: "-" + "9" * 40,
}

# Every arithmetic opcode, LOG / EXP with the selector in X.
OPS = ["macs", "macsn", "macints", "acc3", "macw", "macwn", "macintw", "andxor", "tstneg", "limit", "limitn", "interp", "log", "exp"]


def grid():
    """Per-instance A, X and Y: the cross product of the edge values, A slowest."""
    a, x, y = np.meshgrid(EDGE, EDGE, EDGE, indexing="ij")
    return a.ravel().copy(), x.ravel().copy(), y.ravel().copy()


def periodic_input(channels, s, n, start=0):
    """[C][S][N]: instance i reads EDGE[(i + 7 t) % 30] at period t (every channel alike), so rows change from period to period."""
    i = np.arange(n)[None, :]
    t = np.arange(start, start + s)[:, None]
    row = EDGE[(i + 7 * t) % E]
    return np.ascontiguousarray(np.broadcast_to(row, (channels, s, n))).astype(np.float32)


def _float_bits(a):
    return a.view(np.uint32 if a.dtype.itemsize == 4 else np.uint64)


def assert_edge_equal(got, want, what=""):
    """Floats: bit-equal wherever `want` is not NaN, NaN wherever it is.  Anything else: bit-equal."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    if got.dtype.kind != "f":
        assert_bits_equal(got, want, what)
        return
    assert got.dtype == want.dtype, f"{what}: dtype {got.dtype} vs {want.dtype}"
    nan_w = np.isnan(want)
    bad = (_float_bits(got) != _float_bits(want)) & ~nan_w
    bad |= nan_w & ~np.isnan(got)
    if bad.any():
        idx = np.argwhere(bad)
        f = tuple(idx[0])
        raise AssertionError(f"{what}: {len(idx)} of {got.size} elements differ; first at {f}: {got[f]!r} (0x{int(_float_bits(got)[f]):x}) "
                             f"vs {want[f]!r} (0x{int(_float_bits(want)[f]):x})")


def nan_patterns(a):
    """The set of bit patterns of the NaNs in a float32 array."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    return {int(v) for v in np.unique(a.view(np.uint32)[np.isnan(a)])}


def assert_device_nan(got, want, what=""):
    """The NaN patterns ledger U11 allows on the device: 0x7FFFFFFF (what the FP32 pipe produces and every path propagates), and
    0xFFC00000 where the NaN was born in the FP64 pipe (an invalid operation of LOG / EXP's interpolation, e.g. EXP(+inf): a flat table
    row's zero slope times an infinite distance), whose default NaN 0xFFF8000000000000 narrows to it.  x86 produces that same pattern
    for every invalid operation, so a device 0xFFC00000 must sit where the oracle holds 0xFFC00000 too."""
    got, want = np.ascontiguousarray(got, dtype=np.float32), np.ascontiguousarray(want, dtype=np.float32)
    pats = nan_patterns(got)
    assert pats <= {0x7fffffff, 0xffc00000}, f"{what}: NaN patterns {sorted(hex(p) for p in pats)}"
    odd = got.view(np.uint32) == 0xffc00000
    assert (want.view(np.uint32)[odd] == 0xffc00000).all(), f"{what}: 0xffc00000 where the oracle holds no invalid-operation NaN"


def compare_state_edges(gpu, orc, what, tram_instances=(0,)):
    """test_gpu_parity.compare_state with NaN compared as a class: registers, accumulator, LFSR, latches, TRAM pointers and contents,
    instruction counters and runtime flags."""
    assert_edge_equal(gpu.registers(), orc.registers, what + " registers")
    acc, lfsr, latch, ptrs = gpu.scalars()
    assert_edge_equal(acc, orc.acc, what + " accumulator")
    assert_bits_equal(lfsr, orc.lfsr, what + " lfsr")
    assert_edge_equal(latch, orc.out_latch, what + " out latch")
    assert_bits_equal(ptrs, orc.tram_ptrs, what + " tram pointers")
    assert_bits_equal(gpu.counts(), orc.counts, what + " instruction counters")
    d = gpu.dims()
    for which, size in ((0, d.itram_size), (1, d.xtram_size)):
        if size:
            for i in tram_instances:
                assert_edge_equal(gpu.tram(which, i), orc.tram(which, i), f"{what} tram{which}[{i}]")
    assert gpu.flags() == orc.flags, f"{what} runtime flags {gpu.flags():#x} vs {orc.flags:#x}"


# ---- programs ------------------------------------------------------------------------------------------------------------------

# Consumers of the hot programs' producer/consumer pairs: the forwarded value in A, X or Y, MACS or MACSN, the other operands literals.
_PAIR_CONSUMERS = ["macsn {o}, {t}, 0, 0", "macs {o}, 0, {t}, 1", "macsn {o}, 0, 1, {t}", "macs {o}, -1, 1, {t}"]


def op_program(ops=OPS, ccr=False, extra_head=(), extra_body=(), lead_body=()):
    """Each op once as `op o, ca, cx, cy` and once with A from the input, every result of every period in an output channel.

    ccr=False ("hot"): nobody reads `ccr`; the input form's result goes through a producer/consumer pair (a MACS / MACSN with literal
    other operands), the pattern the instruction-major kernel fuses.  ccr=True: `limit q, 1, ccr, ccr` (q = ccr) after the first form,
    into an output of its own, so that CCR is materialised per period and reaches the outputs.  Returns (text, channels)."""
    head = ["control ca = 0", "control cx = 0", "control cy = 0", "input in_l 0"] + list(extra_head)
    body = list(lead_body)
    ch = 0
    for k, op in enumerate(ops):
        o1 = f"o{ch}"; ch += 1
        body.append(f"{op} {o1}, ca, cx, cy")
        if ccr:
            oc, o2 = f"o{ch}", f"o{ch + 1}"; ch += 2
            body += [f"limit {oc}, 1, ccr, ccr", f"{op} {o2}, in_l, cx, cy"]
        else:
            o2 = f"o{ch}"; ch += 1
            head.append(f"static t{k}")
            body += [f"{op} t{k}, in_l, cx, cy", _PAIR_CONSUMERS[k % len(_PAIR_CONSUMERS)].format(o=o2, t=f"t{k}")]
    head += [f"output o{c} {c}" for c in range(ch)]
    return "\n".join(head + body + list(extra_body) + ["end"]), ch


def folded_program(ops, pos, spellings=None):
    """Each op with one operand a literal at every spelling (position `pos`: 0 = A, 1 = X, 2 = Y), the other two the controls ca, cx.
    Results go to static registers r<k> (compared in the final state); one output passes the input through."""
    spellings = list(LITERAL_SPELLING.values()) if spellings is None else spellings
    head = ["control ca = 0", "control cx = 0", "input in_l 0", "output out_l 0"]
    body = []
    k = 0
    for op in ops:
        for lit in spellings:
            opr = ["ca", "cx"]
            opr.insert(pos, lit)
            head.append(f"static r{k}")
            body.append(f"{op} r{k}, {opr[0]}, {opr[1]}, {opr[2]}")
            k += 1
    body.append("macs out_l, in_l, ca, cx")
    return "\n".join(head + body + ["end"])


def all_literal_program(rng, count=100):
    """About `count` instructions whose three operands are all literals at edge spellings (every op in turn)."""
    sp = list(LITERAL_SPELLING.values())
    head, body = ["input in_l 0", "output out_l 0"], []
    for k in range(count):
        op = OPS[k % len(OPS)]
        a, x, y = (sp[int(j)] for j in rng.integers(0, len(sp), 3))
        head.append(f"static r{k}")
        body.append(f"{op} r{k}, {a}, {x}, {y}")
    # ANDXOR where two of its rules hold at once: Y == 0xFFFFFF and Y == ~X (X = -16777216), X == 0xFFFFFF and Y == ~X
    for j, a in enumerate(sp):
        x, y = ("-16777216", "16777215") if j % 2 else ("16777215", "-16777216")
        head.append(f"static r{count + j}")
        body.append(f"andxor r{count + j}, {a}, {x}, {y}")
    body.append("macs out_l, in_l, 0, 0")
    return "\n".join(head + body + ["end"])
