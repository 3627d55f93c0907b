"""The host front-end (hand-written scanner, fx8010-emulator-core_b200/host/fx8010_frontend.cpp)
against the reference's loader: committed records of what the reference decoded / rejected for a
corpus of valid, odd and malformed sources (tests/golden/frontend.json) and, when the compiled
reference is around, a live differential fuzz."""
import json
import os

import numpy as np
import pytest

import progs

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frontend.json")


def record(fx, text, channels=1):
    p = fx.Program(text, channels=channels)
    return {"loaded": bool(p.loaded), "ready": bool(p.ready),
            "registers": [[int(t), int(np.float32(v).view(np.uint32)), int(io), n] for t, v, io, n in p.registers()],
            "instructions": [list(i) for i in p.instructions()],
            "errors": [[d, int(r)] for d, r in p.errors()],
            "controls": p.controls(), "metadata": p.metadata(), "itram": p.itram_size, "xtram": p.xtram_size}


def test_frontend_matches_reference_records(fx):
    gold = json.load(open(GOLD))
    assert len(gold) > 300
    checked = 0
    for name, g in gold.items():
        if g["text"] is None:
            continue
        r = record(fx, g["text"], g["channels"])
        for k in r:
            assert r[k] == g[k], f"{name}: {k} differs\n--- source ---\n{g['text']}\n--- ours ---\n{r[k]}\n--- reference ---\n{g[k]}"
        checked += 1
    assert checked > 300


def test_shipped_testcode_image(fx, tmp_path):
    """Decoded image of the reference's shipped testcode.da (SURVEY.md §8c): 14 registers, 2 instructions."""
    g = json.load(open(GOLD))["shipped_testcode_da"]
    names = [r[3] for r in g["registers"]]
    assert names == ["ccr", "read", "write", "at", "a", "in_l", "volume", "pan", "filter_cutoff", "out_l", "rd", "wr", "noise", "0"]
    assert g["instructions"] == [[0, 9, 13, 5, 6, 1, 1, 0], [18, 0, 0, 0, 0, 0, 0, 0]]
    assert (g["itram"], g["xtram"]) == (1000, 48000)
    # the same program without its comment lines decodes identically through our front-end
    r = record(fx, progs.CFG1A_TESTCODE)
    assert r["registers"] == g["registers"] and r["instructions"] == g["instructions"] and r["controls"] == g["controls"]
    # loaded from a file, with the shipped file's metadata lines (taken from the record) in front of the program:
    # every field of the record, metadata included.  The file's text is rebuilt from the record, so this checks that
    # `key "value"` lines decode to the recorded metadata, not the exact byte layout (comments) of the shipped file.
    meta = "".join(f'{k} "{v}"\n' for k, v in g["metadata"].items())
    path = tmp_path / "testcode.da"
    path.write_text(meta + progs.CFG1A_TESTCODE.split("\n", 2)[2])          # the program after its name and copyright lines
    p = fx.Program(path=str(path))
    assert p.loaded and [list(i) for i in p.instructions()] == g["instructions"]
    assert p.metadata() == g["metadata"]
    assert record(fx, path.read_text()) == {k: g[k] for k in r}


def test_frontend_live_fuzz_vs_reference(fx, po):
    if not po.have_reference():
        pytest.skip("oracle/_ref/libfx8010_ref.so not built (needs /root/reference)")
    rng = np.random.default_rng(20231018)
    for k in range(1500):
        text = progs.fuzz_source(rng)
        ref = po.Reference(text)
        ours = record(fx, text)
        theirs = {"loaded": bool(ref.loaded), "ready": bool(ref.ready),
                  "registers": [[int(t), int(np.float32(v).view(np.uint32)), int(io), n] for t, v, io, n in ref.registers()],
                  "instructions": [list(i) for i in ref.instructions()], "errors": [[d, int(r)] for d, r in ref.errors()],
                  "controls": ref.controls(), "metadata": ref.metadata(),
                  "itram": int(ref.L.ref_itram_size(ref.h)), "xtram": int(ref.L.ref_xtram_size(ref.h))}
        assert ours == theirs, f"fuzz {k}:\n{text!r}\nours   {ours}\ntheirs {theirs}"


def test_second_load_appends_and_rows_continue(fx, po):
    """loadFile twice: registers/instructions append, diagnostic rows keep counting (reference
    errorCounter is never reset, include/FX8010.h:273)."""
    p = fx.Program("static a\nend")
    assert p.loaded
    assert not p.load("static a\nbogus\nend")
    errs = p.errors()
    assert errs[0] == ("Kein Fehler", 1)
    assert ("Mehrfache Variablendeklaration", 3) in errs and ("Ungueltige Syntax", 4) in errs
    assert len(p.instructions()) == 2
    if po.have_reference():
        r = po.Reference("static a\nend")
        r.load("static a\nbogus\nend")
        assert r.errors() == errs


def test_facade_register_api_without_gpu(fx):
    """setRegisterValue / getRegisterValue conventions on the host mirror (source/FX8010.cpp:236-266)."""
    p = fx.Program(progs.CFG1A_TESTCODE)
    assert p.get_register("volume") == 1.0
    assert p.set_register("volume", 0.25) == 0 and p.get_register("volume") == 0.25
    assert p.set_register("0", 3.0) == 0 and p.get_register("0") == 3.0          # literals are registers too
    assert p.set_register("nope", 1.0) == 1 and p.get_register("nope") == 1.0    # "not found" returns 1
    assert p.controls() == ["volume", "pan", "filter_cutoff"]
    assert p.metadata()["name"] == "testcode"
    assert p.instruction_counter == 0


def test_relaxed_mode_accepts_the_readme_forms(fx):
    """Strict mode = the reference (README example is rejected, SURVEY.md §0 F6); relaxed mode loads it and
    decodes it like the strictly spelled source."""
    readme = "static a\r\nitramsize 100\r\ninput in_l 0\r\noutput out_l 0\r\nlog a, in_l, 3, 0\r\nmacs out_l, 0, a, 1.0\r\n  END  \r\n\r\n\r\n"
    strict_src = "static a\nitramsize 100 \ninput in_l 0\noutput out_l 0\nlog a, in_l, 3, 0\nmacs out_l, 0, a, 1.0\nend"
    assert not fx.Program(readme).loaded
    r, s = fx.Program(readme, relaxed=True), fx.Program(strict_src)
    assert r.loaded and s.loaded, r.errors()
    assert r.registers() == s.registers() and r.instructions() == s.instructions() and r.itram_size == s.itram_size == 100
    assert fx.Program("static a\nitramsize 64   \nend", relaxed=True).loaded
    assert not fx.Program("static a\nbogus line\nend\n\n", relaxed=True).loaded          # still an error, just not about END
