"""The translator's kernel cache on the GPU.  The cache counters are process-wide, so each case runs its handles in fresh worker processes
(tests/kernel_cache_common.py) and reads their JSON report.

- Warm start: a second process with the directory of a first one finds every kernel on disk and runs translated from its very first call,
  in mode 1, without libnvrtc (FX8010_NVRTC names a path that does not exist, so none is loaded): it looks its kernels up under the
  NVRTC version the files' headers record.
- A device-free precompile (with the toolkit's libnvrtc, not the one torch brings) serves a later process the same way.
- One compile per process: the 3-shard executor compiles a program no cache has seen exactly once, in mode 2 and in mode 1.
- A file whose payload is not a CUBIN is rejected at module load, recompiled and replaced; an unwritable directory fails no call.
Every output and final state is compared with the oracle bit for bit.
"""
import hashlib
import importlib
import json
import os
import struct
import subprocess
import sys
import time

import pytest

import kernel_cache_common as kc

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
fx = importlib.import_module("fx8010-emulator-core_b200")

HERE = os.path.dirname(os.path.abspath(__file__))
ALL = sorted(kc.programs())
CURVE_BIT = 16


def worker(args, **env):
    e = {k: v for k, v in os.environ.items() if k != "FX8010_KERNEL_CACHE"}
    e.update({k: str(v) for k, v in env.items()})
    r = subprocess.run([sys.executable, os.path.join(HERE, "kernel_cache_common.py"), json.dumps(args)], env=e, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def assert_translated_from_the_start(report):
    assert not report["nvrtc_available"], "the process was meant to run without libnvrtc"
    for name, p in report["programs"].items():
        bit = CURVE_BIT if p["curves"] else kc.VARIANT_TRANSLATED
        assert p["variant"] & bit and p["state"] == 2, f"{name}: the first call did not run translated: {p}"
        assert p["bit_exact"], f"{name}: outputs or state differ from the oracle"


def test_warm_start_without_nvrtc(tmp_path):
    d = tmp_path / "kcache"
    a = worker({"programs": ALL, "mode": 2}, FX8010_KERNEL_CACHE=d)
    assert all(p["bit_exact"] for p in a["programs"].values()), a
    assert a["stats"]["disk_writes"] == len(ALL) and a["stats"]["nvrtc_compiles"] == len(ALL), a["stats"]
    assert len(os.listdir(d / "fx8010-v1")) == len(ALL)
    b = worker({"programs": ALL, "mode": 1}, FX8010_KERNEL_CACHE=d, FX8010_NVRTC=tmp_path / "no" / "libnvrtc.so")
    assert_translated_from_the_start(b)
    assert b["stats"]["nvrtc_compiles"] == 0, b["stats"]
    assert b["stats"]["disk_hits"] == a["stats"]["disk_writes"], b["stats"]
    assert b["stats"]["disk_rejected"] == 0


def test_precompiled_without_a_device(tmp_path):
    d = tmp_path / "kcache"
    code = ("import importlib, json, sys; sys.path[:0] = [%r, %r]; import kernel_cache_common as kc; "
            "fx = importlib.import_module('fx8010-emulator-core_b200'); rc = {}\n"
            "for name, (text, n, s, cv) in kc.programs().items():\n"
            "    prog = fx.Program(text)\n"
            "    rc[name] = fx.precompile(prog, n, 1, [(prog.reg_index(r), b) for r, b in cv])\n"
            "print(json.dumps(rc))" % (HERE, os.path.dirname(HERE)))
    env = {k: v for k, v in os.environ.items() if k != "FX8010_KERNEL_CACHE"}
    env.update(FX8010_KERNEL_CACHE=str(d), CUDA_VISIBLE_DEVICES="")          # no device in the precompiling process
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    assert json.loads(r.stdout.strip().splitlines()[-1]) == {name: 0 for name in ALL}
    b = worker({"programs": ALL, "mode": 1}, FX8010_KERNEL_CACHE=d, FX8010_NVRTC=tmp_path / "no" / "libnvrtc.so")
    assert_translated_from_the_start(b)
    assert b["stats"]["nvrtc_compiles"] == 0 and b["stats"]["disk_hits"] == len(ALL), b["stats"]


@pytest.mark.parametrize("mode", [2, 1])
@pytest.mark.parametrize("devices", [[0, 0, 0], [0, 1, 0]], ids=["3_shards_1_gpu", "3_shards_2_gpus"])
def test_one_compile_per_process(devices, mode):
    if max(devices) >= torch.cuda.device_count():
        pytest.skip("needs two GPUs")
    rep = worker({"multi": devices, "mode": mode, "tag": time.time_ns() + mode})
    assert rep["multi"]["bit_exact"], rep
    assert rep["multi"]["ms_to_translated"] is not None, f"the shards never ran translated: {rep}"
    assert rep["stats"]["nvrtc_compiles"] == 1, rep["stats"]
    # the other two shards joined the compile, or found its CUBIN in the store or its module on the device
    st = rep["stats"]
    assert st["joined_compiles"] + st["store_hits"] + st["memory_hits"] == 2, st


def test_file_that_is_not_a_cubin_is_rejected_at_load(tmp_path):
    d = tmp_path / "kcache"
    a = worker({"programs": ["cfg2"], "mode": 2}, FX8010_KERNEL_CACHE=d)
    (name,) = os.listdir(d / "fx8010-v1")
    path = d / "fx8010-v1" / name
    good = path.read_bytes()
    payload = b"not a cubin, but a payload whose checksum is right " * 64
    hdr = bytearray(good[:96])
    struct.pack_into("<Q32s", hdr, 56, len(payload), hashlib.sha256(payload).digest())
    path.write_bytes(bytes(hdr) + payload)
    b = worker({"programs": ["cfg2"], "mode": 2}, FX8010_KERNEL_CACHE=d)
    p = b["programs"]["cfg2"]
    assert p["bit_exact"] and p["variant"] & kc.VARIANT_TRANSLATED and p["state"] == 2, p
    assert b["stats"]["disk_rejected"] == 1 and b["stats"]["disk_hits"] == 0 and b["stats"]["nvrtc_compiles"] == 1, b["stats"]
    assert b["stats"]["disk_writes"] == 1
    data = path.read_bytes()                                  # replaced by the compiled kernel: a valid file again
    assert data[:8] == good[:8] and data[96:100] == b"\x7fELF" and hashlib.sha256(data[96:]).digest() == data[64:96]
    assert a["stats"]["disk_writes"] == 1


def test_unwritable_directory_fails_no_call(tmp_path):
    blocker = tmp_path / "a_file"
    blocker.write_text("not a directory")
    rep = worker({"programs": ["cfg2", "cfg5_512"], "mode": 2}, FX8010_KERNEL_CACHE=blocker / "kcache")
    for name, p in rep["programs"].items():
        assert p["bit_exact"] and p["variant"] & kc.VARIANT_TRANSLATED and p["state"] == 2, (name, p)
    assert rep["stats"]["disk_write_failures"] >= 1 and rep["stats"]["disk_writes"] == 0, rep["stats"]
