"""The translator's kernel cache on the CPU (no GPU needed; NVRTC compiles for sm_100a without a device).

fx8010_kernel_cache_precompile writes the kernel a handle would compile into the disk store: one file per kernel, named by the SHA-256
of the key bytes documented in include/fx8010_gpu.h (rebuilt here from fx8010_translate_source and nvrtcVersion), holding a 96-byte
header and the CUBIN.  Checked: the name and the header, a second precompile reusing the file without compiling, eight processes
writing one file at once, damaged files rejected and rewritten, an unwritable directory, and no file anywhere when the store is off.
"""
import ctypes as C
import hashlib
import importlib
import os
import struct
import subprocess
import sys

import pytest

import progs

fx = importlib.import_module("fx8010-emulator-core_b200")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVRTC_OPTIONS = ["--gpu-architecture=sm_100a", "--std=c++17", "--fmad=false", "--ftz=false", "--prec-div=true", "--prec-sqrt=true",
                 "-lineinfo", "-default-device"]
HEADER = struct.Struct("<8sIiiI32sQ32s")          # magic, format, NVRTC major, minor, reserved, digest, payload bytes, payload SHA-256
N = 4096


def nvrtc_version():
    for name in (os.environ.get("FX8010_NVRTC"), "libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so",
                 "/usr/local/cuda/lib64/libnvrtc.so"):
        if not name:
            continue
        try:
            lib = C.CDLL(name)
        except OSError:
            continue
        major, minor = C.c_int(), C.c_int()
        assert lib.nvrtcVersion(C.byref(major), C.byref(minor)) == 0
        return major.value, minor.value
    return None


@pytest.fixture(scope="module")
def version():
    v = nvrtc_version()
    if v is None:
        pytest.skip("libnvrtc not loadable here")
    return v


@pytest.fixture
def cache(tmp_path):
    """A fresh directory set as the process's disk store; the store is turned off again afterwards."""
    d = tmp_path / "kcache"
    fx.set_kernel_cache_dir(str(d))
    yield d
    fx.set_kernel_cache_dir(None)


@pytest.fixture(scope="module")
def cfg2():
    prog = fx.Program(progs.CFG2_LOG_GAIN)
    assert prog.loaded, prog.errors()
    yield prog
    prog.close()


def key_bytes(src: str, version) -> bytes:
    head = "fx8010-kernel-v1\nsm_100a\n" + "".join(o + "\n" for o in NVRTC_OPTIONS) + "nvrtc %d.%d\n" % version
    return head.encode() + src.encode()


def files(d):
    sub = d / "fx8010-v1"
    return sorted(os.listdir(sub)) if sub.exists() else []


def check_file(path, digest_hex, version):
    data = path.read_bytes()
    magic, fmt, major, minor, _, digest, n, payload_sha = HEADER.unpack_from(data)
    assert magic == b"FX8010KC" and fmt == 1 and (version is None or (major, minor) == version)
    assert digest.hex() == digest_hex
    assert n == len(data) - HEADER.size > 1000
    assert hashlib.sha256(data[HEADER.size:]).digest() == payload_sha
    assert data[HEADER.size:HEADER.size + 4] == b"\x7fELF"


def test_stats_struct_layout():
    assert C.sizeof(fx.CKernelCacheStats) == 64
    assert set(fx.kernel_cache_stats()) == {"nvrtc_compiles", "memory_hits", "store_hits", "joined_compiles", "disk_hits", "disk_writes",
                                            "disk_rejected", "disk_write_failures"}


def test_precompile_names_the_file_by_the_documented_key(cache, cfg2, version):
    src, _ = fx.translate_source(cfg2, 1, instances=N)
    digest = hashlib.sha256(key_bytes(src, version)).hexdigest()
    before = fx.kernel_cache_stats()
    assert fx.precompile(cfg2, N) == 0
    assert files(cache) == [digest + ".cubin"]
    check_file(cache / "fx8010-v1" / (digest + ".cubin"), digest, version)
    after = fx.kernel_cache_stats()
    assert after["nvrtc_compiles"] == before["nvrtc_compiles"] + 1
    assert after["disk_writes"] == before["disk_writes"] + 1
    # the second time the file is there: nothing is compiled
    assert fx.precompile(cfg2, N) == 1
    assert fx.kernel_cache_stats()["nvrtc_compiles"] == after["nvrtc_compiles"]
    assert files(cache) == [digest + ".cubin"]


def test_curve_translation_is_a_kernel_of_its_own(cache, version):
    prog = fx.Program(progs.CFG4_ONEPOLE)
    curves = [(prog.reg_index("filter_cutoff"), False)]
    assert fx.precompile(prog, N, curves=curves) == 0
    src, _ = fx.translate_source_curves(prog, curves, 1, instances=N)
    assert files(cache) == [hashlib.sha256(key_bytes(src, version)).hexdigest() + ".cubin"]
    prog.close()


def test_bad_arguments(cache, cfg2):
    assert fx.precompile(cfg2, 0) == -1
    assert fx.precompile(cfg2, N, channels=0) == -1
    assert fx.precompile(cfg2, N, curves=[(0, False)]) == -1          # register 0 (ccr) is not CONTROL or STATIC
    assert files(cache) == []


PRECOMPILE = """
import importlib, sys
sys.path[:0] = [{root!r}, {tests!r}]
import progs
fx = importlib.import_module("fx8010-emulator-core_b200")
print(fx.precompile(fx.Program(progs.CFG2_LOG_GAIN), {n}))
"""


def run_precompile(env, n=N):
    code = PRECOMPILE.format(root=ROOT, tests=os.path.join(ROOT, "tests"), n=n)
    return subprocess.Popen([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)


def test_eight_processes_leave_one_valid_file(tmp_path, cfg2, version):
    d = tmp_path / "shared"
    env = dict(os.environ, FX8010_KERNEL_CACHE=str(d))
    procs = [run_precompile(env) for _ in range(8)]
    codes = []
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err
        codes.append(int(out.strip().splitlines()[-1]))
    assert set(codes) <= {0, 1} and 0 in codes, codes
    # (the workers load libnvrtc themselves: it may be another version than this process's, hence no digest from here)
    names = files(d)
    assert len(names) == 1 and names[0].endswith(".cubin"), f"a temporary file was left behind, or another file appeared: {names}"
    check_file(d / "fx8010-v1" / names[0], names[0][:-len(".cubin")], None)


def _truncate(data):
    return data[: len(data) // 2]


def _flip_payload_byte(data):
    b = bytearray(data)
    b[HEADER.size + len(b[HEADER.size:]) // 2] ^= 0x40
    return bytes(b)


def _wrong_magic(data):
    return b"FX8010KX" + data[8:]


@pytest.mark.parametrize("damage", [_truncate, _flip_payload_byte, _wrong_magic], ids=["truncated", "flipped_payload_byte", "wrong_magic"])
def test_damaged_file_is_rejected_and_rewritten(cache, cfg2, version, damage):
    assert fx.precompile(cfg2, N) == 0
    (name,) = files(cache)
    path = cache / "fx8010-v1" / name
    path.write_bytes(damage(path.read_bytes()))
    before = fx.kernel_cache_stats()
    assert fx.precompile(cfg2, N) == 0
    after = fx.kernel_cache_stats()
    assert after["disk_rejected"] == before["disk_rejected"] + 1
    assert after["nvrtc_compiles"] == before["nvrtc_compiles"] + 1
    assert files(cache) == [name]
    check_file(path, name[:-len(".cubin")], version)
    assert fx.precompile(cfg2, N) == 1


def test_unwritable_directory(tmp_path, cfg2, version):
    blocker = tmp_path / "a_file"
    blocker.write_text("not a directory")
    fx.set_kernel_cache_dir(str(blocker / "kcache"))          # below a regular file: no mkdir can succeed, root or not
    try:
        before = fx.kernel_cache_stats()
        assert fx.precompile(cfg2, N) == -5
        assert fx.kernel_cache_stats()["disk_write_failures"] == before["disk_write_failures"] + 1
    finally:
        fx.set_kernel_cache_dir(None)


def test_off_unless_asked(tmp_path, cfg2, version):
    """With no directory set there is no disk store: -3, and nothing appears under HOME or XDG_CACHE_HOME."""
    fx.set_kernel_cache_dir(None)
    assert fx.precompile(cfg2, N) == -3
    home, xdg = tmp_path / "home", tmp_path / "xdg"
    home.mkdir(); xdg.mkdir()
    env = {k: v for k, v in os.environ.items() if k != "FX8010_KERNEL_CACHE"}
    env.update(HOME=str(home), XDG_CACHE_HOME=str(xdg))
    p = run_precompile(env)
    out, err = p.communicate(timeout=300)
    assert p.returncode == 0, err
    assert int(out.strip().splitlines()[-1]) == -3
    assert list(home.rglob("*")) == [] and list(xdg.rglob("*")) == []
    # set_kernel_cache_dir(None) overrides the environment too
    fx.set_kernel_cache_dir(None)
    os.environ["FX8010_KERNEL_CACHE"] = str(tmp_path / "env_dir")
    try:
        assert fx.precompile(cfg2, N) == -3
    finally:
        del os.environ["FX8010_KERNEL_CACHE"]
    assert not (tmp_path / "env_dir").exists()


def test_fx8010_nvrtc_names_the_only_library(tmp_path, version):
    """A path in FX8010_NVRTC that cannot be loaded leaves the process without NVRTC (no other library is tried)."""
    env = dict(os.environ, FX8010_KERNEL_CACHE=str(tmp_path / "kcache"), FX8010_NVRTC=str(tmp_path / "no" / "libnvrtc.so"))
    p = run_precompile(env)
    out, err = p.communicate(timeout=300)
    assert p.returncode == 0, err
    assert int(out.strip().splitlines()[-1]) == -4
    assert not (tmp_path / "kcache").exists()
