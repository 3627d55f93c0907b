"""bench.py --dump-outputs: the file holds the output block of the last timed step, checked bit for bit against the oracle
replaying every block the run processed before it, on a sample of instances."""
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from conftest import PKG, ROOT, assert_bits_equal

pytestmark = pytest.mark.gpu


def test_dump_outputs_is_the_last_timed_step(po, tmp_path):
    import torch
    n, steps, warmup, repeats = 512, 3, 3, 2
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--instances", str(n), "--steps", str(steps), "--warmup", str(warmup),
                        "--repeats", str(repeats), "--no-cpu-baseline", "--no-e2e", "--no-interpreter-leg", "--no-sharded", "--no-parity",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    y = np.load(tmp_path / "out.npy")
    assert y.dtype == np.float32 and y.shape == (bench.BLOCK, n)

    W = bench.Workload(importlib.import_module(PKG), torch, "cfg2", n, 0, 0)      # the run's inputs, controls and buffer rotation
    W.close()
    idx = np.array(sorted({0, 1, n // 2, n - 1} | set(np.random.default_rng(7).integers(0, n, 28).tolist())))
    prog = W.prog
    img = po.Image(prog.instructions(), prog.registers(), prog.itram_size, prog.xtram_size, prog.controls(), prog.tables())
    orc = po.Oracle(img, len(idx), 1)
    for name, v in W.controls.items():
        orc.set_register(prog.reg_index(name), np.ascontiguousarray(v[idx]))
    # Workload.timed: a warm-up call of max(warmup, n_bufs) blocks, the timed call once untimed, then `repeats` timed regions;
    # block i of each call reads input buffer i % n_bufs, which holds host_in[(i % n_bufs) % 2]
    for blocks in [max(warmup, W.n_bufs), steps] + [steps] * repeats:
        for i in range(blocks):
            x = W.host_in[(i % W.n_bufs) % 2]
            want = orc.process(np.ascontiguousarray(x[:, idx]).reshape(1, bench.BLOCK, len(idx)))[0]
    assert_bits_equal(y[:, idx], want, "dumped block vs the oracle's last timed step")
