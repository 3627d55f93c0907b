"""Control curves from host memory, without a GPU: the new entry points are exported from both libraries with the layout the headers
declare, and the executor hands each shard the columns shard_range gives it."""
import ctypes

import numpy as np


def test_host_curve_symbols_exported(fx):
    gpu = ctypes.CDLL(fx.GPU_SO)
    for name in ("fx8010_gpu_process_batch_host_curves", "fx8010_multi_process_batch_host_curves", "fx8010_multi_shard_curves"):
        assert hasattr(gpu, name), name
    fx.gpu_lib()
    assert hasattr(ctypes.CDLL(fx.HOST_SO), "fx8010_host_process_block_curves")
    assert ctypes.sizeof(fx.CHostCurve) == 16 and fx.CHostCurve.values.offset == 8


def test_shard_curve_columns_follow_shard_range(fx):
    """A per-instance curve's values move to the shard's first column; a broadcast curve and a NULL pointer pass as they are."""
    L = fx.gpu_lib()
    base = np.zeros(16, np.float32)
    p = base.ctypes.data
    for n, G in [(1000, 3), (1002, 2), (65536, 8), (4096, 3), (7, 7), (5, 2), (65537, 6)]:
        curves = (fx.CHostCurve * 3)()
        for j, (reg, bc, ptr) in enumerate([(3, 0, p), (5, 1, p + 4), (9, 0, None)]):
            curves[j].reg_index, curves[j].broadcast, curves[j].values = reg, bc, ptr
        for g in range(G):
            lo, _ = fx.shard_range(n, g, G)
            out = (fx.CHostCurve * 3)()
            L.fx8010_multi_shard_curves(ctypes.addressof(curves), 3, n, g, G, ctypes.addressof(out))
            assert [(c.reg_index, c.broadcast) for c in out] == [(3, 0), (5, 1), (9, 0)]
            assert out[0].values == p + 4 * lo, (n, g, G)
            assert out[1].values == p + 4 and out[2].values is None
