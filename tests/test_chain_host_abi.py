"""Program chains from host memory, without a GPU: the new entry points are exported from both libraries with the layout the headers
declare, and a multi-GPU chain hands each shard the curve columns shard_range gives it."""
import ctypes

import numpy as np


def test_chain_host_symbols_exported(fx):
    gpu = ctypes.CDLL(fx.GPU_SO)
    for name in ("fx8010_chain_process_batch_host", "fx8010_chain_process_batch_host_curves", "fx8010_chain_synchronize",
                 "fx8010_multi_chain_create", "fx8010_multi_chain_destroy", "fx8010_multi_chain_process_batch_host",
                 "fx8010_multi_chain_process_batch_host_curves", "fx8010_multi_chain_synchronize", "fx8010_multi_chain_shard",
                 "fx8010_multi_chain_last_error", "fx8010_multi_shard_chain_curves"):
        assert hasattr(gpu, name), name
    fx.gpu_lib()
    host = ctypes.CDLL(fx.HOST_SO)
    for name in ("fx8010_host_chain_process_block", "fx8010_host_chain_process_block_curves"):
        assert hasattr(host, name), name
    assert ctypes.sizeof(fx.CChainHostCurve) == 24 and fx.CChainHostCurve.values.offset == 16
    assert ctypes.sizeof(fx.CChainHostCurve) == ctypes.sizeof(fx.CChainCurve)


def test_shard_chain_curve_columns_follow_shard_range(fx):
    """A per-instance curve's values move to the shard's first column; a broadcast curve and a NULL pointer pass as they are; stage and
    register are kept."""
    L = fx.gpu_lib()
    base = np.zeros(16, np.float32)
    p = base.ctypes.data
    spec = [(0, 3, 0, p), (2, 5, 1, p + 4), (1, 9, 0, None), (7, 1, 0, p + 8)]
    for n, G in [(1000, 3), (1002, 2), (65536, 8), (4096, 3), (7, 7), (5, 2), (65537, 6)]:
        curves = (fx.CChainHostCurve * len(spec))()
        for j, (stage, reg, bc, ptr) in enumerate(spec):
            curves[j].stage, curves[j].reg_index, curves[j].broadcast, curves[j].values = stage, reg, bc, ptr
        for g in range(G):
            lo, _ = fx.shard_range(n, g, G)
            out = (fx.CChainHostCurve * len(spec))()
            L.fx8010_multi_shard_chain_curves(ctypes.addressof(curves), len(spec), n, g, G, ctypes.addressof(out))
            assert [(c.stage, c.reg_index, c.broadcast) for c in out] == [(s, r, b) for s, r, b, _ in spec]
            assert out[0].values == p + 4 * lo, (n, g, G)
            assert out[1].values == p + 4 and out[2].values is None
            assert out[3].values == p + 8 + 4 * lo, (n, g, G)


def test_multi_chain_create_refuses_bad_lists_without_a_device(fx):
    """create checks its arguments before it looks at any executor."""
    L = fx.gpu_lib()
    h = ctypes.c_void_p()
    assert L.fx8010_multi_chain_create(None, 1, ctypes.byref(h)) == 1 and not h.value
    assert "stage count" in L.fx8010_multi_chain_last_error(None).decode()
    arr = (ctypes.c_void_p * 9)()
    assert L.fx8010_multi_chain_create(arr, 9, ctypes.byref(h)) == 1
    assert L.fx8010_multi_chain_create(arr, 1, ctypes.byref(h)) == 1
    assert "NULL" in L.fx8010_multi_chain_last_error(None).decode()
    assert L.fx8010_multi_chain_shard(None, 0) is None


def test_new_output_block_holds_every_row_a_slice_call_writes(fx):
    """With host_instances, a host-buffer chain call writes C * S rows host_instances floats apart: the output block the bindings allocate
    when the caller gives none is the first N columns of a block that wide, so every row lies inside it."""
    c, s, n, wide = 2, 4, 8, 16
    out = fx._host_out(None, c, s, n, wide)
    assert out.shape == (c, s, n) and out.dtype == np.float32
    assert out.strides == (4 * s * wide, 4 * wide, 4)
    assert out.base is not None and out.base.nbytes >= 4 * ((c * s - 1) * wide + n)
    fx._host_block(out, c * s, n, wide)                         # what the call's own check accepts
    plain = fx._host_out(None, c, s, n, 0)
    assert plain.shape == (c, s, n) and plain.flags.c_contiguous
