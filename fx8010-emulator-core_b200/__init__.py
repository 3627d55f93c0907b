"""fx8010-emulator-core_b200 — Python (ctypes) view of the product libraries.

The product is native: ``libfx8010_gpu.so`` (CUDA kernels + the C ABI of ``include/fx8010_gpu.h``)
and ``libfx8010_host.so`` (C++ front-end + the ``Klangraum::FX8010`` facade, C view in
``include/fx8010_host.h``).  This module only binds them so that tests and ``bench.py`` can drive
them; it holds no arithmetic of its own and never touches ``oracle/``.  Import it with
``importlib.import_module("fx8010-emulator-core_b200")`` (the directory name is not an identifier).

There is no CPU fallback: when the libraries are missing the import fails, and every compute call
raises ``FxError`` when no CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import weakref

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GPU_SO = os.path.join(HERE, "libfx8010_gpu.so")
HOST_SO = os.path.join(HERE, "libfx8010_host.so")

STATUS = {0: "OK", 1: "ERR_ARG", 2: "ERR_CUDA", 3: "ERR_NO_PROGRAM", 4: "ERR_PROGRAM", 5: "ERR_CAPACITY"}
RT_END_SKIPPED_CAP, RT_TABLE_RANGE = 1, 2
OPT_STREAM_EXCLUSIVE = 1
OPT_TRANSLATE = 2          # 0 never, 1 background compile (default), 2 compile before the first launch


class FxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{STATUS.get(code, code)}: {msg}")
        self.code = code


class CInstr(C.Structure):
    _fields_ = [("opcode", C.c_int32), ("r", C.c_int32), ("a", C.c_int32), ("x", C.c_int32),
                ("y", C.c_int32), ("has_input", C.c_uint8), ("has_output", C.c_uint8),
                ("has_noise", C.c_uint8), ("reserved", C.c_uint8)]


class CReg(C.Structure):
    _fields_ = [("type", C.c_int32), ("init_value", C.c_float), ("io_index", C.c_int32),
                ("is_noise", C.c_int32)]


class CImage(C.Structure):
    _fields_ = [("instrs", C.POINTER(CInstr)), ("n_instrs", C.c_int32),
                ("regs", C.POINTER(CReg)), ("n_regs", C.c_int32),
                ("itram_size", C.c_int32), ("xtram_size", C.c_int32),
                ("log_tables", C.POINTER(C.c_double)), ("exp_tables", C.POINTER(C.c_double))]


class CDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_instances", "n_channels", "n_regs", "n_instrs", "itram_size",
                                         "xtram_size", "itram_alloc", "xtram_alloc")]


class CControlEvent(C.Structure):
    _fields_ = [("sample", C.c_int32), ("reg_index", C.c_int32), ("broadcast", C.c_int32), ("reserved", C.c_int32), ("values", C.c_void_p)]


class CControlCurve(C.Structure):
    _fields_ = [("reg_index", C.c_int32), ("broadcast", C.c_int32), ("d_values", C.c_void_p)]


class CHostCurve(C.Structure):
    _fields_ = [("reg_index", C.c_int32), ("broadcast", C.c_int32), ("values", C.c_void_p)]


class CChainCurve(C.Structure):
    _fields_ = [("stage", C.c_int32), ("reg_index", C.c_int32), ("broadcast", C.c_int32), ("reserved", C.c_int32), ("d_values", C.c_void_p)]


class CChainHostCurve(C.Structure):
    _fields_ = [("stage", C.c_int32), ("reg_index", C.c_int32), ("broadcast", C.c_int32), ("reserved", C.c_int32), ("values", C.c_void_p)]


MAX_CONTROL_CURVES = 8
VARIANT_CURVES = 16        # fx8010_launch_info.kernel_variant: the last launch read control curves inside the kernel


class CLaunchInfo(C.Structure):
    _fields_ = [("kernel_launches", C.c_ulonglong), ("last_grid", C.c_int32), ("last_block", C.c_int32),
                ("last_time_split", C.c_int32), ("last_smem_bytes", C.c_int32), ("last_late_wait", C.c_int32),
                ("last_fused_blocks", C.c_int32), ("last_tma", C.c_int32), ("reserved", C.c_int32), ("kernel_variant", C.c_int32)]


class CKernelCacheStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("nvrtc_compiles", "memory_hits", "store_hits", "joined_compiles", "disk_hits", "disk_writes",
                                          "disk_rejected", "disk_write_failures")]


TRACE_DTYPE = np.dtype([("index", np.int32), ("executed", np.int32), ("r", np.float32), ("a", np.float32), ("x", np.float32),
                        ("y", np.float32), ("ccr", np.float32), ("opcode", np.int32), ("acc", np.float64)])


def build(force: bool = False) -> None:
    """Compile both libraries in-tree through the package Makefile (nvcc cross-compiles sm_100a)."""
    if force:
        subprocess.run(["make", "-s", "-C", HERE, "clean"], check=True)
    subprocess.run(["make", "-s", "-C", HERE, "all"], check=True)


_gpu = None
_host = None

GPU_SYMBOLS = {
    "fx8010_gpu_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "fx8010_gpu_destroy": (None, [C.c_void_p]),
    "fx8010_gpu_load_program": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fx8010_gpu_set_controls": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "fx8010_gpu_set_controls_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "fx8010_gpu_get_register": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_gpu_process_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_gpu_process_blocks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "fx8010_gpu_set_option": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "fx8010_gpu_process_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "fx8010_gpu_process_batch_host_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "fx8010_gpu_process_batch_host_slice": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_int]),
    "fx8010_gpu_process_batch_host_broadcast": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_int]),
    "fx8010_gpu_host_alloc": (C.c_void_p, [C.c_size_t]),
    "fx8010_gpu_host_free": (None, [C.c_void_p]),
    "fx8010_gpu_synchronize": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fx8010_gpu_get_instruction_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_ulonglong)]),
    "fx8010_gpu_get_instruction_counts": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fx8010_gpu_get_dims": (C.c_int, [C.c_void_p, C.POINTER(CDims)]),
    "fx8010_gpu_get_registers": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fx8010_gpu_set_registers": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fx8010_gpu_get_scalars": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fx8010_gpu_set_scalars": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fx8010_gpu_get_tram": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "fx8010_gpu_set_tram": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "fx8010_gpu_get_runtime_flags": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint), C.c_int]),
    "fx8010_gpu_last_error": (C.c_char_p, [C.c_void_p]),
    "fx8010_gpu_process_batch_events": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_gpu_process_batch_planar": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_gpu_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "fx8010_gpu_get_launch_info": (C.c_int, [C.c_void_p, C.POINTER(CLaunchInfo)]),
    "fx8010_gpu_translate_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_size_t]),
    "fx8010_translate_source": (C.c_longlong, [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.c_size_t, C.c_int, C.POINTER(C.c_int)]),
    "fx8010_gpu_translate_status_curves": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                                     C.c_char_p, C.c_size_t]),
    "fx8010_gpu_process_batch_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_translate_source_curves": (C.c_longlong, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_char_p, C.c_size_t,
                                                      C.c_int, C.POINTER(C.c_int)]),
    "fx8010_gpu_process_batch_host_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.c_int]),
    "fx8010_kernel_cache_set_dir": (C.c_int, [C.c_char_p]),
    "fx8010_kernel_cache_precompile": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "fx8010_kernel_cache_get_stats": (C.c_int, [C.POINTER(CKernelCacheStats)]),
    "fx8010_chain_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "fx8010_chain_destroy": (None, [C.c_void_p]),
    "fx8010_chain_process_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_chain_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_ulonglong), C.POINTER(C.c_int),
                                      C.POINTER(C.c_int), C.c_char_p, C.c_size_t]),
    "fx8010_chain_last_error": (C.c_char_p, [C.c_void_p]),
    "fx8010_translate_source_chain": (C.c_longlong, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_size_t, C.c_int, C.POINTER(C.c_int)]),
    "fx8010_chain_process_batch_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_chain_status_curves": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_size_t]),
    "fx8010_translate_source_chain_curves": (C.c_longlong, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                            C.c_char_p, C.c_size_t, C.c_int, C.POINTER(C.c_int)]),
    "fx8010_chain_process_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_int]),
    "fx8010_chain_process_batch_host_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.c_int]),
    "fx8010_chain_synchronize": (C.c_int, [C.c_void_p]),
}

MULTI_SYMBOLS = {
    "fx8010_multi_shard_range": (None, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "fx8010_multi_create": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "fx8010_multi_destroy": (None, [C.c_void_p]),
    "fx8010_multi_num_shards": (C.c_int, [C.c_void_p]),
    "fx8010_multi_shard": (C.c_void_p, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "fx8010_multi_load_program": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fx8010_multi_set_controls": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "fx8010_multi_get_register": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_multi_process_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "fx8010_multi_process_batch_host_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "fx8010_multi_process_batch_host_broadcast": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "fx8010_multi_process_batch_host_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "fx8010_multi_shard_curves": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fx8010_multi_synchronize": (C.c_int, [C.c_void_p]),
    "fx8010_multi_set_option": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "fx8010_multi_get_instruction_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_ulonglong)]),
    "fx8010_multi_get_registers": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fx8010_multi_get_runtime_flags": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint), C.c_int]),
    "fx8010_multi_last_error": (C.c_char_p, [C.c_void_p]),
    "fx8010_multi_chain_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "fx8010_multi_chain_destroy": (None, [C.c_void_p]),
    "fx8010_multi_chain_process_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "fx8010_multi_chain_process_batch_host_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "fx8010_multi_chain_synchronize": (C.c_int, [C.c_void_p]),
    "fx8010_multi_chain_shard": (C.c_void_p, [C.c_void_p, C.c_int]),
    "fx8010_multi_chain_last_error": (C.c_char_p, [C.c_void_p]),
    "fx8010_multi_shard_chain_curves": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

HOST_SYMBOLS = {
    "fx8010_host_create": (C.c_void_p, [C.c_int, C.c_int, C.c_int]),
    "fx8010_host_create_multi": (C.c_void_p, [C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int]),
    "fx8010_host_destroy": (None, [C.c_void_p]),
    "fx8010_host_last_error": (C.c_char_p, [C.c_void_p]),
    "fx8010_host_load_file": (C.c_int, [C.c_void_p, C.c_char_p]),
    "fx8010_host_load_text": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t]),
    "fx8010_host_ready": (C.c_int, [C.c_void_p]),
    "fx8010_host_set_relaxed": (None, [C.c_void_p, C.c_int]),
    "fx8010_host_set_translation": (C.c_int, [C.c_void_p, C.c_int]),
    "fx8010_host_set_kernel_cache_dir": (None, [C.c_char_p]),
    "fx8010_host_num_registers": (C.c_int, [C.c_void_p]),
    "fx8010_host_register_info": (None, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_float),
                                         C.POINTER(C.c_int), C.c_char_p, C.c_int]),
    "fx8010_host_num_instructions": (C.c_int, [C.c_void_p]),
    "fx8010_host_instruction_info": (None, [C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "fx8010_host_itram_size": (C.c_int, [C.c_void_p]),
    "fx8010_host_xtram_size": (C.c_int, [C.c_void_p]),
    "fx8010_host_tables": (None, [C.c_void_p, C.c_void_p]),
    "fx8010_host_image": (C.c_void_p, [C.c_void_p]),
    "fx8010_host_num_errors": (C.c_int, [C.c_void_p]),
    "fx8010_host_error_info": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_int]),
    "fx8010_host_num_controls": (C.c_int, [C.c_void_p]),
    "fx8010_host_control_name": (None, [C.c_void_p, C.c_int, C.c_char_p, C.c_int]),
    "fx8010_host_metadata": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int]),
    "fx8010_host_set_register": (C.c_int, [C.c_void_p, C.c_char_p, C.c_float]),
    "fx8010_host_get_register": (C.c_float, [C.c_void_p, C.c_char_p]),
    "fx8010_host_set_register_values": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p]),
    "fx8010_host_get_register_values": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p]),
    "fx8010_host_process": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "fx8010_host_process_block": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "fx8010_host_instruction_counter": (C.c_int, [C.c_void_p]),
    "fx8010_host_instruction_counter_total": (C.c_ulonglong, [C.c_void_p]),
    "fx8010_host_gpu": (C.c_void_p, [C.c_void_p]),
    "fx8010_host_process_block_device_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.c_void_p,
                                                          C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_host_process_block_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.c_void_p,
                                                   C.c_void_p, C.c_int]),
    "fx8010_host_chain_create": (C.c_void_p, [C.c_void_p, C.c_int]),
    "fx8010_host_chain_destroy": (None, [C.c_void_p]),
    "fx8010_host_chain_process_block_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_host_chain_last_error": (C.c_char_p, [C.c_void_p]),
    "fx8010_host_chain_process_block_device_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_char_p),
                                                                C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "fx8010_host_chain_process_block": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "fx8010_host_chain_process_block_curves": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_char_p),
                                                         C.c_void_p, C.c_void_p, C.c_int]),
}


def _bind(path, table):
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run __graft_entry__.build() (there is no CPU fallback)")
    lib = C.CDLL(path)          # RTLD_LOCAL: the facade and the reference harness both define Klangraum::FX8010
    for name, (res, args) in table.items():
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    return lib


def gpu_lib():
    global _gpu
    if _gpu is None:
        _gpu = _bind(GPU_SO, {**GPU_SYMBOLS, **MULTI_SYMBOLS})
    return _gpu


def host_lib():
    global _host
    if _host is None:
        gpu_lib()
        _host = _bind(HOST_SO, HOST_SYMBOLS)
    return _host


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):          # torch tensor
        return a.data_ptr()
    raise TypeError(type(a))


def _host_block(a, rows: int, cols: int, host_instances: int):
    """A host buffer of `rows` rows of `cols` instances for the host-curve calls: a float32 array (copied to a C-contiguous one when it is
    not), or with host_instances a view of `cols` columns of a C-contiguous array `host_instances` wide (its rows stay where they are)."""
    if a is None or isinstance(a, int):
        return a
    if not host_instances:
        return np.ascontiguousarray(a, dtype=np.float32).reshape(rows, cols)
    assert a.dtype == np.float32 and a.shape[-1] == cols and a.strides[-1] == 4 and a.size == rows * cols, "not float32 columns of a wider block"
    assert all(st == 4 * host_instances * int(np.prod(a.shape[k + 1:-1])) for k, st in enumerate(a.strides[:-1])), "rows not host_instances apart"
    return a


def _chain_host_curves(curves, s: int, n: int, host_instances: int):
    """[(stage, register index, ndarray, broadcast)] -> (fx8010_chain_host_curve array, the float32 arrays it points into)."""
    arr = (CChainHostCurve * max(1, len(curves)))()
    keep = []
    for i, (stage, reg, vals, bc) in enumerate(curves):
        v = np.ascontiguousarray(vals, dtype=np.float32).reshape(s) if bc else _host_block(vals, s, n, host_instances)
        keep.append(v)
        arr[i].stage, arr[i].reg_index, arr[i].broadcast, arr[i].values = int(stage), int(reg), 1 if bc else 0, v.ctypes.data
    return arr, keep


def _host_out(out, c: int, s: int, n: int, host_instances: int):
    """The output block of a host-buffer call: the caller's (checked like its input), or a new one — with host_instances, the first n
    columns of a new [C][S][host_instances] block, so that every row the call writes lies inside it."""
    if out is None:
        return np.zeros((c, s, host_instances or n), dtype=np.float32)[:, :, :n]
    if host_instances:
        _host_block(out, c * s, n, host_instances)
    else:
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == c * s * n
    return out


def _register_chain(chain, stages):
    """A chain reads its stages when it is destroyed: closing a stage closes the chains over it first."""
    for st in stages:
        st.__dict__.setdefault("_chains", []).append(weakref.ref(chain))


def _close_chains(obj):
    for ref in obj.__dict__.pop("_chains", []):
        c = ref()
        if c is not None:
            c.close()


def _host_curves(curves, s: int, n: int, host_instances: int):
    """[(register index, ndarray, broadcast)] -> (fx8010_host_curve array, the float32 arrays it points into)."""
    arr = (CHostCurve * max(1, len(curves)))()
    keep = []
    for i, (reg, vals, bc) in enumerate(curves):
        v = np.ascontiguousarray(vals, dtype=np.float32).reshape(s) if bc else _host_block(vals, s, n, host_instances)
        keep.append(v)
        arr[i].reg_index, arr[i].broadcast, arr[i].values = int(reg), 1 if bc else 0, v.ctypes.data
    return arr, keep


class Program:
    """The host front-end (class Klangraum::FX8010 through include/fx8010_host.h)."""

    def __init__(self, text: str | bytes | None = None, channels: int = 1, instances: int = 1, device: int = 0,
                 path: str | None = None, relaxed: bool = False, devices=None):
        self.L = host_lib()
        self.channels, self.instances, self.device = channels, instances, device
        if devices is not None:            # the facade's multi-GPU constructor: instances sharded over `devices`
            dev = (C.c_int * len(devices))(*devices)
            self.h = self.L.fx8010_host_create_multi(channels, instances, dev, len(devices))
        else:
            self.h = self.L.fx8010_host_create(channels, instances, device)
        if not self.h:
            raise ValueError("bad channel / instance count")
        self.loaded = None
        if relaxed:
            self.L.fx8010_host_set_relaxed(self.h, 1)
        if text is not None or path is not None:
            self.loaded = self.load(text=text, path=path)

    def close(self):
        _close_chains(self)
        if getattr(self, "h", None):
            self.L.fx8010_host_destroy(self.h)
            self.h = None

    __del__ = close

    def set_translation(self, mode: int):
        """FX8010::setTranslation — the program translator's mode for this object's device handle(s)."""
        if self.L.fx8010_host_set_translation(self.h, mode):
            raise ValueError("translation mode must be 0, 1 or 2")

    def load(self, text=None, path=None) -> bool:
        if path is not None:
            return bool(self.L.fx8010_host_load_file(self.h, path.encode()))
        data = text if isinstance(text, bytes) else text.encode()
        return bool(self.L.fx8010_host_load_text(self.h, data, len(data)))

    @property
    def ready(self) -> bool:
        return bool(self.L.fx8010_host_ready(self.h))

    def registers(self):
        out = []
        for i in range(self.L.fx8010_host_num_registers(self.h)):
            t, v, io = C.c_int(), C.c_float(), C.c_int()
            nb = C.create_string_buffer(256)
            self.L.fx8010_host_register_info(self.h, i, C.byref(t), C.byref(v), C.byref(io), nb, 256)
            out.append((t.value, np.float32(v.value), io.value, nb.value.decode("latin-1")))
        return out

    def instructions(self):
        out = []
        for i in range(self.L.fx8010_host_num_instructions(self.h)):
            f = (C.c_int * 8)()
            self.L.fx8010_host_instruction_info(self.h, i, f)
            out.append(tuple(int(v) for v in f))
        return out

    @property
    def itram_size(self): return self.L.fx8010_host_itram_size(self.h)
    @property
    def xtram_size(self): return self.L.fx8010_host_xtram_size(self.h)

    def tables(self) -> np.ndarray:
        t = np.zeros((2, 32, 64), dtype=np.float64)
        self.L.fx8010_host_tables(self.h, t.ctypes.data)
        return t

    def errors(self):
        out = []
        for i in range(self.L.fx8010_host_num_errors(self.h)):
            b = C.create_string_buffer(512)
            row = self.L.fx8010_host_error_info(self.h, i, b, 512)
            out.append((b.value.decode("latin-1"), row))
        return out

    def controls(self):
        out = []
        for i in range(self.L.fx8010_host_num_controls(self.h)):
            b = C.create_string_buffer(256)
            self.L.fx8010_host_control_name(self.h, i, b, 256)
            out.append(b.value.decode("latin-1"))
        return out

    def metadata(self):
        out = {}
        for k in ("name", "copyright", "created", "engine", "comment", "guid"):
            b = C.create_string_buffer(1024)
            if self.L.fx8010_host_metadata(self.h, k.encode(), b, 1024):
                out[k] = b.value.decode("latin-1")
        return out

    def reg_index(self, name: str) -> int:
        for i, r in enumerate(self.registers()):
            if r[3] == name:
                return i
        return -1

    def image_ptr(self) -> int:
        """const fx8010_program_image* (valid until the next load)."""
        return self.L.fx8010_host_image(self.h)

    # ---- facade compute members (need a GPU) ----
    def _check(self, rc, what):
        if rc != 0:
            raise FxError(2, f"{what}: {self.L.fx8010_host_last_error(self.h).decode()}")

    def set_register(self, name: str, v: float) -> int:
        rc = self.L.fx8010_host_set_register(self.h, name.encode(), float(v))
        if rc < 0:
            self._check(1, "setRegisterValue")
        return rc

    def get_register(self, name: str) -> float:
        return float(self.L.fx8010_host_get_register(self.h, name.encode()))

    def set_register_values(self, name: str, values) -> int:
        v = np.ascontiguousarray(values, dtype=np.float32)
        assert v.size == self.instances
        rc = self.L.fx8010_host_set_register_values(self.h, name.encode(), v.ctypes.data)
        if rc < 0:
            self._check(1, "setRegisterValues")
        return rc

    def process(self, x) -> np.ndarray:
        """Per-sample legacy path: x [S][C] -> [S][C] (instance 0)."""
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1, self.channels)
        out = np.zeros_like(x)
        self._check(self.L.fx8010_host_process(self.h, x.ctypes.data, out.ctypes.data, x.shape[0]), "process")
        return out

    def process_block_device_curves(self, d_in, d_out, n_samples: int, curves, stream=None):
        """FX8010::processBlockDeviceWithCurves: curves = [(register name, device tensor, broadcast)] (see Gpu.process_device_curves)."""
        n = len(curves)
        names = (C.c_char_p * max(1, n))(*[c[0].encode() for c in curves])
        ptrs = (C.c_void_p * max(1, n))(*[_ptr(c[1]) for c in curves])
        bc = (C.c_int32 * max(1, n))(*[1 if c[2] else 0 for c in curves])
        self._check(self.L.fx8010_host_process_block_device_curves(self.h, _ptr(d_in), _ptr(d_out), n_samples, names, ptrs, bc, n, stream),
                    "processBlockDeviceWithCurves")

    def process_block_curves(self, x, curves, n_samples=None) -> np.ndarray:
        """FX8010::processBlockWithCurves: x [C][S][N] (None: no input) -> [C][S][N]; curves = [(register name, ndarray, broadcast)], each
        [S][N] float32, or [S] with broadcast.  On one device or, with `devices`, on several."""
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.channels, -1, self.instances)
            n_samples = x.shape[1]
        out = np.zeros((self.channels, n_samples, self.instances), dtype=np.float32)
        vals = [np.ascontiguousarray(v, dtype=np.float32).reshape(n_samples) if bc else
                np.ascontiguousarray(v, dtype=np.float32).reshape(n_samples, self.instances) for _, v, bc in curves]
        n = len(curves)
        names = (C.c_char_p * max(1, n))(*[c[0].encode() for c in curves])
        ptrs = (C.c_void_p * max(1, n))(*[v.ctypes.data for v in vals])
        bc = (C.c_int * max(1, n))(*[1 if c[2] else 0 for c in curves])
        self._check(self.L.fx8010_host_process_block_curves(self.h, _ptr(x), out.ctypes.data, n_samples, names, ptrs, bc, n), "processBlockWithCurves")
        return out

    def process_block(self, x, n_samples=None) -> np.ndarray:
        """Batched path with host buffers: x [C][S][N] -> [C][S][N]."""
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.channels, -1, self.instances)
            n_samples = x.shape[1]
        out = np.zeros((self.channels, n_samples, self.instances), dtype=np.float32)
        self._check(self.L.fx8010_host_process_block(self.h, _ptr(x), out.ctypes.data, n_samples), "processBlock")
        return out

    def chain(self, later):
        """Klangraum::FX8010Chain of this object followed by the Programs `later`: a callable (d_in, d_out, n_samples, stream=None) that runs
        processBlockDevice, with .close().  Close it before the objects."""
        return ProgramChain([self] + list(later))

    @property
    def instruction_counter(self) -> int:
        return self.L.fx8010_host_instruction_counter(self.h)

    @property
    def instruction_counter_total(self) -> int:
        return self.L.fx8010_host_instruction_counter_total(self.h)


class ProgramChain:
    """Klangraum::FX8010Chain through include/fx8010_host.h (see Program.chain)."""

    def __init__(self, programs):
        self.L = host_lib()
        self.programs = list(programs)
        arr = (C.c_void_p * max(1, len(self.programs)))(*[p.h for p in self.programs])
        self.h = self.L.fx8010_host_chain_create(arr, len(self.programs))
        if not self.h:
            raise FxError(1, self.L.fx8010_host_chain_last_error(None).decode())
        _register_chain(self, self.programs)

    def __call__(self, d_in, d_out, n_samples: int, stream=None):
        if self.L.fx8010_host_chain_process_block_device(self.h, _ptr(d_in), _ptr(d_out), n_samples, stream):
            raise FxError(2, self.L.fx8010_host_chain_last_error(self.h).decode())

    def process_block(self, x, n_samples=None) -> np.ndarray:
        """FX8010Chain::processBlock: host buffers, x [C][S][N] (None: no input) -> [C][S][N]."""
        p0 = self.programs[0]
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(p0.channels, -1, p0.instances)
            n_samples = x.shape[1]
        out = np.zeros((p0.channels, n_samples, p0.instances), dtype=np.float32)
        if self.L.fx8010_host_chain_process_block(self.h, _ptr(x), out.ctypes.data, n_samples):
            raise FxError(2, self.L.fx8010_host_chain_last_error(self.h).decode())
        return out

    def process_block_curves(self, x, curves, n_samples=None) -> np.ndarray:
        """FX8010Chain::processBlockWithCurves: curves = [(stage, register name, ndarray, broadcast)], each [S][N] float32, or [S] with
        broadcast."""
        p0 = self.programs[0]
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(p0.channels, -1, p0.instances)
            n_samples = x.shape[1]
        out = np.zeros((p0.channels, n_samples, p0.instances), dtype=np.float32)
        n = len(curves)
        vals = [np.ascontiguousarray(c[2], dtype=np.float32) for c in curves]
        stages = (C.c_int * max(1, n))(*[int(c[0]) for c in curves])
        names = (C.c_char_p * max(1, n))(*[c[1].encode() for c in curves])
        ptrs = (C.c_void_p * max(1, n))(*[v.ctypes.data for v in vals])
        bc = (C.c_int * max(1, n))(*[1 if c[3] else 0 for c in curves])
        if self.L.fx8010_host_chain_process_block_curves(self.h, _ptr(x), out.ctypes.data, n_samples, stages, names, ptrs, bc, n):
            raise FxError(2, self.L.fx8010_host_chain_last_error(self.h).decode())
        return out

    def process_curves(self, d_in, d_out, n_samples: int, curves, stream=None):
        """FX8010Chain::processBlockDeviceWithCurves: curves = [(stage, register name, device tensor, broadcast)]."""
        n = len(curves)
        stages = (C.c_int * max(1, n))(*[int(c[0]) for c in curves])
        names = (C.c_char_p * max(1, n))(*[c[1].encode() for c in curves])
        ptrs = (C.c_void_p * max(1, n))(*[_ptr(c[2]) for c in curves])
        bc = (C.c_int * max(1, n))(*[1 if c[3] else 0 for c in curves])
        if self.L.fx8010_host_chain_process_block_device_curves(self.h, _ptr(d_in), _ptr(d_out), n_samples, stages, names, ptrs, bc, n, stream):
            raise FxError(2, self.L.fx8010_host_chain_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.fx8010_host_chain_destroy(self.h)
            self.h = None

    __del__ = close


def translate_source(prog: "Program", channels: int = 1, compile_check: bool = False, instances: int = 1):
    """CUDA source the translator generates for a decoded program (no device needed).  Returns (source or None when the
    program is not eligible, CUBIN size when compile_check else None)."""
    L = gpu_lib()
    n = L.fx8010_translate_source(prog.image_ptr(), instances, channels, None, 0, 0, None)
    if n < 0:
        return None, None
    buf = C.create_string_buffer(int(n) + 1)
    cub = C.c_int(0)
    L.fx8010_translate_source(prog.image_ptr(), instances, channels, buf, int(n) + 1, 1 if compile_check else 0, C.byref(cub))
    return buf.value.decode(), (cub.value if compile_check else None)


def translate_source_curves(prog: "Program", curves, channels: int = 1, compile_check: bool = False, instances: int = 1):
    """translate_source for the translation fx8010_gpu_process_batch_curves uses: curves = [(register index, broadcast)].
    Returns (None, None) when the program is not eligible (e.g. an automated SKIP count)."""
    L = gpu_lib()
    k = len(curves)
    regs = (C.c_int32 * max(1, k))(*[int(c[0]) for c in curves])
    bc = (C.c_int32 * max(1, k))(*[1 if c[1] else 0 for c in curves])
    n = L.fx8010_translate_source_curves(prog.image_ptr(), instances, channels, regs, bc, k, None, 0, 0, None)
    if n < 0:
        return None, None
    buf = C.create_string_buffer(int(n) + 1)
    cub = C.c_int(0)
    L.fx8010_translate_source_curves(prog.image_ptr(), instances, channels, regs, bc, k, buf, int(n) + 1, 1 if compile_check else 0, C.byref(cub))
    return buf.value.decode(), (cub.value if compile_check else None)


def translate_source_chain(progs, channels: int = 1, compile_check: bool = False, instances: int = 1):
    """The source of the fused kernel of a chain of the decoded programs `progs` (fx8010_translate_source_chain; no device needed).
    Returns (source or None when some stage is not stateless, CUBIN size when compile_check else None)."""
    L = gpu_lib()
    imgs = (C.c_void_p * max(1, len(progs)))(*[p.image_ptr() for p in progs])
    n = L.fx8010_translate_source_chain(imgs, len(progs), instances, channels, None, 0, 0, None)
    if n == -1:
        raise ValueError("bad image list")
    if n < 0:
        return None, None
    buf = C.create_string_buffer(int(n) + 1)
    cub = C.c_int(0)
    L.fx8010_translate_source_chain(imgs, len(progs), instances, channels, buf, int(n) + 1, 1 if compile_check else 0, C.byref(cub))
    return buf.value.decode(), (cub.value if compile_check else None)


def translate_source_chain_curves(progs, curves, channels: int = 1, compile_check: bool = False, instances: int = 1):
    """translate_source_chain for the kernel fx8010_chain_process_batch_curves uses: curves = [(stage, register index, broadcast)].
    Returns (None, None) when some stage is not stateless; raises ValueError for an image or curve list the call refuses."""
    L = gpu_lib()
    imgs = (C.c_void_p * max(1, len(progs)))(*[p.image_ptr() for p in progs])
    k = len(curves)
    stage = (C.c_int32 * max(1, k))(*[int(c[0]) for c in curves])
    regs = (C.c_int32 * max(1, k))(*[int(c[1]) for c in curves])
    bc = (C.c_int32 * max(1, k))(*[1 if c[2] else 0 for c in curves])
    n = L.fx8010_translate_source_chain_curves(imgs, len(progs), instances, channels, stage, regs, bc, k, None, 0, 0, None)
    if n == -1:
        raise ValueError("bad image or curve list")
    if n < 0:
        return None, None
    buf = C.create_string_buffer(int(n) + 1)
    cub = C.c_int(0)
    L.fx8010_translate_source_chain_curves(imgs, len(progs), instances, channels, stage, regs, bc, k, buf, int(n) + 1, 1 if compile_check else 0,
                                           C.byref(cub))
    return buf.value.decode(), (cub.value if compile_check else None)


def set_kernel_cache_dir(path) -> None:
    """Directory of the translator's disk kernel cache for the whole process (overrides FX8010_KERNEL_CACHE); None or "" turns it off."""
    gpu_lib().fx8010_kernel_cache_set_dir(os.fsencode(path) if path else None)


def kernel_cache_stats() -> dict:
    """Process-wide kernel cache counters (fx8010_kernel_cache_stats)."""
    st = CKernelCacheStats()
    gpu_lib().fx8010_kernel_cache_get_stats(C.byref(st))
    return {name: int(getattr(st, name)) for name, _ in CKernelCacheStats._fields_}


def precompile(prog: "Program", instances: int, channels: int = 1, curves=None) -> int:
    """Compile the translated kernel a handle of `instances` instances would use for `prog` (curves = [(register index, broadcast)] for
    the control-curve translation) into the disk kernel cache, without a device.  Returns fx8010_kernel_cache_precompile's code:
    0 written, 1 already there, -1 bad arguments, -2 not eligible, -3 no cache directory, -4 compile failed, -5 write failed."""
    curves = curves or []
    k = len(curves)
    regs = (C.c_int32 * max(1, k))(*[int(c[0]) for c in curves])
    bc = (C.c_int32 * max(1, k))(*[1 if c[1] else 0 for c in curves])
    return gpu_lib().fx8010_kernel_cache_precompile(prog.image_ptr(), instances, channels, regs, bc, k)


class Gpu:
    """One fx8010_gpu handle: N instances of one decoded program on one GPU (include/fx8010_gpu.h)."""

    def __init__(self, instances: int, channels: int = 1, device: int = 0):
        self.L = gpu_lib()
        self.n, self.c = instances, channels
        h = C.c_void_p()
        rc = self.L.fx8010_gpu_create(device, instances, channels, C.byref(h))
        if rc != 0:
            raise FxError(rc, self.L.fx8010_gpu_last_error(None).decode())
        self.h = h
        self._keep = None

    def close(self):
        _close_chains(self)
        if getattr(self, "h", None):
            self.L.fx8010_gpu_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc):
        if rc != 0:
            raise FxError(rc, self.L.fx8010_gpu_last_error(self.h).decode())

    def load_image_ptr(self, image_ptr: int):
        self._check(self.L.fx8010_gpu_load_program(self.h, image_ptr))

    def load(self, instrs, regs, itram_size=0, xtram_size=0, tables=None):
        """instrs: (opcode, r, a, x, y, has_input, has_output, has_noise); regs: (type, init, io, name);
        tables: [2][32][64] float64 (LOG, EXP) — they come from the host front-end."""
        ins = (CInstr * max(1, len(instrs)))()
        for k, t in enumerate(instrs):
            ins[k].opcode, ins[k].r, ins[k].a, ins[k].x, ins[k].y = [int(v) for v in t[:5]]
            ins[k].has_input, ins[k].has_output, ins[k].has_noise = int(t[5]), int(t[6]), int(t[7])
        rg = (CReg * max(1, len(regs)))()
        for k, t in enumerate(regs):
            rg[k].type = int(t[0]); rg[k].init_value = float(np.float32(t[1]))
            rg[k].io_index = int(t[2]); rg[k].is_noise = 1 if t[3] == "noise" else 0
        tabs = np.ascontiguousarray(tables, dtype=np.float64)
        img = CImage(ins, len(instrs), rg, len(regs), int(itram_size), int(xtram_size),
                     tabs[0].ctypes.data_as(C.POINTER(C.c_double)), tabs[1].ctypes.data_as(C.POINTER(C.c_double)))
        self._keep = (ins, rg, tabs, img)
        self._check(self.L.fx8010_gpu_load_program(self.h, C.addressof(img)))
        self.n_regs = len(regs)

    def load_program(self, prog: Program):
        self._check(self.L.fx8010_gpu_load_program(self.h, prog.image_ptr()))
        self.n_regs = len(prog.registers())

    def dims(self) -> CDims:
        d = CDims()
        self._check(self.L.fx8010_gpu_get_dims(self.h, C.byref(d)))
        return d

    def set_controls(self, reg: int, values, broadcast: bool = False):
        v = np.ascontiguousarray(np.atleast_1d(values), dtype=np.float32)
        self._check(self.L.fx8010_gpu_set_controls(self.h, reg, v.ctypes.data, 1 if broadcast else 0))

    def set_controls_device(self, reg: int, d_values, stream=None):
        self._check(self.L.fx8010_gpu_set_controls_device(self.h, reg, _ptr(d_values), stream))

    def get_register(self, reg: int) -> np.ndarray:
        out = np.zeros(self.n, dtype=np.float32)
        self._check(self.L.fx8010_gpu_get_register(self.h, reg, out.ctypes.data))
        return out

    def process_device(self, d_in, d_out, n_samples: int, stream=None):
        self._check(self.L.fx8010_gpu_process_batch(self.h, _ptr(d_in), _ptr(d_out), n_samples, stream))

    def process_blocks(self, d_ins, d_outs, n_samples: int, stream=None):
        """Consecutive blocks in one call: d_ins / d_outs are sequences of device buffers (d_ins may be None)."""
        nb = len(d_outs)
        outs = (C.c_void_p * max(1, nb))(*[_ptr(o) for o in d_outs])
        ins = None if d_ins is None else (C.c_void_p * max(1, nb))(*[_ptr(i) for i in d_ins])
        self._check(self.L.fx8010_gpu_process_blocks(self.h, ins, outs, nb, n_samples, stream))

    def block_pointers(self, d_ins, d_outs):
        """Pointer arrays for process_blocks_raw (built once, reused across calls)."""
        nb = len(d_outs)
        return (None if d_ins is None else (C.c_void_p * nb)(*[_ptr(i) for i in d_ins])), (C.c_void_p * nb)(*[_ptr(o) for o in d_outs]), nb

    def process_blocks_raw(self, ptrs, n_samples: int, stream=None):
        self._check(self.L.fx8010_gpu_process_blocks(self.h, ptrs[0], ptrs[1], ptrs[2], n_samples, stream))

    def set_option(self, option: int, value: int):
        self._check(self.L.fx8010_gpu_set_option(self.h, option, value))

    def translate_status(self) -> dict:
        """State of the program translator (FX8010_OPT_TRANSLATE): 0 not attempted, 1 compiling, 2 in use, -1 not translated."""
        st, regs, loc = C.c_int(0), C.c_int(0), C.c_int(0)
        msg = C.create_string_buffer(4096)
        self._check(self.L.fx8010_gpu_translate_status(self.h, C.byref(st), C.byref(regs), C.byref(loc), msg, 4096))
        return {"state": st.value, "regs_per_thread": regs.value, "local_bytes": loc.value, "message": msg.value.decode(errors="replace")}

    def translate_status_curves(self) -> dict:
        """translate_status for the most recent control-curve set (process_device_curves), plus the kernel kind in use (-1: none)."""
        st, regs, loc, kind = C.c_int(0), C.c_int(0), C.c_int(0), C.c_int(-1)
        msg = C.create_string_buffer(4096)
        self._check(self.L.fx8010_gpu_translate_status_curves(self.h, C.byref(st), C.byref(regs), C.byref(loc), C.byref(kind), msg, 4096))
        return {"state": st.value, "regs_per_thread": regs.value, "local_bytes": loc.value, "kind": kind.value,
                "message": msg.value.decode(errors="replace")}

    def process_device_events(self, d_in, d_out, n_samples: int, events, stream=None):
        """events: iterable of (sample, reg_index, value) with value a float (broadcast) or an array of N floats."""
        arr = (CControlEvent * max(1, len(events)))()
        keep = []
        for i, (sample, reg, val) in enumerate(events):
            v = np.ascontiguousarray(np.atleast_1d(val), dtype=np.float32)
            keep.append(v)
            arr[i].sample, arr[i].reg_index, arr[i].broadcast, arr[i].values = sample, reg, int(v.size == 1), v.ctypes.data
        self._check(self.L.fx8010_gpu_process_batch_events(self.h, _ptr(d_in), _ptr(d_out), n_samples, C.addressof(arr), len(events), stream))

    def process_device_curves(self, d_in, d_out, n_samples: int, curves, stream=None):
        """curves: iterable of (reg_index, device buffer, broadcast) — [n_samples][N] float32 values, or [n_samples] with broadcast —
        followed sample period by sample period (fx8010_gpu_process_batch_curves)."""
        curves = list(curves)
        arr = (CControlCurve * max(1, len(curves)))()
        for i, (reg, vals, bc) in enumerate(curves):
            arr[i].reg_index, arr[i].broadcast, arr[i].d_values = int(reg), 1 if bc else 0, _ptr(vals)
        self._check(self.L.fx8010_gpu_process_batch_curves(self.h, _ptr(d_in), _ptr(d_out), n_samples, C.addressof(arr), len(curves), stream))

    def process_device_planar(self, d_in, d_out, n_samples: int, stream=None):
        self._check(self.L.fx8010_gpu_process_batch_planar(self.h, _ptr(d_in), _ptr(d_out), n_samples, stream))

    def process_host(self, x, n_samples=None, out=None) -> np.ndarray:
        if x is not None and not isinstance(x, int):
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1, self.n)
            n_samples = x.shape[1]
        if out is None:
            out = np.zeros((self.c, n_samples, self.n), dtype=np.float32)
        self._check(self.L.fx8010_gpu_process_batch_host(self.h, _ptr(x), _ptr(out), n_samples))
        return out

    def process_host_broadcast(self, x, out=None, wait: bool = True) -> np.ndarray:
        """x: [C][S] — one input signal for all instances; returns / fills out [C][S][N]."""
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1)
        if out is None:
            out = np.zeros((self.c, x.shape[1], self.n), dtype=np.float32)
        self._check(self.L.fx8010_gpu_process_batch_host_broadcast(self.h, _ptr(x), _ptr(out), x.shape[1], 0, 1 if wait else 0))
        self._keep_bcast = x
        return out

    def process_host_curves(self, x, curves, out=None, wait: bool = True, host_instances: int = 0, n_samples=None) -> np.ndarray:
        """fx8010_gpu_process_batch_host_curves: x [C][S][N] (None: no input) -> out [C][S][N]; curves = [(reg_index, ndarray, broadcast)],
        each [S][N] float32, or [S] with broadcast.  With host_instances, x, out and the per-instance curves are views of N columns of
        C-contiguous arrays host_instances wide (e.g. big[..., lo:lo + N]).  wait=False queues the work; the arrays are kept until
        synchronize()."""
        if x is not None:
            n_samples = x.shape[1]
        x = _host_block(x, self.c * n_samples, self.n, host_instances)
        if out is None:
            out = np.zeros((self.c, n_samples, self.n), dtype=np.float32)
        if host_instances:
            _host_block(out, self.c * n_samples, self.n, host_instances)
        else:
            assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == self.c * n_samples * self.n
        arr, keep = _host_curves(curves, n_samples, self.n, host_instances)
        self._check(self.L.fx8010_gpu_process_batch_host_curves(self.h, _ptr(x), _ptr(out), n_samples, C.addressof(arr), len(curves),
                                                                host_instances, 1 if wait else 0))
        self._pending = [] if wait else getattr(self, "_pending", []) + [(x, out, arr, keep)]
        return out

    def process_host_ptr(self, in_ptr: int, out_ptr: int, n_samples: int, wait: bool = True):
        f = self.L.fx8010_gpu_process_batch_host if wait else self.L.fx8010_gpu_process_batch_host_async
        self._check(f(self.h, in_ptr, out_ptr, n_samples))

    def synchronize(self, stream=None):
        self._check(self.L.fx8010_gpu_synchronize(self.h, stream))
        self._pending = []

    def registers(self) -> np.ndarray:
        out = np.zeros((self.dims().n_regs, self.n), dtype=np.float32)
        self._check(self.L.fx8010_gpu_get_registers(self.h, out.ctypes.data))
        return out

    def set_registers(self, regs):
        v = np.ascontiguousarray(regs, dtype=np.float32)
        self._check(self.L.fx8010_gpu_set_registers(self.h, v.ctypes.data))

    def scalars(self):
        acc = np.zeros(self.n, dtype=np.float64); lfsr = np.zeros((2, self.n), dtype=np.uint32)
        latch = np.zeros((self.c, self.n), dtype=np.float32); ptrs = np.zeros((4, self.n), dtype=np.int32)
        self._check(self.L.fx8010_gpu_get_scalars(self.h, acc.ctypes.data, lfsr.ctypes.data, latch.ctypes.data, ptrs.ctypes.data))
        return acc, lfsr, latch, ptrs

    def set_scalars(self, acc=None, lfsr=None, latch=None, ptrs=None):
        conv = lambda a, dt: None if a is None else np.ascontiguousarray(a, dtype=dt)
        acc, lfsr, latch, ptrs = conv(acc, np.float64), conv(lfsr, np.uint32), conv(latch, np.float32), conv(ptrs, np.int32)
        self._check(self.L.fx8010_gpu_set_scalars(self.h, _ptr(acc), _ptr(lfsr), _ptr(latch), _ptr(ptrs)))

    def tram(self, which: int, instance: int) -> np.ndarray:
        d = self.dims()
        out = np.zeros(d.itram_size if which == 0 else d.xtram_size, dtype=np.float32)
        self._check(self.L.fx8010_gpu_get_tram(self.h, which, instance, out.ctypes.data))
        return out

    def set_tram(self, which: int, instance: int, values):
        v = np.ascontiguousarray(values, dtype=np.float32)
        self._check(self.L.fx8010_gpu_set_tram(self.h, which, instance, v.ctypes.data))

    def counts(self) -> np.ndarray:
        out = np.zeros(self.n, dtype=np.uint64)
        self._check(self.L.fx8010_gpu_get_instruction_counts(self.h, out.ctypes.data))
        return out

    def count_total(self) -> int:
        t = C.c_ulonglong(0)
        self._check(self.L.fx8010_gpu_get_instruction_count(self.h, C.byref(t)))
        return int(t.value)

    def flags(self, clear: bool = False) -> int:
        f = C.c_uint(0)
        self._check(self.L.fx8010_gpu_get_runtime_flags(self.h, C.byref(f), 1 if clear else 0))
        return int(f.value)

    def trace(self, x, instance: int, n_samples=None):
        """Runs the block like process_host and returns (out [C][S][N], records [S][n_instrs]) for one instance."""
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1, self.n)
            n_samples = x.shape[1]
        out = np.zeros((self.c, n_samples, self.n), dtype=np.float32)
        rec = np.zeros((n_samples, self.dims().n_instrs), dtype=TRACE_DTYPE)
        self._check(self.L.fx8010_gpu_trace(self.h, _ptr(x), out.ctypes.data, n_samples, instance, rec.ctypes.data))
        return out, rec

    def launch_info(self) -> CLaunchInfo:
        i = CLaunchInfo()
        self._check(self.L.fx8010_gpu_get_launch_info(self.h, C.byref(i)))
        return i


MAX_CHAIN_STAGES = 8


class Chain:
    """Several Gpu handles run one after another within every sample period (include/fx8010_gpu.h, fx8010_chain_*).  It is closed
    before the handles: closing a handle closes the chains over it first."""

    def __init__(self, stages):
        self.L = gpu_lib()
        self.stages = list(stages)
        arr = (C.c_void_p * max(1, len(self.stages)))(*[g.h.value for g in self.stages])
        h = C.c_void_p()
        rc = self.L.fx8010_chain_create(arr, len(self.stages), C.byref(h))
        if rc != 0:
            raise FxError(rc, self.L.fx8010_chain_last_error(None).decode())
        self.h = h
        _register_chain(self, self.stages)

    def close(self):
        if getattr(self, "h", None):
            self.L.fx8010_chain_destroy(self.h)
            self.h = None

    __del__ = close

    def process_batch(self, d_in, d_out, n: int, stream=None):
        rc = self.L.fx8010_chain_process_batch(self.h, _ptr(d_in), _ptr(d_out), n, stream)
        if rc != 0:
            raise FxError(rc, self.L.fx8010_chain_last_error(self.h).decode())

    def status(self) -> dict:
        return _chain_status(self.L, self.h)

    def process_batch_curves(self, d_in, d_out, n: int, curves, stream=None):
        """fx8010_chain_process_batch_curves: curves = [(stage, register index, device buffer, broadcast)] — [n][N] float32 values, or [n]
        with broadcast."""
        curves = list(curves)
        arr = (CChainCurve * max(1, len(curves)))()
        for i, (stage, reg, vals, bc) in enumerate(curves):
            arr[i].stage, arr[i].reg_index, arr[i].broadcast, arr[i].d_values = int(stage), int(reg), 1 if bc else 0, _ptr(vals)
        rc = self.L.fx8010_chain_process_batch_curves(self.h, _ptr(d_in), _ptr(d_out), n, C.addressof(arr), len(curves), stream)
        if rc != 0:
            raise FxError(rc, self.L.fx8010_chain_last_error(self.h).decode())

    def status_curves(self) -> dict:
        """fx8010_chain_status_curves: the fused kernel of the most recent curve list."""
        st, regs, loc = C.c_int(0), C.c_int(0), C.c_int(0)
        msg = C.create_string_buffer(4096)
        self.L.fx8010_chain_status_curves(self.h, C.byref(st), C.byref(regs), C.byref(loc), msg, 4096)
        return {"state": st.value, "regs_per_thread": regs.value, "local_bytes": loc.value, "message": msg.value.decode(errors="replace")}

    def process_host(self, x, n_samples=None, out=None, wait: bool = True, host_instances: int = 0) -> np.ndarray:
        """fx8010_chain_process_batch_host: x [C][S][N] (None: no input) -> out [C][S][N].  With host_instances, x and out are views of N
        columns of C-contiguous arrays host_instances wide (as in Gpu.process_host_curves).  wait=False queues the work; the arrays are
        kept until synchronize()."""
        return self.process_host_curves(x, [], n_samples=n_samples, out=out, wait=wait, host_instances=host_instances)

    def process_host_curves(self, x, curves, n_samples=None, out=None, wait: bool = True, host_instances: int = 0) -> np.ndarray:
        """fx8010_chain_process_batch_host_curves: curves = [(stage, register index, ndarray, broadcast)], each [S][N] float32 (N columns of
        a host_instances-wide array with host_instances), or [S] with broadcast; the rest as in process_host."""
        g0 = self.stages[0]
        if x is not None:
            n_samples = x.shape[1]
        x = _host_block(x, g0.c * n_samples, g0.n, host_instances)
        out = _host_out(out, g0.c, n_samples, g0.n, host_instances)
        arr, keep = _chain_host_curves(curves, n_samples, g0.n, host_instances)
        rc = self.L.fx8010_chain_process_batch_host_curves(self.h, _ptr(x), _ptr(out), n_samples, C.addressof(arr), len(curves), host_instances,
                                                           1 if wait else 0)
        if rc != 0:
            raise FxError(rc, self.L.fx8010_chain_last_error(self.h).decode())
        self._pending = [] if wait else getattr(self, "_pending", []) + [(x, out, arr, keep)]
        return out

    def synchronize(self):
        rc = self.L.fx8010_chain_synchronize(self.h)
        if rc != 0:
            raise FxError(rc, self.L.fx8010_chain_last_error(self.h).decode())
        self._pending = []


def _chain_status(L, h) -> dict:
    st, fused, regs, loc, launches = C.c_int(0), C.c_int(0), C.c_int(0), C.c_int(0), C.c_ulonglong(0)
    msg = C.create_string_buffer(4096)
    L.fx8010_chain_status(h, C.byref(st), C.byref(fused), C.byref(launches), C.byref(regs), C.byref(loc), msg, 4096)
    return {"state": st.value, "fused_last": fused.value, "launches": int(launches.value), "regs_per_thread": regs.value,
            "local_bytes": loc.value, "message": msg.value.decode(errors="replace")}


class MultiGpu:
    """One program over N instances spread across several GPUs (include/fx8010_multi.h): contiguous instance ranges,
    one host thread per device, outputs gathered into ONE host buffer [channel][sample][instance]."""

    def __init__(self, devices, instances: int, channels: int = 1):
        self.L = gpu_lib()
        self.n, self.c = instances, channels
        dev = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = self.L.fx8010_multi_create(dev, len(devices), instances, channels, C.byref(h))
        if rc != 0:
            raise FxError(rc, self.L.fx8010_multi_last_error(None).decode())
        self.h = h

    def close(self):
        _close_chains(self)
        if getattr(self, "h", None):
            self.L.fx8010_multi_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc):
        if rc != 0:
            raise FxError(rc, self.L.fx8010_multi_last_error(self.h).decode())

    def shards(self):
        out = []
        for g in range(self.L.fx8010_multi_num_shards(self.h)):
            lo, hi = C.c_int(), C.c_int()
            self.L.fx8010_multi_shard(self.h, g, C.byref(lo), C.byref(hi))
            out.append((lo.value, hi.value))
        return out

    def load_program(self, prog: "Program"):
        self._check(self.L.fx8010_multi_load_program(self.h, prog.image_ptr()))
        self.n_regs = len(prog.registers())

    def set_controls(self, reg: int, values, broadcast: bool = False):
        v = np.ascontiguousarray(np.atleast_1d(values), dtype=np.float32)
        assert broadcast or v.size == self.n
        self._check(self.L.fx8010_multi_set_controls(self.h, reg, v.ctypes.data, 1 if broadcast else 0))

    def get_register(self, reg: int) -> np.ndarray:
        out = np.zeros(self.n, dtype=np.float32)
        self._check(self.L.fx8010_multi_get_register(self.h, reg, out.ctypes.data))
        return out

    def process_host(self, x, n_samples=None, out=None, wait: bool = True) -> np.ndarray:
        if x is not None and not isinstance(x, int):
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1, self.n)
            n_samples = x.shape[1]
        if out is None:
            out = np.zeros((self.c, n_samples, self.n), dtype=np.float32)
        f = self.L.fx8010_multi_process_batch_host if wait else self.L.fx8010_multi_process_batch_host_async
        self._check(f(self.h, _ptr(x), _ptr(out), n_samples))
        return out

    def process_host_broadcast(self, x, out=None, wait: bool = True) -> np.ndarray:
        """x: [C][S] — one input signal for all instances of all shards."""
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1)
        if out is None:
            out = np.zeros((self.c, x.shape[1], self.n), dtype=np.float32)
        self._check(self.L.fx8010_multi_process_batch_host_broadcast(self.h, _ptr(x), _ptr(out), x.shape[1], 1 if wait else 0))
        self._keep_bcast = x
        return out

    def process_host_curves(self, x, curves, out=None, wait: bool = True, n_samples=None) -> np.ndarray:
        """fx8010_multi_process_batch_host_curves: x [C][S][N] over all instances (None: no input) -> out [C][S][N]; curves =
        [(reg_index, ndarray, broadcast)], each [S][N] float32, or [S] with broadcast.  wait=False queues the work; the arrays are
        kept until synchronize()."""
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.c, -1, self.n)
            n_samples = x.shape[1]
        if out is None:
            out = np.zeros((self.c, n_samples, self.n), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == self.c * n_samples * self.n
        arr, keep = _host_curves(curves, n_samples, self.n, 0)
        self._check(self.L.fx8010_multi_process_batch_host_curves(self.h, _ptr(x), _ptr(out), n_samples, C.addressof(arr), len(curves),
                                                                  1 if wait else 0))
        self._pending = [] if wait else getattr(self, "_pending", []) + [(x, out, arr, keep)]
        return out

    def synchronize(self):
        self._check(self.L.fx8010_multi_synchronize(self.h))
        self._pending = []

    def set_option(self, option: int, value: int):
        self._check(self.L.fx8010_multi_set_option(self.h, option, value))

    def registers(self) -> np.ndarray:
        out = np.zeros((self.n_regs, self.n), dtype=np.float32)
        self._check(self.L.fx8010_multi_get_registers(self.h, out.ctypes.data))
        return out

    def count_total(self) -> int:
        t = C.c_ulonglong(0)
        self._check(self.L.fx8010_multi_get_instruction_count(self.h, C.byref(t)))
        return int(t.value)

    def flags(self, clear: bool = False) -> int:
        f = C.c_uint(0)
        self._check(self.L.fx8010_multi_get_runtime_flags(self.h, C.byref(f), 1 if clear else 0))
        return int(f.value)


class MultiChain:
    """Several MultiGpu executors run one after another within every sample period (include/fx8010_multi.h, fx8010_multi_chain_*): one
    chain per shard, driven by the shard threads of the first executor.  It is closed before the executors: closing an executor closes the
    chains over it first."""

    def __init__(self, stages):
        self.L = gpu_lib()
        self.stages = list(stages)
        arr = (C.c_void_p * max(1, len(self.stages)))(*[m.h.value for m in self.stages])
        h = C.c_void_p()
        rc = self.L.fx8010_multi_chain_create(arr, len(self.stages), C.byref(h))
        if rc != 0:
            raise FxError(rc, self.L.fx8010_multi_chain_last_error(None).decode())
        self.h = h
        _register_chain(self, self.stages)

    def close(self):
        if getattr(self, "h", None):
            self.L.fx8010_multi_chain_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc):
        if rc != 0:
            raise FxError(rc, self.L.fx8010_multi_chain_last_error(self.h).decode())

    def process_host(self, x, n_samples=None, out=None, wait: bool = True) -> np.ndarray:
        """fx8010_multi_chain_process_batch_host: x [C][S][N] over all instances (None: no input) -> out [C][S][N].  wait=False queues
        the work; the arrays are kept until synchronize()."""
        return self.process_host_curves(x, [], n_samples=n_samples, out=out, wait=wait)

    def process_host_curves(self, x, curves, n_samples=None, out=None, wait: bool = True) -> np.ndarray:
        """fx8010_multi_chain_process_batch_host_curves: curves = [(stage, register index, ndarray, broadcast)], each [S][N] float32 over
        all instances, or [S] with broadcast."""
        m0 = self.stages[0]
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32).reshape(m0.c, -1, m0.n)
            n_samples = x.shape[1]
        out = _host_out(out, m0.c, n_samples, m0.n, 0)
        arr, keep = _chain_host_curves(curves, n_samples, m0.n, 0)
        self._check(self.L.fx8010_multi_chain_process_batch_host_curves(self.h, _ptr(x), _ptr(out), n_samples, C.addressof(arr), len(curves),
                                                                        1 if wait else 0))
        self._pending = [] if wait else getattr(self, "_pending", []) + [(x, out, arr, keep)]
        return out

    def synchronize(self):
        self._check(self.L.fx8010_multi_chain_synchronize(self.h))
        self._pending = []

    def shard_status(self, g: int) -> dict:
        """fx8010_chain_status of shard g's chain."""
        c = self.L.fx8010_multi_chain_shard(self.h, g)
        if not c:
            raise FxError(1, f"no shard {g}")
        return _chain_status(self.L, c)


def shard_range(n_total: int, rank: int, world: int):
    """Contiguous instance range of one rank (SURVEY.md §8e): [lo, hi)."""
    return (n_total * rank) // world, (n_total * (rank + 1)) // world


def pinned_array(shape, dtype=np.float32):
    """numpy array over page-locked memory from fx8010_gpu_host_alloc (keep the returned owner alive)."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = gpu_lib().fx8010_gpu_host_alloc(n)
    if not p:
        raise FxError(2, "fx8010_gpu_host_alloc failed")
    buf = (C.c_char * n).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)

    class _Owner:
        def __init__(self, ptr): self.ptr = ptr
        def __del__(self):
            try: gpu_lib().fx8010_gpu_host_free(self.ptr)
            except Exception: pass
    return arr, _Owner(p)
