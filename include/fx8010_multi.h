/*
 * fx8010_multi.h — one FX8010 program over N instances spread across several GPUs of one box.
 *
 * The reference's only remark on this axis is README.md:13 ("if we factor in the multi-core processing, we're able
 * to emulate much more DSP's"): instances are independent objects (include/FX8010.h:49-75 holds all state per object),
 * so they shard trivially.  This executor owns one fx8010_gpu handle (include/fx8010_gpu.h) per device, gives device g
 * the contiguous instance range [g * N / G, (g + 1) * N / G), replicates the program and its tables, and runs every
 * device from its own host thread on its own streams.  There is NO collective on the data path: inputs are scattered
 * and outputs gathered by per-device strided host<->device copies straight from / into ONE caller buffer laid out
 * [channel][sample][instance] over all N instances (page-locked memory from fx8010_gpu_host_alloc recommended).
 *
 * Same conventions as fx8010_gpu.h: plain C, status codes, no CPU fallback.  Calls on one executor are serialised by
 * the caller.
 */
#ifndef FX8010_MULTI_H
#define FX8010_MULTI_H

#include "fx8010_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fx8010_multi fx8010_multi;

/* Instance range of shard g of G over n_total instances (pure function, no device needed). */
FX8010_API void fx8010_multi_shard_range(int n_total, int g, int G, int* lo, int* hi);

/* devices: CUDA ordinals, one shard per entry (an ordinal may repeat: several shards on one GPU).  Replaces
 * n_instances FX8010 constructors (include/FX8010.h:51) spread over the devices. */
FX8010_API int fx8010_multi_create(const int* devices, int n_devices, int n_instances, int n_channels, fx8010_multi** out);
FX8010_API void fx8010_multi_destroy(fx8010_multi* m);
FX8010_API int fx8010_multi_num_shards(fx8010_multi* m);
/* The per-device handle of shard g and its instance range (for state access through fx8010_gpu.h). */
FX8010_API fx8010_gpu* fx8010_multi_shard(fx8010_multi* m, int g, int* lo, int* hi);

/* loadFile's result on every device (fx8010_gpu_load_program per shard, in parallel). */
FX8010_API int fx8010_multi_load_program(fx8010_multi* m, const fx8010_program_image* image);
/* setRegisterValue: values[N] split by the shard ranges, or values[0] to every instance when broadcast != 0. */
FX8010_API int fx8010_multi_set_controls(fx8010_multi* m, int reg_index, const float* values, int broadcast);
/* out: N floats, gathered from the shards. */
FX8010_API int fx8010_multi_get_register(fx8010_multi* m, int reg_index, float* out);

/* FX8010::process x n_samples x N (source/FX8010.cpp:1023-1249): in / out are HOST buffers
 * [n_channels][n_samples][n_instances]; every device moves and computes its own columns concurrently; returns when
 * `out` is complete.  `in` may be NULL when the program has no INPUT operand.  `out` may equal `in` (in place, as in
 * fx8010_gpu_process_batch, for every call below); any other overlap is undefined. */
FX8010_API int fx8010_multi_process_batch_host(fx8010_multi* m, const float* in, float* out, int n_samples);
/* Same, but returns once every device has QUEUED its work (consecutive calls pipeline copies and kernels per
 * device); fx8010_multi_synchronize waits for everything. */
FX8010_API int fx8010_multi_process_batch_host_async(fx8010_multi* m, const float* in, float* out, int n_samples);
/* One input signal for all instances: `in` is [n_channels][n_samples] (fx8010_gpu_process_batch_host_broadcast per shard). */
FX8010_API int fx8010_multi_process_batch_host_broadcast(fx8010_multi* m, const float* in, float* out, int n_samples, int wait);
/* Sample-accurate control curves from host memory (fx8010_gpu_process_batch_host_curves per shard): in / out as for
 * fx8010_multi_process_batch_host; a per-instance curve is [n_samples][n_instances] over ALL instances, and shard g reads its own
 * columns through a strided copy; a broadcast curve ([n_samples]) goes to every shard as it is.  The same curve list reaches every
 * shard, all with the same program, and each checks it before queuing: a refused list (FX8010_ERR_ARG) leaves every shard untouched.
 * wait == 0 queues the work: in, out and every values array stay untouched until fx8010_multi_synchronize. */
FX8010_API int fx8010_multi_process_batch_host_curves(fx8010_multi* m, const float* in, float* out, int n_samples,
                                                      const fx8010_host_curve* curves, int n_curves, int wait);
/* The curve list shard g of G (over n_total instances) passes to its handle: a per-instance curve's values moved to the shard's first
 * column (fx8010_multi_shard_range), a broadcast one as it is.  out: n_curves entries.  Pure function, no device needed. */
FX8010_API void fx8010_multi_shard_curves(const fx8010_host_curve* curves, int n_curves, int n_total, int g, int G, fx8010_host_curve* out);
FX8010_API int fx8010_multi_synchronize(fx8010_multi* m);
/* fx8010_gpu_set_option on every shard (FX8010_OPT_STREAM_EXCLUSIVE, FX8010_OPT_TRANSLATE). */
FX8010_API int fx8010_multi_set_option(fx8010_multi* m, int option, int value);

/* Executed instructions summed over all instances (getInstructionCounter, source/FX8010.cpp:986-989). */
FX8010_API int fx8010_multi_get_instruction_count(fx8010_multi* m, unsigned long long* total);
/* Full register file [n_regs][N], gathered. */
FX8010_API int fx8010_multi_get_registers(fx8010_multi* m, float* out);
/* OR of the shards' runtime flags (fx8010_gpu_get_runtime_flags). */
FX8010_API int fx8010_multi_get_runtime_flags(fx8010_multi* m, unsigned int* flags, int clear);

FX8010_API const char* fx8010_multi_last_error(fx8010_multi* m);

/* ---- program chains across GPUs -------------------------------------------------------------------------------------------
 * Executors run one after another within every sample period (fx8010_chain_* of fx8010_gpu.h, shard by shard): shard g's chain is
 * fx8010_chain_create over the stages' shard-g handles, and a call runs fx8010_chain_process_batch_host(_curves) on every shard's own
 * columns of the one caller buffer, from the shard threads of stage 0's executor. */
typedef struct fx8010_multi_chain fx8010_multi_chain;
/* stages[n_stages]: 1..FX8010_MAX_CHAIN_STAGES distinct executors with the same shard count, the same ordinal per shard and equal instance
 * and channel counts (so their shard ranges match); FX8010_ERR_ARG otherwise, and fx8010_multi_chain_last_error(NULL) says why.  Calls on
 * a multi chain and on its executors are serialised by the caller; destroy the multi chain before its executors. */
FX8010_API int fx8010_multi_chain_create(fx8010_multi* const* stages, int n_stages, fx8010_multi_chain** out);
FX8010_API void fx8010_multi_chain_destroy(fx8010_multi_chain* mc);
/* in / out as in fx8010_multi_process_batch_host (out may equal in); wait == 0 queues the work: in and out stay untouched until
 * fx8010_multi_chain_synchronize. */
FX8010_API int fx8010_multi_chain_process_batch_host(fx8010_multi_chain* mc, const float* in, float* out, int n_samples, int wait);
/* With control curves: a per-instance curve is [n_samples][n_instances] over ALL instances, and shard g reads its own columns; a broadcast
 * one ([n_samples]) reaches every shard as it is.  Every shard checks the list before it queues anything, so a refused list
 * (FX8010_ERR_ARG) leaves every shard untouched.  wait == 0: every values array also stays untouched until the synchronize. */
FX8010_API int fx8010_multi_chain_process_batch_host_curves(fx8010_multi_chain* mc, const float* in, float* out, int n_samples,
                                                            const fx8010_chain_host_curve* curves, int n_curves, int wait);
FX8010_API int fx8010_multi_chain_synchronize(fx8010_multi_chain* mc);
/* Shard g's chain (for fx8010_chain_status), NULL for g out of range. */
FX8010_API fx8010_chain* fx8010_multi_chain_shard(fx8010_multi_chain* mc, int g);
/* NULL: the last error of fx8010_multi_chain_create on this thread. */
FX8010_API const char* fx8010_multi_chain_last_error(fx8010_multi_chain* mc);
/* The curve list shard g of G (over n_total instances) passes to its chain: a per-instance curve's values moved to the shard's first column
 * (fx8010_multi_shard_range), a broadcast one and a NULL pointer as they are; stage and reg_index kept.  out: n_curves entries.  Pure
 * function, no device needed. */
FX8010_API void fx8010_multi_shard_chain_curves(const fx8010_chain_host_curve* curves, int n_curves, int n_total, int g, int G,
                                                fx8010_chain_host_curve* out);

#ifdef __cplusplus
}
#endif
#endif /* FX8010_MULTI_H */
