/*
 * fx8010_host.h — C view of the host-side front-end and facade (libfx8010_host.so).
 *
 * The product's host language is C++ (class Klangraum::FX8010 in
 * fx8010-emulator-core_b200/host/FX8010.h mirrors reference include/FX8010.h:49-75).  These plain-C
 * entry points exist so that tests and bench.py can drive that class through ctypes; each one
 * forwards to the member named in its comment.  Compute entry points return a non-zero status and
 * leave a message in fx8010_host_last_error() when the GPU path fails — there is no CPU fallback.
 */
#ifndef FX8010_HOST_H
#define FX8010_HOST_H

#include "fx8010_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fx8010_host fx8010_host;

/* FX8010(int numChannels) / the batched constructor FX8010(channels, instances, device) */
FX8010_API fx8010_host* fx8010_host_create(int n_channels, int n_instances, int device);
/* FX8010(channels, instances, devices): the instances spread over several GPUs (include/fx8010_multi.h) */
FX8010_API fx8010_host* fx8010_host_create_multi(int n_channels, int n_instances, const int* devices, int n_devices);
FX8010_API void fx8010_host_destroy(fx8010_host* h);
FX8010_API const char* fx8010_host_last_error(fx8010_host* h);

/* loadFile (reference source/FX8010.cpp:777-875): 1 = loaded, 0 = open failure or syntax errors */
FX8010_API int fx8010_host_load_file(fx8010_host* h, const char* path);
FX8010_API int fx8010_host_load_text(fx8010_host* h, const char* text, size_t len);
FX8010_API int fx8010_host_ready(fx8010_host* h);                      /* getReadyStatus */
/* extension: relaxed syntax (accepts the reference README's `itramsize 100`, CR-LF files, blank lines after `end`) */
FX8010_API void fx8010_host_set_relaxed(fx8010_host* h, int on);
/* FX8010::setTranslation: the program translator's mode (FX8010_OPT_TRANSLATE of fx8010_gpu.h: 0, 1 or 2); 0 ok / 1 bad mode */
FX8010_API int fx8010_host_set_translation(fx8010_host* h, int mode);
/* FX8010::setKernelCacheDir: the translator's disk kernel cache, process-wide (fx8010_kernel_cache_set_dir of fx8010_gpu.h); NULL or "" = off */
FX8010_API void fx8010_host_set_kernel_cache_dir(const char* dir);

/* decoded image (what loadFile leaves in the object) */
FX8010_API int fx8010_host_num_registers(fx8010_host* h);
FX8010_API void fx8010_host_register_info(fx8010_host* h, int i, int* type, float* value, int* io_index, char* name, int cap);
FX8010_API int fx8010_host_num_instructions(fx8010_host* h);
FX8010_API void fx8010_host_instruction_info(fx8010_host* h, int i, int* fields /* opcode,R,A,X,Y,hasInput,hasOutput,hasNoise */);
FX8010_API int fx8010_host_itram_size(fx8010_host* h);
FX8010_API int fx8010_host_xtram_size(fx8010_host* h);
FX8010_API void fx8010_host_tables(fx8010_host* h, double* out /* [2][32][64]: LOG, EXP */);
FX8010_API const fx8010_program_image* fx8010_host_image(fx8010_host* h);

/* getErrorList / getControlRegisters / getMetaData */
FX8010_API int fx8010_host_num_errors(fx8010_host* h);
FX8010_API int fx8010_host_error_info(fx8010_host* h, int i, char* buf, int cap);   /* returns the row */
FX8010_API int fx8010_host_num_controls(fx8010_host* h);
FX8010_API void fx8010_host_control_name(fx8010_host* h, int i, char* buf, int cap);
FX8010_API int fx8010_host_metadata(fx8010_host* h, const char* key, char* buf, int cap);  /* 1 = present */

/* setRegisterValue / getRegisterValue (source/FX8010.cpp:236-266) and their per-instance forms */
FX8010_API int fx8010_host_set_register(fx8010_host* h, const char* name, float v);
FX8010_API float fx8010_host_get_register(fx8010_host* h, const char* name);
FX8010_API int fx8010_host_set_register_values(fx8010_host* h, const char* name, const float* values);
FX8010_API int fx8010_host_get_register_values(fx8010_host* h, const char* name, float* out);

/* process(): in/out [n_samples][channels], one process() call per sample (source/main.cpp:103-122) */
FX8010_API int fx8010_host_process(fx8010_host* h, const float* in, float* out, int n_samples);
/* processBlock(): host buffers [channel][sample][instance] */
FX8010_API int fx8010_host_process_block(fx8010_host* h, const float* in, float* out, int n_samples);
/* processBlockDeviceWithCurves(): DEVICE buffers, curve j drives register names[j] (d_values[j], broadcast[j]: see fx8010_gpu_process_batch_curves) */
FX8010_API int fx8010_host_process_block_device_curves(fx8010_host* h, const float* d_in, float* d_out, int n_samples, const char* const* names,
                                                       const float* const* d_values, const int* broadcast, int n_curves, void* stream);
/* processBlockWithCurves(): host buffers as in processBlock, curve j drives register names[j] (values[j]: HOST pointer, broadcast[j]: see
 * fx8010_gpu_process_batch_host_curves); on one device or several */
FX8010_API int fx8010_host_process_block_curves(fx8010_host* h, const float* in, float* out, int n_samples, const char* const* names,
                                                const float* const* values, const int* broadcast, int n_curves);
FX8010_API int fx8010_host_instruction_counter(fx8010_host* h);                 /* getInstructionCounter */
FX8010_API unsigned long long fx8010_host_instruction_counter_total(fx8010_host* h);
FX8010_API fx8010_gpu* fx8010_host_gpu(fx8010_host* h);

/* Klangraum::FX8010Chain: the programs of stages[n_stages] one after another within every sample period (fx8010_chain_* of fx8010_gpu.h,
 * fx8010_multi_chain_* of fx8010_multi.h for objects on several devices).  create returns NULL when the objects do not share one device, or
 * one device list of the multi-device constructor, and one channel and instance count (fx8010_host_chain_last_error(NULL) says why);
 * destroy the chain before its objects. */
typedef struct fx8010_host_chain fx8010_host_chain;
FX8010_API fx8010_host_chain* fx8010_host_chain_create(fx8010_host* const* stages, int n_stages);
FX8010_API void fx8010_host_chain_destroy(fx8010_host_chain* c);
/* processBlockDevice(): DEVICE buffers [channel][sample][instance], asynchronous on `stream` */
FX8010_API int fx8010_host_chain_process_block_device(fx8010_host_chain* c, const float* d_in, float* d_out, int n_samples, void* stream);
/* processBlockDeviceWithCurves(): curve j drives register names[j] of stage stages[j] (d_values[j], broadcast[j]: see
 * fx8010_chain_process_batch_curves) */
FX8010_API int fx8010_host_chain_process_block_device_curves(fx8010_host_chain* c, const float* d_in, float* d_out, int n_samples,
                                                             const int* stages, const char* const* names, const float* const* d_values,
                                                             const int* broadcast, int n_curves, void* stream);
/* processBlock(): HOST buffers [channel][sample][instance], on one device or several; returns when `out` is complete */
FX8010_API int fx8010_host_chain_process_block(fx8010_host_chain* c, const float* in, float* out, int n_samples);
/* processBlockWithCurves(): curve j drives register names[j] of stage stages[j] (values[j]: HOST pointer, broadcast[j]: see
 * fx8010_chain_process_batch_host_curves); on one device or several */
FX8010_API int fx8010_host_chain_process_block_curves(fx8010_host_chain* c, const float* in, float* out, int n_samples, const int* stages,
                                                      const char* const* names, const float* const* values, const int* broadcast, int n_curves);
FX8010_API const char* fx8010_host_chain_last_error(fx8010_host_chain* c);                          /* NULL on failure */

#ifdef __cplusplus
}
#endif
#endif
