/*
 * fx8010_gpu.h — C ABI of the B200-native batched FX8010 executor.
 *
 * This is the drop-in boundary for the reference's per-sample interpreter path.
 * The reference (easypx/FX8010-Emulator-Core) has no FFI of its own: its boundary is the
 * public section of class Klangraum::FX8010 (reference include/FX8010.h:49-75).  Each entry
 * point below names the reference member(s) it replaces.  One handle drives N independent
 * emulated DSP instances of ONE decoded program on ONE GPU.
 *
 * Conventions
 *   - plain C types only, no exceptions cross the boundary, every call returns an
 *     fx8010_status (0 = ok); fx8010_gpu_last_error() gives the text of the last failure.
 *   - sample blocks are float32, laid out [channel][sample][instance] (instance fastest):
 *       element (c, s, i) lives at  base[(c * n_samples + s) * n_instances + i].
 *     With n_instances == 1 this is the reference's per-sample vector repeated over time.
 *   - per-instance state blocks are laid out [register][instance].
 *   - calls on one handle are serialised by the caller; different handles (GPUs) may be
 *     driven from different host threads / processes.  Any number of handles may be live on
 *     a device.  Work queued on different streams by one handle is ordered on the device in
 *     call order (a stream switch inserts an event wait).
 *   - there is NO CPU fallback: every compute entry point fails with FX8010_ERR_CUDA when no
 *     CUDA device is usable.
 */
#ifndef FX8010_GPU_H
#define FX8010_GPU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define FX8010_API __attribute__((visibility("default")))
#else
#define FX8010_API
#endif

/* ---- enumerations shared with the reference's decoded image ------------------------- */

/* Opcode numbering = reference enum Opcode, include/FX8010.h:79-100. */
enum fx8010_opcode {
    FX_MACS = 0x0, FX_MACSN = 0x1, FX_MACW = 0x2, FX_MACWN = 0x3, FX_MACINTS = 0x4,
    FX_MACINTW = 0x5, FX_ACC3 = 0x6, FX_MACMV = 0x7, FX_ANDXOR = 0x8, FX_TSTNEG = 0x9,
    FX_LIMIT = 0xa, FX_LIMITN = 0xb, FX_LOG = 0xc, FX_EXP = 0xd, FX_INTERP = 0xe,
    FX_SKIP = 0xf, FX_IDELAY = 0x10, FX_XDELAY = 0x11, FX_END = 0x12,
    FX_NUM_OPCODES = 0x13
};

/* Register type numbering = reference enum RegisterType, include/FX8010.h:127-142. */
enum fx8010_regtype {
    FX_REG_STATIC = 0, FX_REG_TEMP, FX_REG_CONTROL, FX_REG_INPUT, FX_REG_OUTPUT, FX_REG_CONST,
    FX_REG_ITRAMSIZE, FX_REG_XTRAMSIZE, FX_REG_READ, FX_REG_WRITE, FX_REG_AT, FX_REG_CCR
};

enum fx8010_status {
    FX8010_OK = 0,
    FX8010_ERR_ARG = 1,          /* null pointer, bad size, index out of range             */
    FX8010_ERR_CUDA = 2,         /* no device / CUDA runtime failure (no CPU fallback)      */
    FX8010_ERR_NO_PROGRAM = 3,   /* process before load_program (reference: UB, SURVEY U10) */
    FX8010_ERR_PROGRAM = 4,      /* image rejected (bad index, IDELAY without itramsize…)   */
    FX8010_ERR_CAPACITY = 5      /* register file / TRAM does not fit the device            */
};

/* Sticky per-handle runtime flags, OR-ed over all instances (fx8010_gpu_get_runtime_flags). */
enum fx8010_runtime_flag {
    FX8010_RT_END_SKIPPED_CAP = 1, /* END skipped FX8010_MAX_PASSES times in one sample (SURVEY U9) */
    FX8010_RT_TABLE_RANGE = 2      /* LOG/EXP with |A|>1, NaN, or selector outside 0..31 (SURVEY U6) */
};

#define FX8010_MAX_PASSES        8      /* program re-runs per sample while END stays skipped     */
#define FX8010_MAX_INSTRUCTIONS  1000   /* decoded programs live in __constant__ memory (a 64 KiB arena shared by a device's handles) */
#define FX8010_TABLE_COUNT       32     /* reference source/FX8010.cpp:63                          */
#define FX8010_TABLE_ENTRIES     64     /* 32 mirrored + 32 generated, source/FX8010.cpp:73-105    */
#define FX8010_LFSR_SEED1        0x70f4f854u /* include/FX8010.h:290 */
#define FX8010_LFSR_SEED2        0xe1e9f0a7u /* include/FX8010.h:291 */

/* ---- decoded program image ------------------------------------------------------------ */

/* One decoded instruction; mirrors struct Instruction, include/FX8010.h:180-191. */
typedef struct fx8010_instr {
    int32_t opcode;              /* enum fx8010_opcode                                    */
    int32_t r, a, x, y;          /* GPR indices (operand1..4)                             */
    uint8_t has_input;           /* some of A/X/Y is an INPUT register                    */
    uint8_t has_output;          /* R is an OUTPUT register                               */
    uint8_t has_noise;           /* some non-INPUT one of A/X/Y is named "noise"          */
    uint8_t reserved;
} fx8010_instr;

/* One GPR record; mirrors struct GPR, include/FX8010.h:167-174 (name reduced to the one
 * property the execution path looks at: whether it is spelled "noise", FX8010.cpp:1065-1070). */
typedef struct fx8010_reg {
    int32_t type;                /* enum fx8010_regtype                                   */
    float   init_value;          /* declaration value or literal                          */
    int32_t io_index;            /* channel for INPUT/OUTPUT, else 0                      */
    int32_t is_noise;            /* registerName == "noise"                               */
} fx8010_reg;

/* What load_program consumes: the result of the reference's loadFile()/syntaxCheck()
 * (source/FX8010.cpp:777-875, 365-741) plus the host-built LOG/EXP tables
 * (source/FX8010.cpp:63-105) — the tables come from the host libm `pow` and are uploaded,
 * never recomputed on the device. */
typedef struct fx8010_program_image {
    const fx8010_instr* instrs;  int32_t n_instrs;
    const fx8010_reg*   regs;    int32_t n_regs;
    int32_t itram_size;          /* iTRAMSize, 0 = none declared                          */
    int32_t xtram_size;          /* xTRAMSize                                             */
    const double* log_tables;    /* [32][64] doubles                                      */
    const double* exp_tables;    /* [32][64] doubles                                      */
} fx8010_program_image;

typedef struct fx8010_gpu fx8010_gpu;

/* ---- lifecycle -------------------------------------------------------------------------- */

/* Replaces FX8010::FX8010(int numChannels) (include/FX8010.h:51, source/FX8010.cpp:9-12) for
 * n_instances objects at once.  device = CUDA ordinal. */
FX8010_API int fx8010_gpu_create(int device, int n_instances, int n_channels, fx8010_gpu** out);
FX8010_API void fx8010_gpu_destroy(fx8010_gpu* h);

/* Replaces the state that loadFile() leaves in the object (source/FX8010.cpp:777-875):
 * uploads the decoded program, (re)allocates and resets all per-instance state to what a
 * freshly constructed reference object holds (registers = init values, TRAM zero (SURVEY U2),
 * pointers 0, accumulator 0, LFSR seeds, output latch 0, counters 0). */
FX8010_API int fx8010_gpu_load_program(fx8010_gpu* h, const fx8010_program_image* image);

/* Options (fx8010_gpu_set_option).
 * FX8010_OPT_STREAM_EXCLUSIVE (default 0): the caller promises that between two fx8010_gpu_process_batch calls of this
 * handle on one stream nothing else is queued on that stream that launches kernels with programmatic completion
 * events (other handles of this library included).  Consecutive launches of a program without state across sample
 * periods may then overlap on the device (programmatic dependent launch with a postponed wait) whenever their buffers
 * are disjoint from those of every launch that can still be running.  Without the promise every launch waits for
 * its predecessor on the stream at its start.  The stage launches a chain queues (fx8010_chain_process_batch) never
 * postpone their wait, whatever the stages' options: each stage reads what the stage before it has just written.
 *
 * FX8010_OPT_TRANSLATE (default 1; env FX8010_TRANSLATE): programs that need the general interpreter (SKIP, noise, MACMV,
 * state carried between instructions) are translated into one straight-line sm_100a kernel with NVRTC — registers in
 * hardware registers, literals as immediates, SKIP as a forward branch — with results bit-identical to the interpreter's.
 * 0 = never; 1 = compile in a background thread when such a program first runs and switch to the kernel once it is
 * loaded (no call waits for the compiler; until then, and on a box without libnvrtc, the interpreter kernel runs);
 * 2 = compile before the first launch (the call waits).  fx8010_gpu_translate_status reports what happened. */
enum fx8010_option { FX8010_OPT_STREAM_EXCLUSIVE = 1, FX8010_OPT_TRANSLATE = 2 };
FX8010_API int fx8010_gpu_set_option(fx8010_gpu* h, int option, int value);

/* ---- controls: setRegisterValue / getRegisterValue (source/FX8010.cpp:236-266) ---------- */

/* values: host pointer; broadcast != 0 → values[0] goes to every instance, else values[N]. */
FX8010_API int fx8010_gpu_set_controls(fx8010_gpu* h, int reg_index, const float* values, int broadcast);
/* Same, values is a DEVICE pointer holding N floats (no host round trip). */
FX8010_API int fx8010_gpu_set_controls_device(fx8010_gpu* h, int reg_index, const float* d_values, void* stream);
/* out: host pointer to N floats. */
FX8010_API int fx8010_gpu_get_register(fx8010_gpu* h, int reg_index, float* out);

/* ---- the hot path: FX8010::process (source/FX8010.cpp:1023-1249) × n_samples × N -------- */

/* d_in / d_out: DEVICE pointers, [n_channels][n_samples][n_instances] float32.  Asynchronous
 * on `stream` (a cudaStream_t, NULL = default stream).  d_in may be NULL when the program has
 * no INPUT operand.
 * In place: d_out may equal d_in exactly (same pointer, same layout), and the call then gives the same outputs and the
 * same final state as with separate buffers.  That holds for every call of this header and of fx8010_multi.h that takes
 * an input and an output: process_batch, each block of process_blocks (d_out[b] == d_in[b]), process_batch_curves,
 * process_batch_host with its _async, _slice and _host_curves forms, the fx8010_multi_process_batch_* calls and
 * fx8010_chain_process_batch with its _curves form.  Any other overlap between an input and an output buffer is undefined. */
FX8010_API int fx8010_gpu_process_batch(fx8010_gpu* h, const float* d_in, float* d_out,
                                        int n_samples, void* stream);
/* n_blocks consecutive blocks of n_samples each in one call: block b reads d_in[b] and writes d_out[b] (arrays of
 * DEVICE pointers, each block laid out as above; d_in may be NULL, or all of its entries NULL, when the program has no
 * INPUT operand).  A d_in whose entries are neither all NULL nor all non-NULL is refused with FX8010_ERR_ARG before
 * anything is queued.  Equivalent to n_blocks fx8010_gpu_process_batch calls in order; a program without state across sample
 * periods runs up to 32 blocks per kernel launch, and the library knows that its own launches follow one another
 * on the stream (see FX8010_OPT_STREAM_EXCLUSIVE). */
FX8010_API int fx8010_gpu_process_blocks(fx8010_gpu* h, const float* const* d_in, float* const* d_out, int n_blocks,
                                         int n_samples, void* stream);
/* Same call with HOST buffers (pageable or pinned): host→device copy, kernels and
 * device→host copy are pipelined over sample sub-blocks on internal streams; returns when
 * `out` is complete. */
FX8010_API int fx8010_gpu_process_batch_host(fx8010_gpu* h, const float* in, float* out, int n_samples);
/* Same, but returns as soon as the work is queued: `in` must stay untouched and `out` unread until
 * fx8010_gpu_synchronize(h, NULL).  Consecutive calls chain in order on the handle's internal streams, so the
 * host->device copy of one block overlaps the device->host copy of the previous one (needs page-locked
 * buffers; with pageable memory the driver makes the copies synchronous anyway). */
FX8010_API int fx8010_gpu_process_batch_host_async(fx8010_gpu* h, const float* in, float* out, int n_samples);

/* Same for a handle whose instances are a SLICE of a wider host block: `in` / `out` point at this handle's first
 * instance inside host buffers laid out [channel][sample][host_instances] (host_instances >= n_instances); rows are
 * moved with strided copies.  wait == 0 queues the work like the _async form.  This is what the multi-GPU executor
 * (fx8010_multi.h) uses to gather every device's outputs into ONE host buffer. */
FX8010_API int fx8010_gpu_process_batch_host_slice(fx8010_gpu* h, const float* in, float* out, int n_samples,
                                                   size_t host_instances, int wait);

/* One input signal for ALL instances (a parameter sweep: N filter settings listening to the same audio, BASELINE.json
 * configs[3]): `in` is a HOST buffer [n_channels][n_samples] — 4 bytes per channel and sample period instead of 4 N — copied
 * as it is and spread over the instances on the device; `out` as in the _slice form ([channel][sample][host_instances],
 * host_instances == 0 means n_instances).  Halves the PCIe traffic of a step, which is what bounds the host-buffer path. */
FX8010_API int fx8010_gpu_process_batch_host_broadcast(fx8010_gpu* h, const float* in, float* out, int n_samples,
                                                       size_t host_instances, int wait);

/* ---- the caller's block loop (SURVEY.md §8f-2) -------------------------------------------
 * The reference's driver changes sliders BETWEEN process() calls, every 8 sample periods
 * (source/main.cpp:107-114: setRegisterValue, then process).  A batched caller would have to cut its
 * batches at every change; these entry points take the schedule instead. */

/* One control change inside a batch: register `reg_index` takes `values` right before sample period
 * `sample` of the batch (0 <= sample < n_samples).  values: HOST pointer; broadcast != 0 -> values[0]
 * goes to every instance, else values[N]. */
typedef struct fx8010_control_event {
    int32_t sample;
    int32_t reg_index;
    int32_t broadcast;
    int32_t reserved;
    const float* values;
} fx8010_control_event;

/* fx8010_gpu_process_batch with `n_events` control changes (sorted by `sample`, several may share one):
 * equivalent to set_controls + process_batch on every stretch between changes, queued on `stream` without a
 * host round trip in between (the value arrays are copied to the device before the first launch; they may be
 * reused when the call returns). */
FX8010_API int fx8010_gpu_process_batch_events(fx8010_gpu* h, const float* d_in, float* d_out, int n_samples,
                                               const fx8010_control_event* events, int n_events, void* stream);

/* Sample-accurate automation: one control value per sample period (fades, filter sweeps, a host's LFO) without cutting the batch. */
#define FX8010_MAX_CONTROL_CURVES 8
typedef struct fx8010_control_curve {
    int32_t reg_index;     /* a CONTROL or STATIC register                                                 */
    int32_t broadcast;     /* 0: d_values is [n_samples][n_instances]; != 0: [n_samples], one value for all */
    const float* d_values; /* DEVICE pointer, float32                                                      */
} fx8010_control_curve;
/* fx8010_gpu_process_batch with up to FX8010_MAX_CONTROL_CURVES registers following curves: equivalent, bit for bit in outputs and
 * in the final state, to `for s in 0..n_samples-1: set_controls(reg_j, curve_j[s]) for every j; process_batch(1 period)` — and to
 * process_batch_events with one event per curve at every period.  An automated register ends holding its last curve value, or what
 * the program itself wrote to it in the last period.  The curves are read on the device while the block runs (FX8010_OPT_TRANSLATE
 * != 0: inside the translated kernels, fx8010_launch_info.kernel_variant bit 4 set); without a translated kernel for the curve set
 * (mode 0, no libnvrtc, still compiling in mode 1, a SKIP count automated, unaligned buffers) the call runs one sample period per
 * launch: correct, but slow.  A curve buffer may be the output of earlier work on `stream` (another handle's output, say): the
 * call's first launch waits for everything before it.  FX8010_ERR_ARG, with nothing queued, for more than 8 curves or a negative
 * count, a NULL list or d_values, a register out of range, named twice, or neither CONTROL nor STATIC. */
FX8010_API int fx8010_gpu_process_batch_curves(fx8010_gpu* h, const float* d_in, float* d_out, int n_samples,
                                               const fx8010_control_curve* curves, int n_curves, void* stream);

/* The same automation for the host-buffer path: curve values in HOST memory (pageable or page-locked, float32). */
typedef struct fx8010_host_curve {
    int32_t reg_index;     /* a CONTROL or STATIC register                                                                       */
    int32_t broadcast;     /* 0: values is [n_samples][host_instances], this handle's first column at `values`;                  */
                           /* != 0: [n_samples], one value for every instance                                                    */
    const float* values;   /* HOST pointer                                                                                       */
} fx8010_host_curve;
/* fx8010_gpu_process_batch_host_slice with control curves: bit for bit, in outputs and in the whole final state, what
 * fx8010_gpu_process_batch_curves gives on device copies of the same buffers (the same definition: set_controls(reg_j, curve_j[s]) before
 * every period s).  `in`, `out` and host_instances (0 = n_instances) mean what they mean in the _slice form.  Each sub-block of the
 * pipeline copies its rows of every curve host->device together with its inputs and runs the curve kernels on them, so a per-instance
 * curve adds 4 * n_instances bytes per period to the PCIe traffic (a broadcast one 4 bytes) and shortens the sub-blocks to keep about
 * 16 MiB of staging per buffer set.  wait == 0 queues the work like the _async form: `in`, `out` and every `values` array must then stay
 * untouched until fx8010_gpu_synchronize(h, NULL).  FX8010_ERR_ARG, with nothing queued, for the lists fx8010_gpu_process_batch_curves
 * refuses and for host_instances below n_instances.  With n_curves == 0 it is fx8010_gpu_process_batch_host_slice. */
FX8010_API int fx8010_gpu_process_batch_host_curves(fx8010_gpu* h, const float* in, float* out, int n_samples,
                                                    const fx8010_host_curve* curves, int n_curves, size_t host_instances, int wait);

/* fx8010_gpu_process_batch for PLANAR audio buffers, as an audio host keeps them: DEVICE pointers,
 * [n_channels][n_instances][n_samples] float32 (one contiguous block of samples per instance and channel).
 * The [sample][instance] layout the interpreter streams is produced and undone by tiled transposes on `stream`. */
FX8010_API int fx8010_gpu_process_batch_planar(fx8010_gpu* h, const float* d_in, float* d_out, int n_samples, void* stream);

/* Page-locked host memory for process_batch_host buffers: with these the host<->device copies run
 * asynchronously at full PCIe rate (pageable buffers work too, through the driver's staging). */
FX8010_API void* fx8010_gpu_host_alloc(size_t bytes);
FX8010_API void fx8010_gpu_host_free(void* p);

/* Blocks until all work queued on the handle's internal streams and `stream` is done. */
FX8010_API int fx8010_gpu_synchronize(fx8010_gpu* h, void* stream);

/* ---- state access (parity tests, checkpoint/resume) ------------------------------------- */

/* Sum over instances of executed instructions (FX8010::getInstructionCounter,
 * source/FX8010.cpp:986-989; counted per executed instruction incl. END, :1222). */
FX8010_API int fx8010_gpu_get_instruction_count(fx8010_gpu* h, unsigned long long* total);
/* Per-instance counters, out: host pointer to N uint64. */
FX8010_API int fx8010_gpu_get_instruction_counts(fx8010_gpu* h, unsigned long long* out);

typedef struct fx8010_state_dims {
    int32_t n_instances, n_channels, n_regs, n_instrs;
    int32_t itram_size, xtram_size;       /* ring sizes                                   */
    int32_t itram_alloc, xtram_alloc;     /* floats allocated per instance (>= size)      */
} fx8010_state_dims;
FX8010_API int fx8010_gpu_get_dims(fx8010_gpu* h, fx8010_state_dims* out);

/* Full register file, host pointer to [n_regs][N] floats. */
FX8010_API int fx8010_gpu_get_registers(fx8010_gpu* h, float* out);
FX8010_API int fx8010_gpu_set_registers(fx8010_gpu* h, const float* in);
/* Per-instance scalars; any pointer may be NULL.  acc: double[N] (include/FX8010.h:162);
 * lfsr: uint32[2][N] (g_x1, g_x2, include/FX8010.h:290-291); out_latch: float[C][N]
 * (outputBuffer, include/FX8010.h:164); tram_ptrs: int32[4][N] in the order iTRAM write,
 * iTRAM read, xTRAM write, xTRAM read (include/FX8010.h:214-217). */
FX8010_API int fx8010_gpu_get_scalars(fx8010_gpu* h, double* acc, uint32_t* lfsr, float* out_latch, int32_t* tram_ptrs);
FX8010_API int fx8010_gpu_set_scalars(fx8010_gpu* h, const double* acc, const uint32_t* lfsr, const float* out_latch, const int32_t* tram_ptrs);
/* Ring contents of one instance: which = 0 iTRAM / 1 xTRAM; out: host pointer to `size` floats
 * (ring positions 0..size-1). */
FX8010_API int fx8010_gpu_get_tram(fx8010_gpu* h, int which, int instance, float* out);
FX8010_API int fx8010_gpu_set_tram(fx8010_gpu* h, int which, int instance, const float* in);

/* OR of enum fx8010_runtime_flag since load_program; clear != 0 resets it. */
FX8010_API int fx8010_gpu_get_runtime_flags(fx8010_gpu* h, unsigned int* flags, int clear);

/* ---- diagnostics -------------------------------------------------------------------------- */

/* One record per program instruction and sample period for ONE instance: the GPU counterpart of the
 * reference's PRINT_REGISTERS dump (printRegisters, source/FX8010.cpp:970-984, called at :1225-1226
 * after each executed instruction).  Values are those in the register file right after the instruction. */
typedef struct fx8010_trace_entry {
    int32_t index;               /* instruction index in the program (END included)                      */
    int32_t executed;            /* 0 = skipped by a SKIP (values then show the untouched registers)       */
    float r, a, x, y;            /* R, A, X, Y register values                                             */
    float ccr;                   /* GPR 0                                                                  */
    int32_t opcode;              /* enum fx8010_opcode                                                     */
    double acc;                  /* accumulator                                                            */
} fx8010_trace_entry;
/* Runs n_samples sample periods exactly like fx8010_gpu_process_batch_host (state advances, `out` may be
 * NULL) and fills entries[n_samples][n_instrs] (host memory) for `instance`.  Debug path: one instance per
 * thread, every instruction fetched and recorded; when END is skipped and the program re-runs, the records
 * of the last pass remain. */
FX8010_API int fx8010_gpu_trace(fx8010_gpu* h, const float* in, float* out, int n_samples, int instance,
                                fx8010_trace_entry* entries);


/* Program translator (FX8010_OPT_TRANSLATE).  state: 0 not attempted yet, 1 compiling, 2 translated kernel in use,
 * -1 not translated (message says why: not eligible, no libnvrtc, compiler output).  regs_per_thread / local_bytes
 * describe the loaded kernel.  Any pointer may be NULL. */
FX8010_API int fx8010_gpu_translate_status(fx8010_gpu* h, int* state, int* regs_per_thread, int* local_bytes,
                                           char* message, size_t message_cap);
/* The same for the translation of the most recent control-curve set (fx8010_gpu_process_batch_curves): state 0 also before any curve
 * call; -1 with the reason (e.g. an automated SKIP count) when the calls run one launch per period.  kind: 0 serial kernel, 1 streaming
 * kernel, 2 streaming kernel cut along time, -1 none loaded. */
FX8010_API int fx8010_gpu_translate_status_curves(fx8010_gpu* h, int* state, int* regs_per_thread, int* local_bytes, int* kind,
                                                  char* message, size_t message_cap);
/* The CUDA source the translator generates for an image on n_instances instances (no device needed; a test and inspection aid — the generated
 * source also compiles as plain C++ with -DFXT_HOST_CHECK, which is how tests/test_translate.py checks it on the CPU).
 * Returns the source length (copied, truncated, into buf when given), -1 for a bad image, -2 when the program is not
 * eligible.  compile_check != 0 also runs NVRTC for sm_100a and stores the CUBIN size (or -1) in *cubin_bytes. */
FX8010_API long long fx8010_translate_source(const fx8010_program_image* image, int n_instances, int n_channels, char* buf, size_t cap,
                                             int compile_check, int* cubin_bytes);
/* Same for the translation fx8010_gpu_process_batch_curves uses for curves on registers regs[n_curves] (broadcast[j] != 0: one value
 * per period for all instances).  With n_curves == 0 it is fx8010_translate_source.  -1 also for a curve list the call would reject. */
FX8010_API long long fx8010_translate_source_curves(const fx8010_program_image* image, int n_instances, int n_channels, const int32_t* regs,
                                                    const int32_t* broadcast, int n_curves, char* buf, size_t cap, int compile_check, int* cubin_bytes);

/* ---- program chains ----------------------------------------------------------------------------------------------------
 * A chain runs the programs of several handles one after another within every sample period: output channel c of stage j is input
 * channel c of stage j + 1.  fx8010_chain_process_batch(c, d_in, d_out, n, stream) is, bit for bit in d_out and in every stage's whole
 * final state, process_batch(stage 0, d_in, t0); process_batch(stage 1, t0, t1); ...; process_batch(stage k-1, t(k-2), d_out).
 * When every stage is stateless, the instance count is a multiple of 4, both buffers are 16-byte aligned and stage 0's
 * FX8010_OPT_TRANSLATE is not 0, the chain runs as ONE translated kernel that keeps the intermediate samples in registers (mode 1
 * compiles it in the background — the calls until then run stage by stage —, mode 2 before the call).  Otherwise it runs stage by stage
 * through intermediate blocks the chain owns.  The fused launch is booked in fx8010_chain_status, not in the stages' launch info; it
 * follows every stage's earlier work on any stream, and later work of any stage follows it.  Control curves on any stage's registers:
 * fx8010_chain_process_batch_curves.  Host buffers: fx8010_chain_process_batch_host(_curves); several GPUs: fx8010_multi_chain_* of
 * fx8010_multi.h. */
#define FX8010_MAX_CHAIN_STAGES 8
typedef struct fx8010_chain fx8010_chain;
/* stages[n_stages] (1..FX8010_MAX_CHAIN_STAGES distinct handles of one device, instance count and channel count; FX8010_ERR_ARG
 * otherwise).  Programs may be loaded or reloaded after creation: the chain looks at its stages at every call.  Destroy the chain
 * before any of its handles: fx8010_chain_destroy reads them (it waits for the work a host-buffer call left on stage 0's stream). */
FX8010_API int fx8010_chain_create(fx8010_gpu* const* stages, int n_stages, fx8010_chain** out);
FX8010_API void fx8010_chain_destroy(fx8010_chain* c);
/* d_in / d_out as in fx8010_gpu_process_batch (d_out may equal d_in).  Checks everything before it queues anything: FX8010_ERR_NO_PROGRAM when a stage has no
 * program, FX8010_ERR_ARG for a NULL d_out, a negative count, or a NULL d_in while stage 0 reads an input. */
FX8010_API int fx8010_chain_process_batch(fx8010_chain* c, const float* d_in, float* d_out, int n_samples, void* stream);
/* state: the fused kernel's translation state (values of fx8010_gpu_translate_status); fused_last: the last call ran it; launches: its
 * launches so far; regs_per_thread / local_bytes: the loaded kernel's; message: why the last call did not run fused ("" when it did).
 * state, regs_per_thread and local_bytes describe the kernel of fx8010_chain_process_batch; fused_last, launches and message the last chain
 * call of either kind (with or without curves).  Any pointer may be NULL. */
FX8010_API int fx8010_chain_status(fx8010_chain* c, int* state, int* fused_last, unsigned long long* launches, int* regs_per_thread,
                                   int* local_bytes, char* message, size_t message_cap);

/* Sample-accurate automation of a chain: control curves on registers of any of its stages, read inside the fused kernel. */
typedef struct fx8010_chain_curve {
    int32_t stage;          /* 0 .. n_stages-1                                              */
    int32_t reg_index;      /* a CONTROL or STATIC register of that stage's program         */
    int32_t broadcast;      /* 0: d_values is [n_samples][n_instances]; != 0: [n_samples]   */
    int32_t reserved;
    const float* d_values;  /* DEVICE pointer, float32                                      */
} fx8010_chain_curve;
/* fx8010_chain_process_batch with up to FX8010_MAX_CONTROL_CURVES curves in total, spread over the stages in any way.  Bit for bit in d_out
 * and in every stage's whole final state it is, stage after stage, fx8010_gpu_process_batch_curves(stage j, t(j-1), t(j), n_samples, the
 * curves of stage j) — fx8010_gpu_process_batch for a stage without curves: before stage j's period s each automated register of stage j
 * holds curve[s], and it ends holding its last curve value or what the stage's program wrote to it in the last period.  The chain runs fused
 * under the conditions of fx8010_chain_process_batch when, in addition, every per-instance curve is 16-byte aligned; the fused kernel loads
 * each period's curve values with the chain's inputs.  Otherwise it runs stage by stage, every stage with curves routing them as
 * fx8010_gpu_process_batch_curves does (fx8010_chain_status says why).  Everything is checked, for every stage, before anything is queued:
 * the rules of fx8010_chain_process_batch, and FX8010_ERR_ARG for a count outside 0..8, a NULL list with a count > 0, a NULL d_values, a
 * stage out of range, a register out of range for its stage, one (stage, register) named twice, or a register neither CONTROL nor STATIC.
 * d_out may equal d_in; a curve buffer that overlaps d_out is undefined.  A curve buffer may be the output of earlier work on `stream`.
 * With n_curves == 0 it is fx8010_chain_process_batch. */
FX8010_API int fx8010_chain_process_batch_curves(fx8010_chain* c, const float* d_in, float* d_out, int n_samples,
                                                 const fx8010_chain_curve* curves, int n_curves, void* stream);
/* The fused kernel of the most recent curve list (stage, register, broadcast) of fx8010_chain_process_batch_curves: its state (values of
 * fx8010_gpu_translate_status; 0 also before any curve call), registers and local memory, and why it is not in use ("" when it is). */
FX8010_API int fx8010_chain_status_curves(fx8010_chain* c, int* state, int* regs_per_thread, int* local_bytes, char* message,
                                          size_t message_cap);

/* A chain over HOST buffers (pageable or page-locked): bit for bit, in `out` and in every stage's whole final state, what
 * fx8010_chain_process_batch gives on device copies of the same buffers, and what the stages' own fx8010_gpu_process_batch_host calls
 * give one after another through host temporaries.  `in`, `out` and host_instances (0 = n_instances) mean what they mean in
 * fx8010_gpu_process_batch_host_slice: `in` may be NULL when stage 0 reads no input, and `out` may equal `in`.  The host pipeline of stage 0
 * (its internal streams, staging buffers and sub-block length, FX8010_TUNE_SUB included) moves the sub-blocks; each sub-block runs the
 * device chain call on its staging buffers, fused or stage by stage as that call decides (in mode 1 a compile that ends inside the call
 * switches the later sub-blocks to the fused kernel), so a chain of k stages moves its samples over PCIe once instead of k times.  Every stage's earlier work on any stream comes first, and every stage's later work (its state getters included) follows.
 * fx8010_chain_status afterwards: fused_last = 1 only when every sub-block ran fused, one launch counted per fused sub-block, and the
 * message of the first sub-block that did not.  wait == 0 queues the work: `in`, `out` (and every curve array of the _curves form) must
 * then stay untouched until fx8010_chain_synchronize; consecutive calls chain in order, and with page-locked buffers their copies overlap.
 * Checks everything before it queues anything: the rules of fx8010_chain_process_batch with `in` / `out` for d_in / d_out, and
 * FX8010_ERR_ARG for host_instances below n_instances. */
FX8010_API int fx8010_chain_process_batch_host(fx8010_chain* c, const float* in, float* out, int n_samples, size_t host_instances, int wait);
/* A control curve of a host-buffer chain call: fx8010_chain_curve with its values in HOST memory. */
typedef struct fx8010_chain_host_curve {
    int32_t stage;          /* 0 .. n_stages-1                                                                            */
    int32_t reg_index;      /* a CONTROL or STATIC register of that stage's program                                       */
    int32_t broadcast;      /* 0: values is [n_samples][host_instances] from the chain's first column; != 0: [n_samples]  */
    int32_t reserved;
    const float* values;    /* HOST pointer, float32                                                                      */
} fx8010_chain_host_curve;
/* fx8010_chain_process_batch_host with control curves: bit for bit what fx8010_chain_process_batch_curves gives on device copies.  Each
 * sub-block copies its rows of every curve with its inputs (a per-instance curve adds 4 * n_instances bytes per period, and every stage's
 * per-instance curves shorten the sub-blocks as in fx8010_gpu_process_batch_host_curves).  FX8010_ERR_ARG, with nothing queued, for the
 * lists fx8010_chain_process_batch_curves refuses and for host_instances below n_instances.  With n_curves == 0 it is
 * fx8010_chain_process_batch_host. */
FX8010_API int fx8010_chain_process_batch_host_curves(fx8010_chain* c, const float* in, float* out, int n_samples,
                                                      const fx8010_chain_host_curve* curves, int n_curves, size_t host_instances, int wait);
/* Blocks until all work queued on every stage's internal streams (and the streams of their latest work) is done. */
FX8010_API int fx8010_chain_synchronize(fx8010_chain* c);
/* NULL: the last error of fx8010_chain_create on this thread. */
FX8010_API const char* fx8010_chain_last_error(fx8010_chain* c);
/* The source of the fused kernel for images[n_stages] (as fx8010_translate_source; -2 when some stage is not stateless). */
FX8010_API long long fx8010_translate_source_chain(const fx8010_program_image* const* images, int n_stages, int n_instances, int n_channels,
                                                   char* buf, size_t cap, int compile_check, int* cubin_bytes);
/* The same with control curves q on register regs[q] of stage stage[q] (broadcast[q] as in fx8010_chain_curve).  With n_curves == 0 it is
 * fx8010_translate_source_chain.  -1 also for a curve list fx8010_chain_process_batch_curves refuses. */
FX8010_API long long fx8010_translate_source_chain_curves(const fx8010_program_image* const* images, int n_stages, int n_instances,
                                                          int n_channels, const int32_t* stage, const int32_t* regs, const int32_t* broadcast,
                                                          int n_curves, char* buf, size_t cap, int compile_check, int* cubin_bytes);

/* ---- kernel cache of the program translator ----------------------------------------------------------------------------
 * A translated kernel is named by SHA-256 over these bytes, concatenated: "fx8010-kernel-v1\n", "sm_100a\n", each NVRTC option
 * followed by "\n" ("--gpu-architecture=sm_100a", "--std=c++17", "--fmad=false", "--ftz=false", "--prec-div=true", "--prec-sqrt=true",
 * "-lineinfo", "-default-device", in this order), "nvrtc <major>.<minor>\n" (nvrtcVersion), then the generated source exactly as
 * fx8010_translate_source(_curves) returns it.  A handle looks its kernel up, at the first launch that can use it, in this order:
 *   1. the module already loaded on its device (another handle with the same program);
 *   2. the process-wide CUBIN store, or a compile of the same source already in flight, which it joins (one compile per process,
 *      whatever the number of handles and devices; in mode 1 the handle runs the interpreter kernels until that compile ends);
 *   3. the disk store, when a directory is set;
 *   4. NVRTC, then the process store and the disk store.
 * Steps 1-3 need no libnvrtc: a box without it runs kernels compiled elsewhere (it looks them up under every NVRTC version the
 * directory's file headers name; the headers are read again only when the directory changes).  A disk hit in mode 1 means the
 * first launch is already translated.  libnvrtc is looked up as "libnvrtc.so.12" and under /usr/local/cuda/lib64; FX8010_NVRTC
 * names the one library to load instead, and when that cannot be loaded the process has no NVRTC.
 *
 * The disk store is off unless FX8010_KERNEL_CACHE=<dir> (read when a handle is created or a precompile runs) or
 * fx8010_kernel_cache_set_dir names a directory.  One file per kernel, <dir>/fx8010-v1/<hex digest>.cubin: a 96-byte header
 * (magic "FX8010KC", format 1, NVRTC major and minor, the digest, the payload length, the SHA-256 of the payload), then the CUBIN.
 * Files are written to a unique temporary file and renamed into place, so concurrent processes never see a partial file.  A file
 * that fails validation, or whose CUBIN the driver refuses, is counted as rejected, recompiled and replaced; an I/O error never fails
 * a call (the kernel is used from memory and the failure counted).  Nothing is evicted: each file stands alone and may be deleted at
 * any time.  The NVRTC version is part of the key: a process that loads another libnvrtc (a Python package may bring its own, and
 * an already loaded one is what dlopen returns) compiles its own kernels, so precompile with the libnvrtc the application loads. */

/* Sets the disk store's directory for the whole process, overriding FX8010_KERNEL_CACHE; NULL or "" turns it off.  Always 0. */
FX8010_API int fx8010_kernel_cache_set_dir(const char* dir);
/* Compiles the kernel a handle would generate for `image` on n_instances instances (with control curves on regs[n_curves], as in
 * fx8010_translate_source_curves) and writes it to the disk store; needs libnvrtc, no device.  0 written, 1 a valid file was already
 * there, -1 bad arguments, -2 not eligible, -3 no cache directory, -4 compile failed, -5 write failed. */
FX8010_API int fx8010_kernel_cache_precompile(const fx8010_program_image* image, int n_instances, int n_channels, const int32_t* regs,
                                              const int32_t* broadcast, int n_curves);
/* Process-wide counters since the library was loaded. */
typedef struct fx8010_kernel_cache_stats {
    uint64_t nvrtc_compiles;       /* NVRTC compiles (fx8010_translate_source's compile_check included)          */
    uint64_t memory_hits;          /* kernels found loaded on the handle's device                                 */
    uint64_t store_hits;           /* CUBINs found in the process store                                           */
    uint64_t joined_compiles;      /* NVRTC compiles in flight joined instead of started                          */
    uint64_t disk_hits;            /* kernels loaded from the disk store                                          */
    uint64_t disk_writes;          /* files written                                                               */
    uint64_t disk_rejected;        /* files that failed validation or module load                                 */
    uint64_t disk_write_failures;  /* writes that failed (directory missing, not writable, disk full)              */
} fx8010_kernel_cache_stats;
FX8010_API int fx8010_kernel_cache_get_stats(fx8010_kernel_cache_stats* out);

/* Text of the last error on this handle (or of the last failed create when h == NULL). */
FX8010_API const char* fx8010_gpu_last_error(fx8010_gpu* h);

typedef struct fx8010_launch_info {
    unsigned long long kernel_launches;   /* kernels launched by this handle so far        */
    int32_t last_grid, last_block;        /* geometry of the last interpreter launch       */
    int32_t last_time_split;              /* sample segments per instance (1 = serial)     */
    int32_t last_smem_bytes;
    int32_t last_late_wait;               /* the last launch postponed its wait for its predecessor (see FX8010_OPT_STREAM_EXCLUSIVE) */
    int32_t last_fused_blocks;            /* sample blocks the last launch covered (fx8010_gpu_process_blocks) */
    int32_t last_tma;                     /* the last launch staged its input with bulk tensor copies (TMA) */
    int32_t reserved;
    int32_t kernel_variant;               /* bit0 SKIP, bit1 TRAM/noise/MACMV, bit2 stateless, bit3 instruction-major kernel, bit4 control curves read inside the kernel (fx8010_gpu_process_batch_curves), bit5 short-program kernel, bit6 producer/consumer pairs fused, bit7 translated kernel (FX8010_OPT_TRANSLATE), bits 8..15 instances per thread, bits 16.. samples per batch */
} fx8010_launch_info;
FX8010_API int fx8010_gpu_get_launch_info(fx8010_gpu* h, fx8010_launch_info* out);

#ifdef __cplusplus
}
#endif
#endif /* FX8010_GPU_H */
