// fx8010_gpu.cu — the C ABI of include/fx8010_gpu.h: handle, program analysis + encoding, device
// state, kernel launches and the pipelined host-buffer path.  There is NO CPU fallback in this
// file: every compute entry point needs a CUDA device and fails with FX8010_ERR_CUDA otherwise.
//
// What the reference does per object and per sample (reference source/FX8010.cpp:1023-1249,
// one FX8010 object = one DSP instance) happens here per handle and per block of samples for
// N instances at once.
#include <cuda.h>            // CUtensorMap and its enums only: cuTensorMapEncodeTiled is resolved at run time (no libcuda link)
#include <cuda_runtime.h>

#include <dirent.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <regex>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "fx8010_families.h"

using namespace fxk;

namespace fxk {
SLKernelFn sl_kernel(int K, bool tram) { return K == 4 ? sl_kernel_4(tram) : (K == 2 ? sl_kernel_2(tram) : sl_kernel_1(tram)); }
cudaError_t upload_program(Family f, const uint4* src, size_t bytes, int word_off, cudaStream_t st) {
    switch (f) {
    case FAM_GENERIC: return upload_generic(src, bytes, word_off, st);
    case FAM_SHORT: return upload_short(src, bytes, word_off, st);
    case FAM_SL1: return upload_sl1(src, bytes, word_off, st);
    case FAM_SL2: return upload_sl2(src, bytes, word_off, st);
    default: return upload_sl4(src, bytes, word_off, st);
    }
}
}  // namespace fxk

namespace {

constexpr int MAX_DEVICES = 64;
constexpr int HOST_PIPE_BUFS = 3;
constexpr int MAX_CHAIN = 16;            // late-waiting launches that may follow one another before a launch waits at its start again
thread_local std::string g_create_error;

// Constant-memory residency: the decoded programs of a device's handles share one arena per kernel family
// (c_prog, fx8010_kernel.cuh).  A handle's range is allocated first-fit when it is about to launch; when the arena
// is full the least recently launched programs are evicted (after a device synchronise: their kernels may still
// be reading them) and simply uploaded again by their owner's next launch.  g_dev_mutex[device] is held from the
// residency check to the kernel launch, so a program cannot lose its range between the two.
struct ArenaBlock { int off, words; fx8010_gpu* owner; unsigned long long stamp; };
std::mutex g_dev_mutex[MAX_DEVICES];
std::vector<ArenaBlock> g_arena[MAX_DEVICES][FAM_COUNT];
unsigned long long g_arena_stamp[MAX_DEVICES];

struct Launch { int K, B, n_seg, seg_len, grid_x; size_t smem; int M; int chunk; int P; };   // M > 0: instruction-major kernel, samples per batch; P: threads sharing one instance column (they split each batch's samples), blockDim = B * P
struct PlanKey { int ns = -1; unsigned align = 0; int deep = -1; int n_blk = -1; int wave = -1; };   // deep: the TRAM delays are known to allow 64-sample batches; n_blk: sample blocks per launch; wave: planned for overlap with the neighbouring launches
enum RowClass { ROW_NONE = 0, ROW_RO, ROW_WO, ROW_RW, ROW_IN, ROW_TR };

typedef std::array<uint8_t, 32> KernelDigest;    // SHA-256 identity of a translated kernel (fx8010_translate.inc)

// One translation of the handle's program (fx8010_translate.inc): the plain one, or the one for a set of control curves.
struct Translation {
    int state = 0;                               // 0 not looked at, 1 compiling, 2 kernel loaded, -1 not eligible / failed (error says why)
    void* fn = nullptr;                          // CUfunction of the translated kernel
    KernelDigest key{}; bool attached = false;   // its entry in the per-process kernel cache (reference-counted)
    int regs = 0, local = 0;                     // its registers per thread / local-memory bytes (spills)
    int kind = 0;                                // 0 serial kernel, 1 streaming kernel (stateless program), 2 streaming kernel with TRAM (time-cut delay line),
                                                 // 3 streaming kernel of a program chain (fx8010_chain)
    int lanes = 1;                               // (serial kernel) instances per thread
    int ring_floats = 0;                         // (serial kernel) floats of the shared-memory input ring per thread
    std::shared_ptr<void> job;                   // the running compilation
    std::string error;
    std::vector<uint8_t> folded;                 // per register: its value is an immediate of the translated kernel ...
    std::vector<float> fold_value;               // ... namely this one
    std::vector<int> cv_reg;                     // control curves the kernel reads (registers; empty = the plain translation) ...
    std::vector<uint8_t> cv_bcast;               // ... and whether each is one value per period for all instances
    bool serial = false;                         // ... and a launch of it did not fit the streaming kernel: it takes the serial kernel
};

// The curves of one call as the kernels take them (a by-value parameter of the automated translated kernels: FxtCurves there).
struct CurveBlock { const float* p[FX8010_MAX_CONTROL_CURVES]; int bcast[FX8010_MAX_CONTROL_CURVES]; };

// Curve q of a chain call (fx8010_chain_process_batch_curves): register `reg` of stage `stage`; the list keys the chain's curve kernel.
struct ChainCurve {
    int stage, reg; uint8_t bcast;
    bool operator==(const ChainCurve& o) const { return stage == o.stage && reg == o.reg && bcast == o.bcast; }
};

}  // namespace

struct fx8010_gpu {
    int device = 0, N = 0, C = 0;
    int num_sms = 148;
    size_t smem_optin = 227 * 1024;
    bool loaded = false;
    int arena_family = -1, arena_off = -1, arena_words = 0;   // this handle's range of the family's constant-memory arena (-1: not resident)
    // program image (host copies)
    std::vector<fx8010_instr> instrs;
    std::vector<fx8010_reg> regs;
    int itram_size = 0, xtram_size = 0;          // ring sizes actually allocated (0 = unused)
    std::vector<TableEntry> h_tabs;
    // analysis
    std::vector<uint8_t> written;                // program may write the register
    std::vector<uint8_t> reg_uniform;            // every instance holds reg_value (host knowledge)
    std::vector<float> reg_value;
    std::vector<uint32_t> wb;                    // shared-memory rows to write back
    std::vector<uint32_t> reg_map;               // row -> register index
    std::vector<uint32_t> load_rows;             // rows loaded from the state arrays at kernel start
    bool load_latch = true, load_acc = true;
    std::vector<int> row_of;                     // register index -> row (-1: the program never refers to it)
    bool has_skip = false, has_ext = false, stateless = false;
    bool nop_out = false;                        // an IDELAY/XDELAY no-op whose R is an OUTPUT register (it still refreshes the latch)
    bool encode_dirty = true;
    int n_smem_tabs = 0;
    int smem_tab_id[MAX_SMEM_TABLES] = {0, 0};
    std::vector<int> tab_of;                     // per instruction: literal table id or -1
    uint4* h_prog = nullptr;                     // pinned, SLOT_WORDS words
    int enc_K = 0, enc_B = 0, enc_chunk = 0;     // geometry the uploaded encoding was made for
    std::vector<uint8_t> enc_sensitive;          // per register: its value / uniformity is folded into the encoding (LOG/EXP selector, SKIP count)
    cudaEvent_t ev_events = nullptr;
    float* d_events = nullptr; size_t events_floats = 0;      // device copies of per-instance control-event values
    float* d_planar_in = nullptr; float* d_planar_out = nullptr; size_t planar_floats = 0;   // [C][S][N] scratch of process_batch_planar
    int enc_family = -1;                         // kernel family whose constant memory holds it
    PlanKey plan_key; Launch plan = {};          // last launch plan (reused while nothing relevant changes)
    std::vector<const void*> smem_optin_fns;     // kernels this handle let use the opt-in shared-memory limit (smem_optin_for)
    // Programmatic dependent launch: the buffers read / written by every launch since (and including) the last one
    // that waited for its predecessor at its START.  A launch that postpones its wait can still be running next to
    // any of them, so a new launch may postpone its own wait only if it is disjoint from the whole chain.
    struct Span { const char* out_lo; const char* out_hi; const char* in_lo; const char* in_hi; };
    std::vector<Span> chain;
    cudaStream_t chain_stream = nullptr;
    int use_pdl = 1;
    int stream_exclusive = 0;                    // FX8010_OPT_STREAM_EXCLUSIVE: between this handle's launches nothing else runs on the caller's stream
    cudaEvent_t ev_order = nullptr;              // orders a launch after this handle's earlier work on a DIFFERENT stream
    bool trace_mode = false;                     // fx8010_gpu_trace in progress: debug geometry and encoding
    fx8010_trace_entry* d_trace = nullptr; int trace_inst = 0;
    // stateless fast path (fx8010_stateless.cuh)
    bool in_alias = false;                       // every INPUT-typed operand is preloaded by its own instruction
    bool sl_ok = false;                          // program qualifies
    // TRAM read streams of the instruction-major kernel: the one IDELAY/XDELAY READ of a TRAM, prefetched like an input
    struct TramStream { int isx, reg, yreg, w_yreg, w_first; } sl_tr[2];
    int sl_n_tr = 0;
    bool sl_tram = false;                        // the program has TRAM instructions (pointers are loaded and kept)
    int use_tram_im = 1;
    unsigned long long tram_periods = 0;         // sample periods launched since load_program (a pristine delay line's pointers are this, modulo the ring size)
    bool tram_ptrs_pristine = true;              // TRAM pointers as load_program left them (read and write pointer of a ring move in lockstep)
    bool sl_ccr_live = false;                    // the uploaded stateless encoding keeps per-sample CCR stores
    bool sl_serial = false;                      // ... with self-carried operands: one time segment, state loaded and kept
    bool acc_writer = false;                     // some instruction sets the accumulator
    std::vector<uint8_t> sl_carry;               // per instruction: bit o set = operand o (A, X, Y) is the instruction's own previous result
    std::vector<uint8_t> sl_carried_reg;         // per register: some instruction carries it from sample to sample
    std::vector<uint8_t> sl_fuse;                // per instruction: 0, or 0x80 | bits (fx8010_stateless.cuh F_FUSE) when the NEXT executed instruction is fused into it
    int use_pairs = 1, use_tsplit = 1;
    int use_tma = 1;                             // 0 never, 1 launches with one time segment (recurrences), 2 every eligible launch
    int use_carry = 1;
    bool short_ok = false;                       // SKIP-free, nobody reads ccr, no noise/MACMV, every channel written: fx_short_kernel when short enough
    int use_sl = 1, tune_M = 0, use_short = 1, tune_chunk = 0, use_fuse = 1;
    std::vector<int> sl_class, sl_index;         // per register: RowClass and index inside its class
    int sl_n_ro = 0, sl_n_wo = 0, sl_n_rw = 0;
    int sl_M = 0;                                // batch length of the uploaded encoding (0 = generic encoding uploaded)
    std::vector<uint2> sl_load, sl_wb;
    uint2* d_sl_load = nullptr; uint2* d_sl_wb = nullptr;
    int n_exec = 0;                              // encoded instructions
    int n_unpred = 0;                            // ... of which no SKIP can reach (general interpreter: counted per pass, not per instruction)
    std::vector<uint32_t> latch_ch;              // channels served from the latch every sample period
    // device state
    float* d_gpr = nullptr; double* d_acc = nullptr; uint32_t* d_lfsr = nullptr; float* d_latch = nullptr;
    int32_t* d_ptrs = nullptr; float* d_itram = nullptr; float* d_xtram = nullptr;
    unsigned long long* d_counts = nullptr; unsigned int* d_flags = nullptr; uint32_t* d_wb = nullptr; uint32_t* d_latch_ch = nullptr; uint32_t* d_reg_map = nullptr; uint32_t* d_load_rows = nullptr;
    TableEntry* d_tabs = nullptr;
    // streams
    cudaStream_t last_stream = nullptr;          // stream of the handle's latest device work (valid only while has_last)
    bool has_last = false;
    cudaStream_t s_h2d = nullptr, s_comp = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[HOST_PIPE_BUFS] = {}, ev_comp[HOST_PIPE_BUFS] = {}, ev_d2h[HOST_PIPE_BUFS] = {};
    float* d_stage_in[HOST_PIPE_BUFS] = {}; float* d_stage_out[HOST_PIPE_BUFS] = {};
    float* d_bcast[HOST_PIPE_BUFS] = {}; size_t bcast_floats = 0;     // [C][sub] staging of a broadcast input (process_batch_host_broadcast)
    size_t stage_floats = 0;
    float* d_curve_stage[HOST_PIPE_BUFS] = {}; size_t curve_floats = 0;   // host control curves: [sub][N] per per-instance curve, then [sub] per broadcast one
    unsigned long long pipe_seq = 0;             // sub-blocks pushed through the staging buffers so far
    // tuning overrides (0 = heuristic)
    int tune_K = 0, tune_B = 0, tune_seg = 0, tune_sub = 0, tune_P = 0, use_split = 1;
    // program translator (fx8010_translate.inc)
    int tr_recurrences = 0;                      // FX8010_TR_RECUR: self-recurrence programs of the instruction-major kernel take the translated serial kernel too
    int use_translate = 1;                       // FX8010_OPT_TRANSLATE: 0 never, 1 background compile + switch when ready, 2 compile before the first launch
    Translation tr;                              // the plain translation
    Translation tr_cv;                           // the translation for the most recent set of control curves (fx8010_gpu_process_batch_curves)
    mutable const Translation* tr_gen = nullptr; // the translation being generated: its curve registers are never folded (tr_generate_chain sets it per stage)
    std::vector<uint8_t> tr_volatile;            // per register: the host changed it after load — never folded again
    unsigned long long tr_epoch = 0;             // bumped whenever both translations are voided (load_program): chains over this handle regenerate
    std::string kc_env_dir;                      // FX8010_KERNEL_CACHE when the handle was created (the disk store; "" = none)
    std::string err;
    fx8010_launch_info info = {};
};

namespace {

int fail(fx8010_gpu* h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}
#define FX_CUDA(h, call)                                                                             \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            return fail(h, FX8010_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));    \
    } while (0)

int env_int(const char* name) { const char* s = getenv(name); return s ? atoi(s) : 0; }

// static_cast<int32_t>(float) with x86-64 semantics (same rule as the kernel's cvt_x86)
int32_t cvt_x86_host(float f) {
    if (!(f < 2147483648.0f) || f < -2147483648.0f) return INT32_MIN;
    return (int32_t)f;
}

Uop uop_of(const fx8010_gpu* h, const fx8010_instr& in) {
    switch (in.opcode) {
    case FX_MACS: case FX_MACINTS: return U_MACS;     // MACINTS == MACS in the reference (:1095-1103)
    case FX_MACSN: return U_MACSN;
    case FX_MACW: return U_MACW;
    case FX_MACWN: return U_MACWN;
    case FX_MACINTW: return U_MACINTW;
    case FX_ACC3: return U_ACC3;
    case FX_MACMV: return U_MACMV;
    case FX_ANDXOR: return U_ANDXOR;
    case FX_TSTNEG: return U_TSTNEG;
    case FX_LIMIT: return U_LIMIT;
    case FX_LIMITN: return U_LIMITN;
    case FX_LOG: return U_LOG;
    case FX_EXP: return U_EXP;
    case FX_INTERP: return U_INTERP;
    case FX_SKIP: return U_SKIP;
    case FX_IDELAY: {
        const int t = h->regs[in.r].type;
        return t == FX_REG_READ ? U_IREAD : (t == FX_REG_WRITE ? U_IWRITE : U_NOP);
    }
    case FX_XDELAY: {
        const int t = h->regs[in.r].type;
        return t == FX_REG_READ ? U_XREAD : (t == FX_REG_WRITE ? U_XWRITE : U_NOP);
    }
    case FX_END: return U_END;
    default: return U_NOP;
    }
}
bool writes_r(Uop u) { return u <= U_INTERP; }   // every one of these also runs setCCR

// Which operands of the instruction are preloaded from the input block / which register gets noise.
void pre_targets(const fx8010_gpu* h, const fx8010_instr& in, bool& pa, bool& px, bool& py, int& noise_reg) {
    pa = px = py = false; noise_reg = -1;
    if (in.has_input) {                                         // source/FX8010.cpp:1053-1061
        pa = h->regs[in.a].type == FX_REG_INPUT;
        px = h->regs[in.x].type == FX_REG_INPUT;
        py = h->regs[in.y].type == FX_REG_INPUT;
    }
    if (in.has_noise) {                                         // :1063-1071 (first match only)
        if (h->regs[in.a].is_noise) noise_reg = in.a;
        else if (h->regs[in.x].is_noise) noise_reg = in.x;
        else if (h->regs[in.y].is_noise) noise_reg = in.y;
    }
}

int encoded_length(const fx8010_gpu* h);

// Load-time analysis: written set, feature flags, statelessness (SURVEY.md §7 H2).
void analyse(fx8010_gpu* h) {
    const int n = (int)h->instrs.size(), nr = (int)h->regs.size();
    h->written.assign(nr, 0);
    h->has_skip = false; h->has_ext = false;
    bool any_ccr_writer = false;
    for (int i = 0; i < n; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        bool pa, px, py; int nz;
        pre_targets(h, in, pa, px, py, nz);
        if (pa) h->written[in.a] = 1;
        if (px) h->written[in.x] = 1;
        if (py) h->written[in.y] = 1;
        if (nz >= 0) { h->written[nz] = 1; h->has_ext = true; }
        if (writes_r(u)) { h->written[in.r] = 1; any_ccr_writer = true; }
        if (u == U_IREAD || u == U_XREAD) { h->written[in.a] = 1; h->has_ext = true; }
        if (u == U_IWRITE || u == U_XWRITE) h->has_ext = true;
        if (u == U_MACMV) h->has_ext = true;
        if (u == U_SKIP) h->has_skip = true;
    }
    if (any_ccr_writer) h->written[0] = 1;
    h->enc_sensitive.assign(nr, 0);
    for (int i = 0; i < n; ++i) {
        const Uop u = uop_of(h, h->instrs[i]);
        if (u == U_LOG || u == U_EXP) h->enc_sensitive[h->instrs[i].x] = 1;     // literal table selectors are resolved at encode time
        if (u == U_SKIP) h->enc_sensitive[h->instrs[i].y] = 1;                  // so is a constant skip count (CCR liveness)
    }
    // Only registers some instruction refers to (plus ccr) get a shared-memory row; the others
    // (unused declarations, the read/write/at pseudo registers) stay in the state arrays untouched.
    std::vector<uint8_t> used(nr, 0);
    used[0] = 1;
    h->nop_out = false;
    for (int i = 0; i < n; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        if (u == U_NOP && h->regs[in.r].type == FX_REG_OUTPUT) {  // IDELAY/XDELAY whose R is an OUTPUT register: no operation, but the
            used[in.r] = 1; h->nop_out = true;                    // output latch is still refreshed from R afterwards (:1229-1233)
        }
        if (u == U_END || u == U_NOP) continue;
        if (writes_r(u) || h->regs[in.r].type == FX_REG_OUTPUT) used[in.r] = 1;   // OUTPUT R feeds the latch after any op
        used[in.a] = used[in.x] = 1;
        if (u != U_LOG && u != U_EXP) used[in.y] = 1;            // LOG/EXP never read Y (the sign operand, :1114 TODO) ...
        bool pa, px, py; int nz;
        pre_targets(h, in, pa, px, py, nz);
        if (py) used[in.y] = 1;                                   // ... but an INPUT register there is still preloaded (:1059)
    }
    h->reg_map.clear(); h->row_of.assign(nr, -1); h->wb.clear();
    for (int r = 0; r < nr; ++r)
        if (used[r]) {
            h->row_of[r] = (int)h->reg_map.size();
            if (h->written[r]) h->wb.push_back((uint32_t)h->reg_map.size());
            h->reg_map.push_back((uint32_t)r);
        }

    // Stateless = no sample period reads anything an earlier period wrote: then the time axis can
    // be cut into independent segments.  Conservative: SKIP / TRAM / noise / MACMV rule it out.
    h->stateless = !h->has_skip && !h->has_ext && !h->nop_out;
    if (h->stateless) {
        std::vector<uint8_t> defined(nr, 0);
        for (int i = 0; i < n && h->stateless; ++i) {
            const fx8010_instr& in = h->instrs[i];
            const Uop u = uop_of(h, in);
            if (u == U_END || u == U_NOP) continue;
            bool pa, px, py; int nz;
            pre_targets(h, in, pa, px, py, nz);
            if (pa) defined[in.a] = 1;
            if (px) defined[in.x] = 1;
            if (py) defined[in.y] = 1;
            const int ops[3] = {in.a, in.x, in.y};
            for (int o : ops)
                if (h->written[o] && !defined[o]) h->stateless = false;
            if (writes_r(u)) { defined[in.r] = 1; defined[0] = 1; }
        }
    }
    // What the kernel has to fetch at start.  A stateless program overwrites every register it
    // writes before reading it, so only the rows it never writes carry information in; likewise the
    // latches when every channel has a writer, and the accumulator when some instruction sets it.
    h->load_rows.clear();
    bool acc_writer = false;
    std::vector<uint8_t> ch_written(h->C, 0);
    for (int i = 0; i < n; ++i) {
        const Uop u = uop_of(h, h->instrs[i]);
        if (writes_r(u) && u != U_MACMV && u != U_ANDXOR) acc_writer = true;
        if (writes_r(u) && h->regs[h->instrs[i].r].type == FX_REG_OUTPUT) ch_written[h->regs[h->instrs[i].r].io_index] = 1;
    }
    bool all_ch = true;
    for (int c = 0; c < h->C; ++c) all_ch = all_ch && ch_written[c];
    for (size_t row = 0; row < h->reg_map.size(); ++row)
        if (!h->stateless || !h->written[h->reg_map[row]]) h->load_rows.push_back((uint32_t)row);
    h->load_latch = !(h->stateless && all_ch);
    h->load_acc = !(h->stateless && acc_writer);
    h->acc_writer = acc_writer;

    // Stateless fast path: additionally every channel needs a writer (its latch is never read then) and
    // every preload of an INPUT register must deliver that register's own channel, so that the input
    // stage rows can stand in for the INPUT registers (the reference loads X and Y from A's channel,
    // source/FX8010.cpp:1057-1060 — a program relying on that quirk takes the generic kernel).
    h->in_alias = true;
    for (int i = 0; i < n; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        if (u == U_END || u == U_NOP) continue;
        bool pa, px, py; int nz;
        pre_targets(h, in, pa, px, py, nz);
        const int ops[3] = {in.a, in.x, in.y};
        const bool pre[3] = {pa, px, py};
        for (int o = 0; o < 3; ++o) if (h->regs[ops[o]].type == FX_REG_INPUT && !pre[o]) h->in_alias = false;   // hand-made image without has_input
        if (nz >= 0 && h->regs[nz].type == FX_REG_INPUT) h->in_alias = false;                                    // an INPUT register named "noise"
        if ((u == U_IREAD || u == U_XREAD) && h->regs[in.a].type == FX_REG_INPUT) h->in_alias = false;           // TRAM read into an INPUT register
    }
    // Short-program kernel (fx8010_short.cuh): SKIP-free, no noise, no MACMV, nobody reads `ccr` (it is produced on the
    // call's last sample only), every channel has a writer (no per-sample latch traffic), INPUT operands aliased.
    h->short_ok = !h->has_skip && h->in_alias && all_ch && !h->nop_out;
    for (int i = 0; i < n; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        if (u == U_END || u == U_NOP) continue;
        if (in.has_noise || u == U_MACMV) h->short_ok = false;
        if (in.a == 0 || in.x == 0 || in.y == 0 || (writes_r(u) && in.r == 0)) h->short_ok = false;
    }
    // The instruction-major kernel also takes programs whose only loop-carried values are SELF recurrences: an operand
    // that is the instruction's own result of the previous sample period (one-pole filters `interp out, out, c, in`,
    // accumulators `macs a, a, x, y`), the register having no other writer.  Running instruction i over a batch of
    // samples before instruction i + 1 keeps every such dependence (loop distribution); a value carried from a LATER
    // instruction to an earlier one would not survive it, and sends the program to the sample-major kernels.
    // TRAM programs qualify when each TRAM has at most one READ and one WRITE instruction (then both pointers advance
    // by one per sample and the distance between them is constant), their offsets come from registers the program never
    // writes, and the READ's target register has no other writer and is never read before the READ: the reads are then
    // prefetched a batch ahead, like an input channel, as long as the delay is longer than two batches (checked per
    // thread at kernel start; shorter delays run the same code one sample at a time).
    bool has_noise_or_macmv = false;
    int n_rd[2] = {0, 0}, n_wr[2] = {0, 0};
    h->sl_n_tr = 0; h->sl_tram = false;
    bool tram_ok = h->use_tram_im != 0;
    for (int i = 0; i < n; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        if (in.has_noise || u == U_MACMV) has_noise_or_macmv = true;
        const bool rd = (u == U_IREAD || u == U_XREAD), wr = (u == U_IWRITE || u == U_XWRITE);
        if (!rd && !wr) continue;
        h->sl_tram = true;
        const int t = (u == U_XREAD || u == U_XWRITE) ? 1 : 0;
        if (h->written[in.y]) tram_ok = false;
        if (rd) {
            if (n_rd[t]++ || h->regs[in.a].type == FX_REG_INPUT || in.a == 0) tram_ok = false;
            else {
                fx8010_gpu::TramStream& q = h->sl_tr[h->sl_n_tr++];
                q.isx = t; q.reg = in.a; q.yreg = in.y; q.w_yreg = -1; q.w_first = 0;
            }
        } else if (n_wr[t]++) tram_ok = false;
    }
    for (int i = 0; i < n && tram_ok; ++i) {               // the WRITE that shares a TRAM with each READ stream
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        if (u != U_IWRITE && u != U_XWRITE) continue;
        for (int q = 0; q < h->sl_n_tr; ++q)
            if (h->sl_tr[q].isx == (u == U_XWRITE ? 1 : 0)) {
                h->sl_tr[q].w_yreg = in.y;
                bool read_seen = false;
                for (int j = 0; j < i; ++j) { const Uop uj = uop_of(h, h->instrs[j]); if (uj == (u == U_XWRITE ? U_XREAD : U_IREAD)) read_seen = true; }
                h->sl_tr[q].w_first = read_seen ? 0 : 1;
            }
    }
    if (!tram_ok) { h->sl_n_tr = 0; }
    h->sl_ok = !h->has_skip && !has_noise_or_macmv && (!h->sl_tram || tram_ok) && all_ch && !h->nop_out;
    if (4 * (encoded_length(h) + 1) > SLOT_WORDS) h->sl_ok = false;     // four words per instruction in this kernel's encoding: longer programs take the general interpreter
    h->sl_serial = h->sl_tram;
    h->sl_carry.assign(n, 0); h->sl_carried_reg.assign(nr, 0);
    std::vector<int> n_writers(nr, 0);
    for (int i = 0; i < n; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        if (u == U_END || u == U_NOP) continue;
        bool pa, px, py; int nz;
        pre_targets(h, in, pa, px, py, nz);
        if (pa) n_writers[in.a]++;
        if (px && in.x != in.a) n_writers[in.x]++;
        if (py && in.y != in.a && in.y != in.x) n_writers[in.y]++;
        if (writes_r(u)) n_writers[in.r]++;
        if (u == U_IREAD || u == U_XREAD) n_writers[in.a]++;
    }
    std::vector<uint8_t> sl_defined(nr, 0);
    std::vector<uint8_t> is_read(nr, 0);
    for (int i = 0; i < n && h->sl_ok; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        if (u == U_END || u == U_NOP) continue;
        bool pa, px, py; int nz;
        pre_targets(h, in, pa, px, py, nz);
        if (pa) sl_defined[in.a] = 1;
        if (px) sl_defined[in.x] = 1;
        if (py) sl_defined[in.y] = 1;
        {
            const int opr[3] = {in.a, in.x, in.y};
            const bool tram_rd = (u == U_IREAD || u == U_XREAD);
            for (int o = 0; o < 3; ++o) {
                const int g = opr[o];
                if (tram_rd && o == 0) continue;                        // A of a TRAM READ is its target
                if (!h->written[g] || sl_defined[g]) continue;          // never written, or produced earlier in this period
                if (h->use_carry && g != 0 && writes_r(u) && in.r == g && n_writers[g] == 1 && h->regs[g].type != FX_REG_INPUT) {
                    h->sl_carry[i] |= (uint8_t)(1u << o); h->sl_carried_reg[g] = 1; h->sl_serial = true;
                } else h->sl_ok = false;
            }
            if (writes_r(u)) { sl_defined[in.r] = 1; sl_defined[0] = 1; }
            if (tram_rd) {
                if (n_writers[in.a] != 1) h->sl_ok = false;             // the stage rows stand in for the register: no other writer
                sl_defined[in.a] = 1;
            }
        }
        const int ch = h->regs[in.a].io_index;
        if ((pa && h->regs[in.a].io_index != ch) || (px && h->regs[in.x].io_index != ch) || (py && h->regs[in.y].io_index != ch)) h->sl_ok = false;
        // an INPUT-typed operand that is NOT preloaded here (has_input clear in a hand-made image) would read a stale row
        const int ops[3] = {in.a, in.x, in.y};
        const bool pre[3] = {pa, px, py};
        for (int o = 0; o < 3; ++o) if (h->regs[ops[o]].type == FX_REG_INPUT && !pre[o]) h->sl_ok = false;
        if (!(u == U_IREAD || u == U_XREAD)) is_read[in.a] = 1;
        is_read[in.x] = 1;
        if (u != U_LOG && u != U_EXP) is_read[in.y] = 1;
    }
    // Producer/consumer pairs: an instruction whose result has exactly ONE reader — the next executed instruction, a
    // MACS / MACSN (:1077-1094) whose other two operands hold one value for the whole batch — is run together with
    // it: the result is forwarded in a hardware register and never stored (the register keeps a single row that only
    // the final-state pass writes).  `log a, in, 3, 0` / `macs out, 0, a, volume` (cfg2) is the typical case.
    h->sl_fuse.assign(n, 0);
    std::vector<uint8_t> fused_away(nr, 0);
    if (h->sl_ok && h->use_pairs) {
        std::vector<int> n_reads(nr, 0);
        bool ccr_live = false;
        for (int i = 0; i < n; ++i) {
            const fx8010_instr& in = h->instrs[i];
            const Uop u = uop_of(h, in);
            if (u == U_END || u == U_NOP) continue;
            if (!(u == U_IREAD || u == U_XREAD)) n_reads[in.a]++;
            n_reads[in.x]++; n_reads[in.y]++;                   // (counted even where the value is ignored: conservative)
            if (writes_r(u) && in.r == 0) ccr_live = true;
        }
        if (n_reads[0]) ccr_live = true;                        // every setCCR is then materialised per sample: no pairs
        int prev = -1;
        for (int j = 0; j < n && !ccr_live; ++j) {
            const fx8010_instr& c = h->instrs[j];
            const Uop uc = uop_of(h, c);
            if (uc == U_END || uc == U_NOP) continue;
            const int i = prev;
            prev = j;
            if (i < 0 || h->sl_fuse[i]) continue;
            const fx8010_instr& pr = h->instrs[i];
            const Uop up = uop_of(h, pr);
            const bool tram_consumer = (uc == U_IWRITE || uc == U_XWRITE);      // `macs a, ...` / `idelay write, a, at, 0`: the result goes straight to the ring
            if (!writes_r(up) || up == U_MACMV || (uc != U_MACS && uc != U_MACSN && !tram_consumer)) continue;
            const int g = pr.r;
            if (g == 0 || h->regs[g].type == FX_REG_OUTPUT || h->regs[g].type == FX_REG_INPUT || n_writers[g] != 1 || n_reads[g] != 1) continue;
            if (h->sl_carry[i] || h->sl_carry[j] || h->sl_carried_reg[g]) continue;
            bool is_stream = false;
            for (int q = 0; q < h->sl_n_tr; ++q) if (h->sl_tr[q].reg == g) is_stream = true;
            if (is_stream) continue;
            const int pos = c.a == g ? 0 : (c.x == g ? 1 : (c.y == g ? 2 : -1));
            if (pos < 0 || (tram_consumer && pos != 0)) continue;
            const int others[2] = {pos == 0 ? c.x : c.a, pos == 2 ? c.x : c.y};
            bool constant = true;
            for (int o : others) constant = constant && !h->written[o] && h->regs[o].type != FX_REG_INPUT && h->row_of[o] >= 0;
            if (!constant || (writes_r(uc) && c.r == g)) continue;
            bool pre_a, pre_x, pre_y; int nz;
            pre_targets(h, c, pre_a, pre_x, pre_y, nz);
            if (pre_a || pre_x || pre_y || nz >= 0) continue;
            if (tram_consumer) h->sl_fuse[i] = (uint8_t)(0x80 | 8 | (uc == U_XWRITE ? 16 : 0));
            else h->sl_fuse[i] = (uint8_t)(0x80 | (pos != 0 ? 1 : 0) | (uc == U_MACSN ? 2 : 0) | (pos == 1 ? 4 : 0));
            fused_away[g] = 1;
            prev = -1;                                           // the consumer cannot start another pair
        }
    }
    h->sl_class.assign(nr, ROW_NONE); h->sl_index.assign(nr, 0);
    h->sl_n_ro = h->sl_n_wo = h->sl_n_rw = 0;
    if (h->sl_ok)
        for (int r = 0; r < nr; ++r) {
            if (h->row_of[r] < 0) continue;
            if (h->regs[r].type == FX_REG_INPUT) { h->sl_class[r] = ROW_IN; continue; }
            bool is_tr = false;
            for (int q = 0; q < h->sl_n_tr; ++q) if (h->sl_tr[q].reg == r) { h->sl_class[r] = ROW_TR; h->sl_index[r] = q; is_tr = true; }
            if (is_tr) continue;
            if (!h->written[r]) { h->sl_class[r] = ROW_RO; h->sl_index[r] = h->sl_n_ro++; }
            else if (!is_read[r] || fused_away[r]) { h->sl_class[r] = ROW_WO; h->sl_index[r] = h->sl_n_wo++; }   // (a forwarded result: one row, written by the final-state pass only)
            else { h->sl_class[r] = ROW_RW; h->sl_index[r] = h->sl_n_rw++; }
        }
}

size_t sl_smem_bytes(const fx8010_gpu* h, int B, int K, int M) {
    return (size_t)h->n_smem_tabs * TAB_SMEM_BYTES +
           (size_t)B * K * 4 * ((size_t)h->sl_n_ro + h->sl_n_wo + (size_t)h->sl_n_rw * M + 2 * (size_t)(h->C + h->sl_n_tr) * M);
}

// Operand word of register r for the stateless kernel (see fx8010_stateless.cuh).
uint32_t sl_word(const fx8010_gpu* h, int r, int B, int K, int M) {
    const uint32_t row_bytes = (uint32_t)B * K * 4u, stride16 = row_bytes >> 4;
    const uint32_t wo0 = (uint32_t)h->sl_n_ro * row_bytes, rw0 = wo0 + (uint32_t)h->sl_n_wo * row_bytes;
    const uint32_t st0 = rw0 + (uint32_t)h->sl_n_rw * M * row_bytes;
    switch (h->sl_class[r]) {
    case ROW_RO: return (uint32_t)h->sl_index[r] * row_bytes;
    case ROW_WO: return wo0 + (uint32_t)h->sl_index[r] * row_bytes;
    case ROW_RW: return (rw0 + (uint32_t)h->sl_index[r] * M * row_bytes) | (stride16 << SL_STRIDE_SHIFT);
    case ROW_IN: return (st0 + (uint32_t)h->regs[r].io_index * 2u * M * row_bytes) | (stride16 << SL_STRIDE_SHIFT) | SL_BUF;
    case ROW_TR: return (st0 + (uint32_t)(h->C + h->sl_index[r]) * 2u * M * row_bytes) | (stride16 << SL_STRIDE_SHIFT) | SL_BUF;   // TRAM read stream: stage rows after the input channels'
    default: return 0;   // never referenced
    }
}

void encode_stateless(fx8010_gpu* h, int K, int B, int M) {
    const int n = (int)h->instrs.size(), nr = (int)h->regs.size(), C = h->C;
    std::vector<int> last_writer(C, -1);
    bool ccr_read = h->sl_class[0] == ROW_RW;
    h->sl_ccr_live = false;
    for (int i = 0; i < n; ++i) {
        const Uop u = uop_of(h, h->instrs[i]);
        if (writes_r(u) && h->regs[h->instrs[i].r].type == FX_REG_OUTPUT) last_writer[h->regs[h->instrs[i].r].io_index] = i;
    }
    int e = 0;
    for (int i = 0; i < n; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const Uop u = uop_of(h, in);
        if (u == U_END || u == U_NOP) continue;
        uint32_t w0 = (uint32_t)u, aux = 0;
        if (h->sl_class[in.r] == ROW_WO) w0 |= F_ST_LAST;
        if (ccr_read || in.r == 0) { w0 |= F_CCR; h->sl_ccr_live = true; }                 // a `ccr` operand somewhere: every setCCR is kept per sample
        w0 |= (uint32_t)h->sl_carry[i] << SL_CARRY_SHIFT;       // operands that are this instruction's own previous result
        if (h->regs[in.r].type == FX_REG_OUTPUT) {
            const int c = h->regs[in.r].io_index;
            if (last_writer[c] == i) w0 |= F_OUT | F_OUT_DIRECT;
            w0 |= (uint32_t)c << 24;
        }
        if (h->tab_of[i] >= 0) {
            int slot = -1;
            for (int t = 0; t < h->n_smem_tabs; ++t) if (h->smem_tab_id[t] == h->tab_of[i]) slot = t;
            if (slot >= 0) { w0 |= F_TAB_SMEM; aux = (uint32_t)slot << 24; }
            else { w0 |= F_TAB_IMM; aux = (uint32_t)h->tab_of[i] << 24; }
        }
        if (h->sl_fuse[i]) w0 |= F_FUSE;
        // Four words per instruction, everything pre-computed (format: fx8010_stateless.cuh, sl_exec): offset at sample 0 and
        // bytes per sample of R, A, X, Y and CCR.  A self-carried operand (this instruction's own previous result) starts
        // at the register's row M - 1 and does not move; bit 31 of an offset marks a stage row (the buffer in use is added).
        const uint32_t wr = sl_word(h, in.r, B, K, M), wc = sl_word(h, 0, B, K, M);
        const uint32_t wo[3] = {sl_word(h, in.a, B, K, M), sl_word(h, in.x, B, K, M), sl_word(h, in.y, B, K, M)};
        uint32_t off[3], str[3];
        for (int o = 0; o < 3; ++o) {
            const bool carried = (h->sl_carry[i] >> o) & 1;
            str[o] = carried ? 0u : sl_stride(wo[o]);
            off[o] = carried ? (wo[o] & SL_OFF_MASK) + (uint32_t)(M - 1) * sl_stride(wo[o]) : ((wo[o] & SL_OFF_MASK) | (wo[o] & SL_BUF));
        }
        h->h_prog[4 * e] = make_uint4(w0, aux, (uint32_t)(h->sl_fuse[i] & 0x7f), 0);
        h->h_prog[4 * e + 1] = make_uint4(wr & SL_OFF_MASK, off[0], off[1], off[2]);
        h->h_prog[4 * e + 2] = make_uint4(sl_stride(wr), str[0], str[1], str[2]);
        h->h_prog[4 * e + 3] = make_uint4(wc & SL_OFF_MASK, sl_stride(wc), 0, 0);
        ++e;
    }
    h->n_exec = e;
    for (int j = 0; j < 4; ++j) h->h_prog[4 * e + j] = make_uint4(j == 0 ? (uint32_t)U_NOP : 0u, 0, 0, 0);   // pad record: the kernel prefetches pc + 1
    h->sl_load.clear(); h->sl_wb.clear();
    for (int r = 0; r < nr; ++r) {
        if (h->sl_class[r] == ROW_RO) h->sl_load.push_back(make_uint2(sl_word(h, r, B, K, M), (uint32_t)r));
        if (h->sl_carried_reg[r])        // carried in from the previous call: the row of "the sample before sample 0" is row M - 1
            h->sl_load.push_back(make_uint2((sl_word(h, r, B, K, M) & SL_OFF_MASK) + (uint32_t)(M - 1) * (uint32_t)B * K * 4u, (uint32_t)r));
        if (h->sl_class[r] != ROW_RO && h->sl_class[r] != ROW_NONE && h->written[r]) h->sl_wb.push_back(make_uint2(sl_word(h, r, B, K, M), (uint32_t)r));
    }
    h->enc_K = K; h->enc_B = B; h->sl_M = M;
}

// LOG/EXP with a literal selector (a register the program never writes and that holds one value in
// every instance): the table is known at encode time; the most frequent ones go to shared memory.
// Runs before launch planning because it decides the shared-memory footprint.
void select_tables(fx8010_gpu* h) {
    const int n = (int)h->instrs.size();
    auto is_const = [&](int r) { return !h->written[r] && h->reg_uniform[r]; };
    int freq[2 * FX8010_TABLE_COUNT] = {0};
    h->tab_of.assign(n, -1);
    for (int i = 0; i < n; ++i) {
        const Uop u = uop_of(h, h->instrs[i]);
        if (u != U_LOG && u != U_EXP) continue;
        const int xr = h->instrs[i].x;
        if (!is_const(xr)) continue;
        const int32_t sel = cvt_x86_host(h->reg_value[xr]);
        if (sel < 0 || sel >= FX8010_TABLE_COUNT) continue;      // out of range: dynamic path raises the flag
        h->tab_of[i] = (u == U_EXP ? FX8010_TABLE_COUNT : 0) + sel;
        freq[h->tab_of[i]]++;
    }
    h->n_smem_tabs = 0;
    for (int t = 0; t < MAX_SMEM_TABLES; ++t) {
        int best = -1;
        for (int id = 0; id < 2 * FX8010_TABLE_COUNT; ++id)
            if (freq[id] > 0 && (best < 0 || freq[id] > freq[best])) best = id;
        if (best < 0) break;
        h->smem_tab_id[h->n_smem_tabs++] = best;
        freq[best] = -1;
    }
}

// Encodes the program for the kernel: micro-ops, flags, CCR liveness, table placement.
void encode(fx8010_gpu* h, int K, int B, int chunk) {
    const int n = (int)h->instrs.size();
    const bool skipv = h->has_skip || h->trace_mode;   // trace mode keeps END/NOP and the latch path (SKIP-variant kernel)
    const int RS = K * B, nr = (int)h->reg_map.size(), C = h->C;
    auto row = [&](int r) { return h->row_of[r] < 0 ? 0 : h->row_of[r]; };   // unused operands (R of SKIP/TRAM ops) are never touched
    std::vector<Uop> uops(n);
    for (int i = 0; i < n; ++i) uops[i] = uop_of(h, h->instrs[i]);
    auto is_const = [&](int r) { return !h->written[r] && h->reg_uniform[r]; };

    // instructions a SKIP may jump over
    std::vector<uint8_t> maybe_skipped(n, 0);
    for (int k = 0; k < n; ++k) {
        if (uops[k] != U_SKIP) continue;
        long reach = n;
        const int yr = h->instrs[k].y;
        if (is_const(yr)) {
            const int32_t c = cvt_x86_host(h->reg_value[yr]);
            reach = c > 0 ? c : (c < 0 ? 1 : 0);
        }
        for (long d = 1; d <= std::min<long>(reach, n); ++d) maybe_skipped[(k + d) % n] = 1;
    }
    // CCR liveness: a setCCR result matters only if a SKIP or a `ccr` operand can see it before the
    // next unconditional setCCR (the batch-final value is forced by the kernel on the last sample).
    std::vector<uint8_t> ccr_live(n, 0);
    auto reads_ccr = [&](int j) {
        const Uop u = uops[j];
        if (u == U_END || u == U_NOP) return false;
        if (u == U_SKIP) return true;
        const fx8010_instr& in = h->instrs[j];
        return in.a == 0 || in.x == 0 || in.y == 0;
    };
    for (int i = 0; i < n; ++i) {
        if (!writes_r(uops[i])) continue;
        if (h->instrs[i].r == 0) { ccr_live[i] = 1; continue; }   // R is ccr itself: the store order matters
        bool live = true;                                         // nothing kills it within one lap: keep
        for (int d = 1; d <= n; ++d) {
            const int j = (i + d) % n;
            if (reads_ccr(j)) { live = true; break; }
            if (writes_r(uops[j]) && !maybe_skipped[j]) { live = false; break; }
        }
        ccr_live[i] = live;
    }

    // Accumulator liveness, same reasoning: only MACMV reads the accumulator (:1145), every other arithmetic
    // instruction except ANDXOR overwrites it (a value nobody overwrites within one lap survives to the end of the batch).
    std::vector<uint8_t> acc_live(n, 0);
    for (int i = 0; i < n; ++i) {
        if (!writes_r(uops[i]) || uops[i] == U_ANDXOR || uops[i] == U_MACMV) continue;
        bool live = true;
        for (int d = 1; d <= n; ++d) {
            const int j = (i + d) % n;
            if (uops[j] == U_MACMV) { live = true; break; }
            if (writes_r(uops[j]) && uops[j] != U_ANDXOR && !maybe_skipped[j]) { live = false; break; }
        }
        acc_live[i] = live;
    }

    // SKIP-free programs: the value a channel puts out is what its LAST writer in program order leaves
    // (earlier latch updates are dead), so that writer stores straight to the output block; channels
    // nobody writes — and every channel of a program with SKIP — are served from the latch.
    std::vector<int> last_writer(C, -1);
    std::vector<uint8_t> latch_served(C, 0);      // a no-op with an OUTPUT R refreshes the latch from the register: that channel keeps the latch path
    for (int i = 0; i < n; ++i)
        if (uops[i] == U_NOP && h->regs[h->instrs[i].r].type == FX_REG_OUTPUT) latch_served[h->regs[h->instrs[i].r].io_index] = 1;
    if (!skipv)
        for (int i = 0; i < n; ++i)
            if (h->regs[h->instrs[i].r].type == FX_REG_OUTPUT && writes_r(uops[i]) && !latch_served[h->regs[h->instrs[i].r].io_index])
                last_writer[h->regs[h->instrs[i].r].io_index] = i;
    h->latch_ch.clear();
    for (int c = 0; c < C; ++c) if (last_writer[c] < 0) h->latch_ch.push_back((uint32_t)c);

    int e = 0, n_unpred = 0;
    for (int i = 0; i < n; ++i) {
        const fx8010_instr& in = h->instrs[i];
        const bool nop_latch = uops[i] == U_NOP && h->regs[in.r].type == FX_REG_OUTPUT;
        if (!skipv && (uops[i] == U_END || uops[i] == U_NOP) && !nop_latch) continue;    // no-ops unless a SKIP counts them
        bool pa, px, py; int nz;
        pre_targets(h, in, pa, px, py, nz);
        uint32_t w0 = (uint32_t)uops[i];
        if (pa) w0 |= F_PRE_A;
        if (px) w0 |= F_PRE_X;
        if (py) w0 |= F_PRE_Y;
        uint32_t pre_off = 0, out_off = 0, aux = (uint32_t)(in.opcode & 0xff) << 24;   // bits 24..31: table slot/id, else the opcode (trace)
        if (pa || px || py) pre_off = stage_offset(nr, C, h->regs[in.a].io_index, RS, chunk);      // X and Y use A's IOIndex (:1057-1060)
        if (nz >= 0) { w0 |= F_NOISE; aux |= reg_offset(row(nz), RS); }
        if (h->regs[in.r].type == FX_REG_OUTPUT && uops[i] != U_END && (uops[i] != U_NOP || nop_latch)) { // :1229-1233
            const int c = h->regs[in.r].io_index;
            if (skipv || latch_served[c]) w0 |= F_OUT;
            else if (last_writer[c] == i) w0 |= F_OUT | F_OUT_DIRECT;
            w0 |= (uint32_t)c << 24;
            out_off = latch_offset(nr, c, RS);
        }
        if (ccr_live[i]) w0 |= F_CCR;
        if (acc_live[i] || h->trace_mode) w0 |= F_ACC;
        if (skipv && (maybe_skipped[i] || h->trace_mode)) w0 |= F_PRED;
        else ++n_unpred;
        if (h->tab_of[i] >= 0) {
            int slot = -1;
            for (int t = 0; t < h->n_smem_tabs; ++t) if (h->smem_tab_id[t] == h->tab_of[i]) slot = t;
            aux &= 0xffffffu;
            if (slot >= 0) { w0 |= F_TAB_SMEM; aux |= (uint32_t)slot << 24; }
            else { w0 |= F_TAB_IMM; aux |= (uint32_t)h->tab_of[i] << 24; }
        }
        h->h_prog[2 * e] = make_uint4(w0, reg_offset(row(in.r), RS), reg_offset(row(in.a), RS), reg_offset(row(in.x), RS));
        h->h_prog[2 * e + 1] = make_uint4(reg_offset(row(in.y), RS), aux, pre_off, out_off);
        ++e;
    }
    h->n_exec = e; h->n_unpred = n_unpred;
    h->h_prog[2 * e] = make_uint4((uint32_t)U_NOP, 0, 0, 0);      // pad: the kernel prefetches pc + 1
    h->h_prog[2 * e + 1] = make_uint4(0, 0, 0, 0);
    h->enc_K = K; h->enc_B = B; h->sl_M = 0; h->enc_chunk = chunk;
}

void free_state(fx8010_gpu* h) {
    cudaFree(h->d_gpr); cudaFree(h->d_acc); cudaFree(h->d_lfsr); cudaFree(h->d_latch); cudaFree(h->d_ptrs);
    cudaFree(h->d_itram); cudaFree(h->d_xtram); cudaFree(h->d_counts); cudaFree(h->d_wb); cudaFree(h->d_latch_ch); cudaFree(h->d_reg_map); cudaFree(h->d_load_rows); cudaFree(h->d_sl_load); cudaFree(h->d_sl_wb);
    h->d_gpr = nullptr; h->d_acc = nullptr; h->d_lfsr = nullptr; h->d_latch = nullptr; h->d_ptrs = nullptr;
    h->d_itram = nullptr; h->d_xtram = nullptr; h->d_counts = nullptr; h->d_wb = nullptr; h->d_latch_ch = nullptr; h->d_reg_map = nullptr; h->d_load_rows = nullptr; h->d_sl_load = nullptr; h->d_sl_wb = nullptr;
}

// Encoded length of the program for the generic kernel (END/NOP are dropped when there is no SKIP).
int encoded_length(const fx8010_gpu* h) {
    int e = 0;
    for (const fx8010_instr& in : h->instrs) {
        const Uop u = uop_of(h, in);
        if (!h->has_skip && (u == U_END || u == U_NOP)) continue;
        ++e;
    }
    return e;
}
// fx_short_kernel<K, EXT, NI>: NI = the exact number of executed instructions
bool use_short_kernel(const fx8010_gpu* h) {
    const int e = encoded_length(h);
    return h->use_short && h->short_ok && !h->trace_mode && e >= 1 && e <= SH_MAX_NI_HOST;
}

int tr_kind(const fx8010_gpu* h, const Translation& T);
constexpr int MIN_TSPLIT_SPAN = 64;      // shorter spans would mean too many tiny launches: the serial kernel (with its sample split) takes those

#include "fx8010_translate.inc"

// Every buffer of a call, both channel strides, one channel's ns periods and every per-instance curve of `cv` (n_cv of them) are
// aligned to `bytes`: what a kernel that moves bytes / 4 adjacent instances per access needs.
bool io_aligned(const fx8010_gpu* h, size_t bytes, const float* const* ins, const float* const* outs, int n_blk, size_t in_cs, size_t out_cs, int ns,
                const CurveBlock* cv = nullptr, int n_cv = 0) {
    const uintptr_t a = bytes - 1;
    if (((in_cs * 4) & a) || ((out_cs * 4) & a) || (((size_t)ns * h->N * 4) & a)) return false;
    for (int b = 0; b < n_blk; ++b) if (((uintptr_t)ins[b] | (uintptr_t)outs[b]) & a) return false;
    for (int j = 0; cv && j < n_cv; ++j) if (!cv->bcast[j] && ((uintptr_t)cv->p[j] & a)) return false;
    return true;
}

// Geometry of one launch: contexts per thread, block size, time split.
int plan_launch(fx8010_gpu* h, const float* d_in, const float* d_out, size_t in_cs, size_t out_cs, int n_samples, Launch& L) {
    const int N = h->N, C = h->C, nr = (int)h->reg_map.size();
    auto aligned = [&](int K) { return N % K == 0 && io_aligned(h, (size_t)K * 4, &d_in, &d_out, 1, in_cs, out_cs, n_samples); };
    const int min_seg = 8;
    const long max_seg = h->stateless ? std::max(1, n_samples / min_seg) : 1;
    const long want_threads = (long)h->num_sms * 512;
    int K = 4;
    // (measured on the 512-instruction cfg5 at 32 768 instances: K = 2 130 ms, K = 1 141 ms, K = 4 177 ms)
    while (K > 1 && (!aligned(K) || ((long)(N / K) * max_seg < want_threads && N / K < h->num_sms * 64))) K >>= 1;
    if (h->tune_K && aligned(h->tune_K)) K = h->tune_K;
    if (h->trace_mode) K = 1;
    // block size: spread small jobs over the SMs, keep several blocks per SM resident
    int B = 128;
    // input stage depth: a recurrence has nothing but its own future inputs to keep in flight, so make the
    // stage deep; a time-split (stateless) launch has many short segments and needs little.
    // Roughly 48 KiB of input rows in flight per SM cover HBM latency at full bandwidth; what the resident
    // warps do not provide through their number, each thread provides through a deeper stage.
    int chunk = 4;
    if (!h->stateless) {
        const double warps_per_sm = std::min(48.0, std::max(1.0, (double)N / K / 32.0 / h->num_sms));
        const double want = 49152.0 / (warps_per_sm * 32.0 * 4.0 * K * C);
        while (chunk < 32 && chunk < want) chunk <<= 1;
    }
    if (h->tune_chunk) chunk = h->tune_chunk;
    auto smem = [&](int b, int k, int ch) { return smem_bytes(nr, C, b, k, h->n_smem_tabs, ch); };
    auto fits = [&](int b, int k) { return smem(b, k, chunk) <= h->smem_optin; };
    // (cfg5, K = 2: 64- and 128-thread blocks 120 ms, 32-thread blocks 128 ms — the warps of a block share instruction
    //  and constant fetches — so shrink blocks only until every SM has one)
    while (B > 32 && ((long)((N / K + B - 1) / B) * max_seg < (long)h->num_sms || smem(B, K, chunk) > 80 * 1024)) B >>= 1;
    if (h->tune_B) B = std::min(h->tune_B, 128);
    while (!fits(B, K) && chunk > 4) chunk >>= 1;
    while (!fits(B, K) && K > 1) K >>= 1;
    while (!fits(B, K) && B > 32) B >>= 1;
    if (!fits(B, K)) return fail(h, FX8010_ERR_CAPACITY, "register file does not fit in shared memory");
    L.K = K; L.B = B; L.chunk = chunk; L.P = 1;
    L.smem = smem(B, K, chunk);
    L.grid_x = (N / K + B - 1) / B;
    L.n_seg = 1; L.seg_len = n_samples;
    if (h->stateless && n_samples > min_seg && !h->trace_mode) {
        KernelFn fn = use_short_kernel(h) ? short_kernel(K, h->has_ext, encoded_length(h)) : generic_kernel(K, h->has_skip, h->has_ext);
        int occ = 1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, B, L.smem);
        occ = std::max(occ, 1);
        long slots = (long)h->num_sms * occ;
        long n_seg = std::max(1L, slots / L.grid_x);
        if (h->tune_seg) n_seg = h->tune_seg;
        n_seg = std::min(n_seg, max_seg);
        int seg_len = (int)((n_samples + n_seg - 1) / n_seg);
        L.seg_len = seg_len;
        L.n_seg = (n_samples + seg_len - 1) / seg_len;
    }
    return FX8010_OK;
}

// READ-after-WRITE distance of a written TRAM stream in sample periods (0 = unknown): pointers untouched since load_program (both
// pointers of a ring then advance in lockstep from 0), offsets held by registers that carry one known value in every instance.
int ring_distance(const fx8010_gpu* h, const fx8010_gpu::TramStream& t) {
    if (!h->tram_ptrs_pristine || !h->reg_uniform[t.yreg] || !h->reg_uniform[t.w_yreg]) return 0;
    const int size = t.isx ? h->xtram_size : h->itram_size;
    if (size <= 0) return 0;
    const int pos = std::min(std::max(cvt_x86_host(h->reg_value[t.yreg]), 0), size - 1);
    const int wpos = std::min(std::max(cvt_x86_host(h->reg_value[t.w_yreg]), 0), size - 1);
    const int d = (wpos + pos) % size;
    return (d == 0 && !t.w_first) ? size : d;
}

// Shortest READ-after-WRITE distance of the TRAM streams (0 = unknown).  (The kernel checks the real distance per thread
// anyway; this only decides how long a batch is worth planning for.)
int known_tram_distance(const fx8010_gpu* h) {
    if (!h->tram_ptrs_pristine) return 0;
    int best = 1 << 30;
    for (const fx8010_instr& in : h->instrs) {            // a written ring shorter than a batch would see two samples of one batch in one slot
        const Uop u = uop_of(h, in);
        if (u == U_IWRITE) best = std::min(best, h->itram_size);
        if (u == U_XWRITE) best = std::min(best, h->xtram_size);
    }
    for (int q = 0; q < h->sl_n_tr; ++q) {
        if (h->sl_tr[q].w_yreg < 0) continue;              // nobody writes this ring: any batch length is safe
        const int D = ring_distance(h, h->sl_tr[q]);
        if (D <= 0) return 0;
        best = std::min(best, D);
    }
    return best;
}

// How many consecutive sample periods of a delay-line program are INDEPENDENT of one another, when the host can tell
// (same knowledge as above; 0 = unknown or a register recurrence exists).  A READ at period t fetches what the WRITE of
// period t - D stored (D = the distance above), and the WRITE of period t + (size - D) overwrites the slot the READ of
// period t fetched; within fewer periods than both, no period sees another's effect, so they can run in any order —
// across thread blocks: the time axis of such a launch is cut into segments exactly like a stateless program's
// (cfg3 with itramsize >= the block length: one fully parallel launch instead of 1 024 serial sample periods).
int known_tram_span(const fx8010_gpu* h) {
    if (!h->tram_ptrs_pristine || !h->sl_tram || h->sl_n_tr == 0) return 0;
    for (uint8_t c : h->sl_carry) if (c) return 0;
    int span = 1 << 30;
    for (const fx8010_instr& in : h->instrs) {
        const Uop u = uop_of(h, in);
        if (u == U_IWRITE) span = std::min(span, h->itram_size);
        if (u == U_XWRITE) span = std::min(span, h->xtram_size);
        if ((u == U_IWRITE || u == U_XWRITE || u == U_IREAD || u == U_XREAD) && !h->reg_uniform[in.y]) return 0;
    }
    for (int q = 0; q < h->sl_n_tr; ++q) {
        const fx8010_gpu::TramStream& t = h->sl_tr[q];
        if (t.w_yreg < 0) continue;                        // a ring nobody writes: its periods are independent anyway
        const int size = t.isx ? h->xtram_size : h->itram_size;
        const int D = ring_distance(h, t);
        if (D <= 0) return 0;
        span = std::min(span, D);
        if (D < size) span = std::min(span, size - D);      // write-after-read distance
    }
    // a ring with a WRITE but no READ stream, or a READ of a ring nobody writes, constrains nothing beyond the ring size
    return span == (1 << 30) ? 0 : span;
}

// Which translated kernel translation T gets: 0 = serial (fx_translated), 1 = streaming (a stateless program), 2 = streaming with
// TRAM (a delay line whose only state across periods is its rings and whose known span allows the launches route() cuts along
// time; the instruction-major kernel runs the rest).  With control curves every program the translator accepts runs translated
// (the interpreter kernels read no curves, and one serial launch costs far less than one launch per period): the streaming kernel
// also needs 16-byte accesses to whole groups of 4 instances, ring offsets that follow no curve (the cut needs offsets that are one
// known value), and no launch of this curve set that it did not fit (T.serial).
int tr_kind(const fx8010_gpu* h, const Translation& T) {
    if (!T.cv_reg.empty() && (T.serial || h->N % 4)) return 0;
    if (h->stateless) return 1;
    if (!(h->sl_ok && h->sl_tram && h->use_sl && h->use_tsplit && !(h->tr_recurrences & 2))) return 0;
    if (known_tram_span(h) < MIN_TSPLIT_SPAN) return 0;                 // (0 for a register recurrence)
    for (const fx8010_instr& in : h->instrs) {
        const Uop u = uop_of(h, in);
        if (u == U_IREAD || u == U_XREAD || u == U_IWRITE || u == U_XWRITE)
            for (int r : T.cv_reg) if (r == in.y) return 0;
    }
    return 2;
}

// Lets kernel fn use the device's opt-in dynamic shared-memory limit (once per kernel and handle; the occupancy query honours
// the limit only once it is set on the function).
template <class Fn> int smem_optin_for(fx8010_gpu* h, Fn fn) {
    const void* f = reinterpret_cast<const void*>(fn);
    if (std::find(h->smem_optin_fns.begin(), h->smem_optin_fns.end(), f) != h->smem_optin_fns.end()) return FX8010_OK;
    FX_CUDA(h, cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_optin));
    h->smem_optin_fns.push_back(f);
    return FX8010_OK;
}

// Geometry for the stateless kernel: all the parallelism a launch needs comes from cutting the time
// axis, so K is as wide as alignment allows and the segment count fills exactly one wave.
int plan_stateless(fx8010_gpu* h, const float*, const float*, unsigned align, int n_samples, int n_blk, bool may_overlap, bool tsplit, Launch& L) {
    // tsplit: a delay-line program whose periods within this launch are known to be independent (known_tram_span): planned like a stateless one
    const bool serial = h->sl_serial && !tsplit;
    const int N = h->N;
    auto aligned = [&](int K) { return N % K == 0 && (align & (unsigned)(K * 4 - 1)) == 0; };   // align: low bits of every buffer address and channel stride (bytes)
    int K = 4;
    if (tsplit) K = 2;                       // (the delay-line kernel at K = 4 sits at its register cap: cfg3, itramsize 8192: K = 4, M = 8 97 us; K = 2, M = 16 82 us; K = 1, M = 32 84 us)
    while (K > 1 && !aligned(K)) K >>= 1;
    bool splittable = serial && h->sl_tram && h->use_split;     // (see the sample split below)
    for (uint8_t c : h->sl_carry) splittable = splittable && !c;
    if (serial)                              // one time segment: the warps come from the instances alone — keep two per SM at least
        while (K > 1 && (long)N / K / 32 * (splittable ? 4 : 1) < 2L * h->num_sms * (splittable ? 2 : 1)) K >>= 1;   // (cfg4, 65 536 instances: K = 4 147 us, K = 2 158 us, K = 1 155 us; cfg3 with the split: K = 2 156 us, K = 1 180 us)
    if (h->tune_K && aligned(h->tune_K)) K = h->tune_K;
    // time-split launches: 64-thread blocks with batches of 8 samples (decode amortised over twice the samples at the
    // same shared-memory footprint as 128 x 4; cfg2: 8.7 vs 9.2 us)
    int B = h->tune_B ? std::min(h->tune_B, 128) : (serial ? 128 : 64);
    while (B > 32 && (N / K + B - 1) / B * B >= 2 * (N / K) && N / K <= B / 2) B >>= 1;      // tiny N: do not launch mostly-idle blocks
    if (serial && !h->tune_B)                // one time segment: only N / K threads — spread them over the SMs
        while (B > 32 && (N / K + B - 1) / B < 2 * h->num_sms) B >>= 1;
    // A serial launch has few warps, and the batch is also how far the input stage runs ahead: make it deep.
    // (a split program decodes every instruction once per thread and batch: with a delay known to exceed two 64-sample
    //  batches the longer batch halves that cost — cfg3: 152 -> 98 us)
    const bool deep = splittable && known_tram_distance(h) > 2 * SL_MAX_M;
    int M = h->tune_M ? h->tune_M : (serial ? ((deep || !h->sl_tram) ? SL_MAX_M : 32) : (tsplit ? 16 : 8));   // (a register recurrence: the batch overhead — decode, fetch issue — is serial with it: cfg4 at 8 192 instances, M = 32 79 us, 64 76 us)
    // serial: all blocks are resident at once; give each its share of the SM's shared memory
    // (with more blocks than fit at once the launch runs in waves: 56 KiB keeps four 128-thread blocks per SM)
    const size_t budget = serial ? std::min<size_t>(h->smem_optin, std::max<size_t>(56 * 1024, (size_t)200 * 1024 / std::max(1, ((N / K + B - 1) / B + h->num_sms - 1) / h->num_sms))) : (tsplit ? 48 * 1024 : 36 * 1024);     // (a delay line keeps two more stage rows per sample)
    while (!h->tune_M && M > 1 && sl_smem_bytes(h, B, K, M) > budget) M >>= 1;
    if (tsplit) while (M > 1 && 2 * M >= known_tram_span(h)) M >>= 1;    // the READs of batch b + 1 are prefetched while batch b runs
    if (serial && M < 2) M = 2;        // a carried operand reads row (m - 1) mod M while row m is written
    while (sl_smem_bytes(h, B, K, M) > h->smem_optin && B > 32) B >>= 1;
    // (a long program with many registers and shared-memory tables can need fewer instances per thread, like the general interpreter's plan)
    while (sl_smem_bytes(h, B, K, M) > h->smem_optin && K > 1 && !h->tune_K) K >>= 1;
    if (sl_smem_bytes(h, B, K, M) > h->smem_optin) return fail(h, FX8010_ERR_CAPACITY, "register file does not fit in shared memory");
    // Sample split: a serial program whose only state across sample periods is TRAM (nothing carried in registers) has
    // independent samples inside a batch, so P threads can share one instance column and take M / P samples each — P
    // times the warps for the same instances (cfg3: 16 384 instances are 512 warps otherwise, less than one per scheduler).
    int P = 1;
    bool any_carry = false;
    for (uint8_t c : h->sl_carry) any_carry = any_carry || c;
    if (serial && h->sl_tram && !any_carry && h->use_split) {
        while (P < 8 && (long)((N / K + 31) / 32) * P < 4L * h->num_sms && B * P * 2 <= 128 && M / (P * 2) >= 8) P <<= 1;   // (each thread decodes every instruction once per batch: keep its share of the batch long)
        if (h->tune_P && (h->tune_P & (h->tune_P - 1)) == 0 && B * h->tune_P <= 128 && M / h->tune_P >= 1) P = h->tune_P;
    }
    L.K = K; L.B = B; L.M = M; L.chunk = 0; L.P = P;
    L.smem = sl_smem_bytes(h, B, K, M);
    L.grid_x = (N / K + B - 1) / B;
    int occ = 1;
    const int rc = smem_optin_for(h, sl_kernel(K, h->sl_tram));
    if (rc) return rc;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, sl_kernel(K, h->sl_tram), B, L.smem);
    occ = std::max(occ, 1);
    // A launch that can overlap its neighbours (late wait, programmatic dependent launch) is planned as half a wave:
    // two consecutive launches share the SMs, and fewer, longer segments spend fewer instructions on per-thread start-up.
    // One that waits at its start has the SMs to itself: one full wave.
    const long slots = (long)h->num_sms * occ;
    long n_seg = std::max(1L, slots / ((may_overlap ? 2 : 1) * L.grid_x));
    // ... a launch much longer than its own ramp-up (many instances, or several sample blocks fused into it): all thread
    // blocks do the same amount of work, so the last wave is as long as a full one however few blocks it holds — pick
    // the segment count whose block count sits just below a whole number of waves (cfg2, 20 blocks per launch: 3 segments =
    // 0.93 waves instead of 8 = 2.47), preferring few long segments (less per-block start-up) once every SM is busy.
    const double work = (double)N * n_samples * n_blk;
    if (work > 8.0 * 4096 * 1024 || n_blk > 1) {
        const long items = (long)L.grid_x * n_blk;
        const long max_seg = std::max(1L, (long)n_samples / std::max(M, 16));
        long best = 1; double best_cost = 1e30;
        for (long c = 1; c <= max_seg; ++c) {
            const double w = (double)items * c / (double)slots;
            const double waves = std::ceil(w - 1e-9);
            double cost = waves / w;                                  // time relative to perfectly divisible work
            if (w < 0.8) cost += (0.8 - w) * 4.0;                     // not enough blocks to fill the SMs
            cost += 0.01 * (double)c / (double)max_seg * 4.0;         // mild preference for fewer, longer segments
            if (cost < best_cost - 1e-9) { best_cost = cost; best = c; }
        }
        n_seg = best;
    }
    if (h->tune_seg) n_seg = h->tune_seg;
    n_seg = std::min<long>(n_seg, std::max(1, n_samples / M));
    if (serial) n_seg = 1;                   // a recurrence cannot be cut along time
    int seg_len = (int)((n_samples + n_seg - 1) / n_seg);
    seg_len = (seg_len + M - 1) / M * M;
    L.seg_len = seg_len;
    L.n_seg = (n_samples + seg_len - 1) / seg_len;
    return FX8010_OK;
}

// ---- constant-memory residency (see the comment at g_arena) ----
void arena_release(fx8010_gpu* h) {            // g_dev_mutex[h->device] held
    if (h->arena_family < 0) return;
    std::vector<ArenaBlock>& v = g_arena[h->device][h->arena_family];
    for (size_t i = 0; i < v.size(); ++i)
        if (v[i].owner == h) { v.erase(v.begin() + i); break; }
    h->arena_family = -1; h->arena_off = -1; h->arena_words = 0;
}
// Makes `words` words of family `fam`'s arena belong to `h`; `fresh` = the range is new (its contents must be uploaded).
int arena_acquire(fx8010_gpu* h, int fam, int words, bool& fresh) {   // g_dev_mutex[h->device] held
    fresh = false;
    std::vector<ArenaBlock>& v = g_arena[h->device][fam];
    const unsigned long long stamp = ++g_arena_stamp[h->device];
    if (h->arena_family == fam && h->arena_off >= 0 && h->arena_words >= words) {
        for (ArenaBlock& b : v) if (b.owner == h) b.stamp = stamp;
        return FX8010_OK;
    }
    arena_release(h);
    if (words > ARENA_WORDS) return fail(h, FX8010_ERR_CAPACITY, "program does not fit the constant-memory arena");
    bool synced = false;
    while (true) {
        std::sort(v.begin(), v.end(), [](const ArenaBlock& a, const ArenaBlock& b) { return a.off < b.off; });
        int off = 0, found = -1;
        for (size_t i = 0; i <= v.size(); ++i) {                        // first fit
            const int end = i < v.size() ? v[i].off : ARENA_WORDS;
            if (end - off >= words) { found = off; break; }
            if (i < v.size()) off = v[i].off + v[i].words;
        }
        if (found >= 0) {
            v.push_back(ArenaBlock{found, words, h, stamp});
            h->arena_family = fam; h->arena_off = found; h->arena_words = words;
            fresh = true;
            return FX8010_OK;
        }
        // full: the least recently launched program goes (its kernels may still be running: wait for the device once)
        if (!synced) { FX_CUDA(h, cudaDeviceSynchronize()); synced = true; }
        size_t lru = 0;
        for (size_t i = 1; i < v.size(); ++i) if (v[i].stamp < v[lru].stamp) lru = i;
        fx8010_gpu* const victim = v[lru].owner;
        victim->arena_family = -1; victim->arena_off = -1; victim->arena_words = 0;
        v.erase(v.begin() + lru);
    }
}

// The launch's input block as a 2-D tensor for bulk tensor copies (TMA): [rows][N] float32, box = [M rows][B * K instances].
// Returns false when the driver entry point is missing or the shape does not qualify (the kernel then stages with cp.async).
bool make_input_map(const float* in, size_t N, size_t rows, int box_cols, int box_rows, SLTensorMap* out) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static const EncodeFn encode = []() -> EncodeFn {          // (thread-safe: handles of different devices launch from different host threads)
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess) return (EncodeFn)fn;
        cudaGetLastError();
        return nullptr;
    }();
    if (!encode || box_cols > 256 || box_rows > 256 || (N * 4) % 16 != 0 || ((uintptr_t)in & 15u)) return false;
    static_assert(sizeof(CUtensorMap) == sizeof(SLTensorMap), "CUtensorMap is 128 bytes");
    const cuuint64_t gdim[2] = {(cuuint64_t)N, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)N * 4};
    const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return encode(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(in), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Work this handle queued on another stream comes first (device-side ordering, no host wait).
int order_on(fx8010_gpu* h, cudaStream_t st) {
    if (h->has_last && h->last_stream != st) {
        if (cudaEventRecord(h->ev_order, h->last_stream) == cudaSuccess) FX_CUDA(h, cudaStreamWaitEvent(st, h->ev_order, 0));
        else { cudaGetLastError(); FX_CUDA(h, cudaDeviceSynchronize()); }      // that stream no longer exists: everything on the device comes first
        h->chain.clear();
    }
    h->last_stream = st; h->has_last = true;
    return FX8010_OK;
}

// How the next piece of a call runs (route).
enum Path {
    PATH_SPLIT,           // cut every block into pieces of `len` periods and route each piece again
    PATH_TR_SERIAL,       // the translated serial kernel, block after block
    PATH_TR_STREAM,       // the translated streaming kernel: a stateless program, or a delay line cut along time
    PATH_INTERP,          // the instruction-major kernel, else the short-program kernel, else the general interpreter
    PATH_PER_PERIOD,      // (control curves) per period, one copy of the curves into the registers and one plain one-period call
};
struct Route {
    Path path;
    int len;              // periods per launch: the whole block, a stretch of known_tram_span, the counter limit (PATH_SPLIT), or one
    int fuse = 1;         // sample blocks one launch may take
    bool tsplit = false;  // (PATH_INTERP) a delay line whose periods in this launch are independent: planned like a stateless program
};

// Which kernel runs the next piece of a call: n_blk blocks of ns periods (plain translation h->tr), or one with the curves cv (h->tr_cv).
// Reaching tr_ready starts a compile: the order of the conditions decides which programs ever compile (a plain cfg4 call never does).
Route route(fx8010_gpu* h, const float* const* ins, float* const* outs, int n_blk, size_t in_cs, size_t out_cs, int ns, const CurveBlock* cv) {
    // per-launch executed-instruction counters are 32-bit: split very long batches
    const long long per_sample = (long long)h->instrs.size() * FX8010_MAX_PASSES;
    const int max_samples = (int)std::max<long long>(1, std::min<long long>(0x7fffffffLL, 0xffffffffLL / per_sample));
    if (ns > max_samples) return Route{PATH_SPLIT, max_samples};
    if (cv) {
        // Control curves run translated or period by period (the interpreter kernels read no curves).
        const Route per_period{PATH_PER_PERIOD, 1};
        Translation& T = h->tr_cv;
        const int n_cv = (int)T.cv_reg.size();
        if (h->trace_mode || !tr_ready(h, T)) return per_period;
        if (T.kind != 0) {
            // the streaming kernel: 16-byte accesses at i0 to the samples and to the per-instance curves; a delay line is cut along time
            const int span = T.kind == 2 ? known_tram_span(h) : ns;
            if (io_aligned(h, 16, ins, outs, 1, in_cs, out_cs, ns, cv, n_cv) && span >= std::min(ns, MIN_TSPLIT_SPAN))
                return Route{span < ns ? PATH_SPLIT : PATH_TR_STREAM, std::min(span, ns)};
            // It does not fit this launch (a buffer not 16-byte aligned, a delay line whose span is no longer known): from now on
            // this curve set takes the serial kernel, which needs neither.
            T.serial = true;
            tr_reset(h, T);
            if (!tr_ready(h, T)) return per_period;
        }
        return io_aligned(h, (size_t)T.lanes * 4, ins, outs, 1, in_cs, out_cs, ns, cv, n_cv) ? Route{PATH_TR_SERIAL, ns} : per_period;
    }
    // Delay lines: periods closer than the known span are independent, so a block is cut into stretches of at most that
    // many periods, each one launch cut along time like a stateless program (the stretches themselves run in order).
    const int span = (h->sl_ok && h->use_sl && !h->trace_mode && h->use_tsplit) ? known_tram_span(h) : 0;
    // (worth it when the block needs at most two launches — cfg3 at 16 384 instances x 1 024 periods: span 100, eleven launches,
    //  198 us against 139 us for the serial kernel with its sample split; span 1 000, two launches, 111 against 112; one launch, 82)
    // ... or any number of launches when they run on the translated streaming kernel (tr_kind 2): a stretch of 100 periods
    // of cfg3 is a 6 us launch there (cfg3, ring of 100: 11 launches 66 us against 134 us serial)
    const bool stretch = span >= MIN_TSPLIT_SPAN && 2L * span < ns && tr_kind(h, h->tr) == 2 && h->use_translate && h->N % 4 == 0 &&
                         io_aligned(h, 16, ins, outs, n_blk, in_cs, out_cs, ns) && tr_ready(h, h->tr);
    const bool tsplit = span >= MIN_TSPLIT_SPAN && (2L * span >= ns || stretch);
    if (tsplit && ns > span) return Route{PATH_SPLIT, span};
    // Programs of the general interpreter run on their translated kernel once it exists (fx8010_translate.inc).
    // FX8010_TR_RECUR (developer switch): bit 0 = self recurrences (cfg4), bit 1 = delay lines (cfg3) take the translated serial kernel
    const bool tr_recur = h->sl_ok && h->sl_serial && (((h->tr_recurrences & 1) && !h->sl_tram) || ((h->tr_recurrences & 2) && h->sl_tram));
    if (!h->stateless && (tr_recur || (!(h->sl_ok && h->use_sl) && !use_short_kernel(h))) && !h->trace_mode && tr_ready(h, h->tr) &&
        io_aligned(h, (size_t)h->tr.lanes * 4, ins, outs, n_blk, in_cs, out_cs, ns))
        return Route{PATH_TR_SERIAL, ns};
    // A stateless program, or a delay line cut along time, runs on the translated streaming kernel once that exists: 4 adjacent
    // instances per thread, so the instance count and every buffer must allow 16-byte accesses.
    const bool tr_sl = (h->stateless || (tsplit && tr_kind(h, h->tr) == 2)) && !h->trace_mode && h->N % 4 == 0 &&
                       io_aligned(h, 16, ins, outs, n_blk, in_cs, out_cs, ns) && tr_ready(h, h->tr);
    const bool fuse = (h->sl_ok && h->use_sl && !h->trace_mode && !h->sl_serial && h->use_fuse) || (tr_sl && h->stateless);
    return Route{tr_sl ? PATH_TR_STREAM : PATH_INTERP, ns, fuse ? MAX_FUSED_BLOCKS : 1, tsplit};
}

// Cuts the ns periods of every block into pieces of at most len and hands each to run(in, out, periods, s0, own_prev), blocks in
// order; every piece but the first follows this handle's own launch.
template <class Run> int split_periods(const fx8010_gpu* h, const float* const* ins, float* const* outs, int n_blk, int ns, int len, bool own_prev, Run run) {
    for (int b = 0; b < n_blk; ++b)
        for (int s0 = 0; s0 < ns; s0 += len) {
            const float* in = ins[b] ? ins[b] + (size_t)s0 * h->N : nullptr;
            float* out = outs[b] + (size_t)s0 * h->N;
            const int rc = run(in, out, std::min(len, ns - s0), s0, own_prev || b > 0 || s0 > 0);
            if (rc) return rc;
        }
    return FX8010_OK;
}

// Books one launch on `path` with geometry L over nb blocks of ns periods: the TRAM periods, the chain of late-waiting launches and
// h->info.  `sp`: the buffers the launch touches (plain interpreter and streaming launches join the chain; the other launches wait at
// their start and leave it empty).  `tma` < 0 leaves info.last_tma as it was.  Known discrepancies, kept as they are:
//   * a fused launch of the streaming kernel reports last_grid = grid_x * n_seg, without its nb blocks;
//   * bit 32 (short-program kernel) is set by M == 0 && use_short_kernel(h) for a plain launch of the streaming kernel too;
//   * a launch of the general interpreter or the short-program kernel leaves last_tma as the launch before it set it.
void record_launch(fx8010_gpu* h, Path path, const Launch& L, int nb, int ns, int late_wait, int tma, bool curves, const fx8010_gpu::Span* sp,
                   cudaStream_t st) {
    const bool translated = path == PATH_TR_SERIAL || path == PATH_TR_STREAM;
    const bool lean = L.M == 0 && (path == PATH_INTERP || (path == PATH_TR_STREAM && !curves)) && use_short_kernel(h);
    const bool pairs = L.M > 0 && std::any_of(h->sl_fuse.begin(), h->sl_fuse.end(), [](uint8_t f) { return f != 0; });
    h->tram_periods += (unsigned long long)ns * nb;
    if (!late_wait) h->chain.clear();          // this launch waited at its start: everything before it is complete
    if (sp) { h->chain.push_back(*sp); h->chain_stream = st; }
    h->info.kernel_launches++;
    h->info.last_grid = L.grid_x * L.n_seg * (path == PATH_TR_STREAM ? 1 : nb); h->info.last_block = L.B * L.P; h->info.last_time_split = L.n_seg;
    h->info.last_smem_bytes = (int)L.smem;
    h->info.last_late_wait = late_wait; h->info.last_fused_blocks = nb;
    if (tma >= 0) h->info.last_tma = tma;
    h->info.kernel_variant = (h->has_skip ? 1 : 0) | (h->has_ext ? 2 : 0) | (h->stateless ? 4 : 0) | (L.M > 0 ? 8 : 0) | (curves ? 16 : 0) | (lean ? 32 : 0) |
                             (pairs ? 64 : 0) | (translated ? 128 : 0) | (L.K << 8) | (L.M << 16);
}

// The runtime-API launch of an interpreter kernel: grid = instance groups x (time segments x nb blocks), programmatic dependent
// launch when enabled.
template <class Fn, class P> int interp_drive(fx8010_gpu* h, Fn fn, const Launch& L, int nb, cudaStream_t st, const P& p) {
    const int rc = smem_optin_for(h, fn);
    if (rc) return rc;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(L.grid_x, L.n_seg * nb); cfg.blockDim = dim3(L.B * L.P); cfg.dynamicSmemBytes = L.smem; cfg.stream = st;
    cudaLaunchAttribute attrs[1];
    attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attrs; cfg.numAttrs = h->use_pdl ? 1 : 0;
    FX_CUDA(h, cudaLaunchKernelEx(&cfg, fn, p));
    return FX8010_OK;
}

// nb consecutive blocks on the instruction-major kernel (geometry L from plan_stateless; tsplit as routed).  `tma`: whether its
// input stage uses bulk tensor copies.
int sl_launch(fx8010_gpu* h, const Launch& L, const float* const* ins, float* const* outs, int nb, size_t in_cs, size_t out_cs, int ns, bool tsplit,
              int late_wait, cudaStream_t st, int& tma) {
    SLParams p = {};
    p.gpr = h->d_gpr; p.acc = h->d_acc; p.latch = h->d_latch; p.counts = h->d_counts; p.rt_flags = h->d_flags;
    p.tabs = h->d_tabs; p.load_list = h->d_sl_load; p.wb_list = h->d_sl_wb;
    p.n_blk = nb;
    for (int b = 0; b < nb; ++b) { p.blk_in[b] = ins[b]; p.blk_out[b] = outs[b]; }
    p.in_cstride = in_cs; p.out_cstride = out_cs;
    p.n_samples = ns; p.seg_len = L.seg_len; p.n_seg = L.n_seg;
    p.N = h->N; p.C = h->C; p.n_instrs = (int)h->instrs.size(); p.n_exec = h->n_exec; p.prog_off = h->arena_off;
    p.n_load = (int)h->sl_load.size(); p.n_wb = (int)h->sl_wb.size();
    p.M = L.M;
    p.stage0 = (uint32_t)L.B * L.K * 4u * (uint32_t)(h->sl_n_ro + h->sl_n_wo + h->sl_n_rw * L.M);
    p.n_smem_tabs = h->n_smem_tabs;
    for (int t = 0; t < MAX_SMEM_TABLES; ++t) p.smem_tab_id[t] = h->smem_tab_id[t];
    p.acc_writer = h->acc_writer ? 1 : 0;
    p.ccr_live = h->sl_ccr_live ? 1 : 0;
    p.ptrs = h->d_ptrs; p.itram = h->d_itram; p.xtram = h->d_xtram; p.itram_size = h->itram_size; p.xtram_size = h->xtram_size;
    p.has_tram = h->sl_tram ? 1 : 0; p.n_tr = h->sl_n_tr; p.P = L.P;
    for (int j = 0; j < 4; ++j) p.tr_ops[j] = 0;
    for (const fx8010_instr& ins_ : h->instrs) {         // pointer j (iw, ir, xw, xr) moves once per sample period per executed op
        const Uop u = uop_of(h, ins_);
        if (u == U_IWRITE) p.tr_ops[0]++; else if (u == U_IREAD) p.tr_ops[1]++;
        else if (u == U_XWRITE) p.tr_ops[2]++; else if (u == U_XREAD) p.tr_ops[3]++;
    }
    p.tr_on[0] = p.tr_on[1] = 0;
    for (int q = 0; q < h->sl_n_tr; ++q) {
        const fx8010_gpu::TramStream& t = h->sl_tr[q];
        const int x = t.isx;                             // the kernel indexes streams by TRAM: 0 = iTRAM, 1 = xTRAM
        p.tr_on[x] = 1;
        p.tr_stage[x] = sl_word(h, t.reg, L.B, L.K, L.M) & SL_OFF_MASK;
        p.tr_y[x] = sl_word(h, t.yreg, L.B, L.K, L.M) & SL_OFF_MASK;
        p.tr_wy[x] = t.w_yreg >= 0 ? (sl_word(h, t.w_yreg, L.B, L.K, L.M) & SL_OFF_MASK) : 0xffffffffu;
        p.tr_wfirst[x] = t.w_first;
    }
    // cut along time (the pointers are as load_program left them and have moved once per period launched since — known_tram_span):
    // every segment starts from the host's copy of the pointers, not from the array the last segment's owner rewrites
    p.tr_base_valid = 0;
    if (h->sl_tram && tsplit && L.n_seg > 1 && h->tram_ptrs_pristine) {
        p.tr_base_valid = 1;
        for (int j = 0; j < 4; ++j) {
            const int size = j < 2 ? h->itram_size : h->xtram_size;
            p.tr_base[j] = (size > 0 && p.tr_ops[j]) ? (int)(h->tram_periods * (unsigned long long)p.tr_ops[j] % (unsigned long long)size) : 0;
        }
    }
    p.pdl_late_wait = late_wait;
    p.use_tma = 0;
    // Bulk tensor copies (TMA) for the input stage: one instruction per batch and channel instead of one cp.async per thread and
    // sample row.  Pays where the per-batch overhead is serial with a recurrence (cfg4 at 8 192 instances: 67 -> 59 us, at 65 536:
    // 125 -> 121 us); a time-split launch loses a little to the block-wide barrier per batch (cfg2 per launch: 8.5 -> 8.6 us) and keeps cp.async.
    if ((h->use_tma == 2 || (h->use_tma == 1 && L.n_seg == 1 && h->sl_serial)) && !h->sl_tram && nb == 1 && ins[0] && L.P == 1 && in_cs % (size_t)h->N == 0) {
        const size_t rpc = in_cs / (size_t)h->N;
        if (make_input_map(ins[0], (size_t)h->N, (size_t)(h->C - 1) * rpc + (size_t)ns, L.B * L.K, L.M, &p.in_map)) { p.use_tma = 1; p.tma_rows_per_channel = (int)rpc; }
    }
    tma = p.use_tma;
    return interp_drive(h, sl_kernel(L.K, h->sl_tram), L, nb, st, p);
}

// One block on the general interpreter, or on the short-program kernel when the program is short enough (geometry L from plan_launch).
int generic_launch(fx8010_gpu* h, const Launch& L, const float* in, float* out, size_t in_cs, size_t out_cs, int ns, int late_wait, cudaStream_t st) {
    Params p = {};
    p.gpr = h->d_gpr; p.acc = h->d_acc; p.lfsr = h->d_lfsr; p.latch = h->d_latch; p.ptrs = h->d_ptrs;
    p.itram = h->d_itram; p.xtram = h->d_xtram; p.counts = h->d_counts; p.rt_flags = h->d_flags;
    p.reg_map = h->d_reg_map; p.load_rows = h->d_load_rows; p.wb_regs = h->d_wb; p.latch_ch = h->d_latch_ch; p.tabs = h->d_tabs;
    p.in = in; p.out = out; p.in_cstride = in_cs; p.out_cstride = out_cs;
    p.n_samples = ns; p.seg_len = L.seg_len; p.n_seg = L.n_seg;
    p.N = h->N; p.C = h->C; p.n_regs = (int)h->reg_map.size(); p.n_instrs = (int)h->instrs.size();
    p.n_wb = (int)h->wb.size(); p.prog_off = h->arena_off;
    p.n_exec = h->n_exec; p.n_latch_ch = (int)h->latch_ch.size(); p.n_unpred = h->n_unpred;
    p.n_load = (int)h->load_rows.size(); p.load_latch = h->load_latch; p.load_acc = h->load_acc;
    p.itram_size = h->itram_size; p.xtram_size = h->xtram_size;
    p.n_smem_tabs = h->n_smem_tabs;
    for (int t = 0; t < MAX_SMEM_TABLES; ++t) p.smem_tab_id[t] = h->smem_tab_id[t];
    p.chunk = L.chunk;
    p.pdl_late_wait = late_wait;
    const bool kskip = h->has_skip || h->trace_mode, kext = h->has_ext || h->trace_mode;
    p.trace = h->trace_mode ? h->d_trace : nullptr; p.trace_inst = h->trace_inst;
    return interp_drive(h, use_short_kernel(h) ? short_kernel(L.K, kext, h->n_exec) : generic_kernel(L.K, kskip, kext), L, 1, st, p);
}

// The driver-API launch of translated kernel T (it lives in an NVRTC module): grid = L.grid_x x (L.n_seg x nb blocks), programmatic
// dependent launch when enabled.
int tr_drive(fx8010_gpu* h, const Translation& T, const Launch& L, int nb, cudaStream_t st, void** args) {
    const DriverApi& d = driver_api();
    CUlaunchConfig cfg = {};
    cfg.gridDimX = (unsigned)L.grid_x; cfg.gridDimY = (unsigned)(L.n_seg * nb); cfg.gridDimZ = 1;
    cfg.blockDimX = (unsigned)L.B; cfg.blockDimY = 1; cfg.blockDimZ = 1;
    cfg.sharedMemBytes = (unsigned)L.smem; cfg.hStream = (CUstream)st;
    CUlaunchAttribute attr[1];
    attr[0].id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
    attr[0].value.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = h->use_pdl ? 1 : 0;
    const CUresult rc = d.launchKernelEx(&cfg, (CUfunction)T.fn, args, nullptr);
    if (rc == CUDA_SUCCESS) return FX8010_OK;
    const char* msg = nullptr;
    if (d.getErrorString) d.getErrorString(rc, &msg);
    return fail(h, FX8010_ERR_CUDA, std::string("translated kernel launch: ") + (msg ? msg : "driver error"));
}

// One block on the translated serial kernel.  Same ordering rules as the interpreter launch that waits at its start.  `cv`: the
// call's control curves (the automated translation only).  L: the geometry it ran with.
int tr_launch(fx8010_gpu* h, const Translation& T, const float* in, float* out, size_t in_cs, size_t out_cs, int ns, cudaStream_t st, const CurveBlock* cv,
              Launch& L) {
    const DriverApi& d = driver_api();
    const int N = h->N;
    // block size: one warp per block until every SM holds a few; the kernel's registers bound residency anyway
    int B = 32;
    if ((long)N / T.lanes >= (long)h->num_sms * 32 * 16) B = 64;
    if ((long)N / T.lanes >= (long)h->num_sms * 32 * 64) B = 128;
    if (h->tune_B) B = h->tune_B;
    while (B > 32 && (size_t)T.ring_floats * B * 4 > h->smem_optin) B >>= 1;
    const unsigned smem = (unsigned)(T.ring_floats * B * 4);       // the input ring (<= 64 periods x 128 threads x 4 B per row)
    if (smem > 48 * 1024 &&                                        // beyond the default dynamic shared-memory limit: opt in
        (!d.funcSetAttribute || d.funcSetAttribute((CUfunction)T.fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)h->smem_optin) != CUDA_SUCCESS))
        return fail(h, FX8010_ERR_CAPACITY, "the translated kernel's input ring does not fit in shared memory");
    void* gpr = h->d_gpr; void* acc = h->d_acc; void* lfsr = h->d_lfsr; void* latch = h->d_latch; void* ptrs = h->d_ptrs;
    void* itram = h->d_itram; void* xtram = h->d_xtram; void* counts = h->d_counts; void* flags = h->d_flags; void* tabs = h->d_tabs;
    const void* inp = in; void* outp = out;
    int ns_ = ns, N_ = N, isz = h->itram_size, xsz = h->xtram_size;
    CurveBlock cvb = cv ? *cv : CurveBlock{};
    void* args[] = {&gpr, &acc, &lfsr, &latch, &ptrs, &itram, &xtram, &counts, &flags, &tabs, &inp, &outp, &in_cs, &out_cs, &ns_, &N_, &isz, &xsz, &cvb};
    L.K = T.lanes; L.B = B; L.P = 1; L.grid_x = (N / T.lanes + B - 1) / B; L.n_seg = 1; L.seg_len = ns; L.smem = smem;
    return tr_drive(h, T, L, 1, st, args);
}

// Time segments of a launch of a translated streaming kernel (fx_translated_sl, fx_translated_chain) over nb blocks of ns periods, gx thread
// blocks of B threads per segment row: every thread takes `seg_len` samples (whole 4-sample load groups).  Short segments mean more threads — a
// lone block ramps up faster (cfg2, one block per call: 11 us at 8 samples, 15-19 at 16-32) — long ones amortise the per-thread start-up once
// the launch holds a couple of waves anyway (cfg2, 20 blocks per launch: 6.3 us per block at 8, 5.9 at 32): the shortest power of two that
// keeps the launch within about 2.5 full waves of warps.
void sl_segments(const fx8010_gpu* h, int gx, int B, int ns, int nb, int& seg_len, int& n_seg) {
    seg_len = 8;
    const long warps_per_row = ((long)gx * B + 31) / 32;
    while (seg_len < ns && warps_per_row * ((ns + seg_len - 1) / seg_len) * nb > (long)h->num_sms * 64 * 5 / 2) seg_len <<= 1;
    if (env_int("FX8010_TUNE_SEGLEN") > 0) seg_len = env_int("FX8010_TUNE_SEGLEN");
    n_seg = (ns + seg_len - 1) / seg_len;
    while ((long)n_seg * nb > 65535) { seg_len <<= 1; n_seg = (ns + seg_len - 1) / seg_len; }
}

// nb consecutive blocks of a stateless program (or one stretch of a delay line) on its translated streaming kernel (late_wait as
// launch_blocks computes it).  `cv`: the call's control curves (the automated translation only; nb == 1).  L: the geometry it ran with.
int tr_sl_launch(fx8010_gpu* h, const Translation& T, const float* const* ins, float* const* outs, int nb, size_t in_cs, size_t out_cs, int ns, cudaStream_t st,
                 int late_wait, Launch& L, const CurveBlock* cv) {
    const int N = h->N, K = 4;
    struct { const float* in[32]; float* out[32]; } io = {};
    for (int b = 0; b < nb; ++b) { io.in[b] = ins[b]; io.out[b] = outs[b]; }
    int B = 128;
    if (h->tune_B) B = h->tune_B;
    const int gx = (N / K + B - 1) / B;
    int seg_len, n_seg;
    sl_segments(h, gx, B, ns, nb, seg_len, n_seg);
    void* gpr = h->d_gpr; void* acc = h->d_acc; void* latch = h->d_latch; void* counts = h->d_counts; void* flags = h->d_flags; void* tabs = h->d_tabs;
    int ns_ = ns, nb_ = nb, N_ = N, lw = late_wait, isz = h->itram_size, xsz = h->xtram_size;
    void* ptrs = h->d_ptrs; void* itram = h->d_itram; void* xtram = h->d_xtram;
    // ring pointers at this launch's first period (delay lines only: every pointer of a ring that has the instruction has moved once per period since load_program)
    int base[4] = {0, 0, 0, 0};
    if (T.kind == 2) {
        const unsigned long long done = h->tram_periods;
        if (h->itram_size > 0) base[0] = base[1] = (int)(done % (unsigned long long)h->itram_size);
        if (h->xtram_size > 0) base[2] = base[3] = (int)(done % (unsigned long long)h->xtram_size);
    }
    CurveBlock cvb = cv ? *cv : CurveBlock{};
    void* args[] = {&io, &gpr, &acc, &latch, &counts, &flags, &tabs, &in_cs, &out_cs, &ns_, &seg_len, &n_seg, &nb_, &N_, &lw, &ptrs, &itram, &xtram, &isz, &xsz,
                    &base[0], &base[1], &base[2], &base[3], &cvb};
    L.K = K; L.B = B; L.P = 1; L.M = 0; L.grid_x = gx; L.n_seg = n_seg; L.seg_len = seg_len; L.smem = 0; L.chunk = 0;
    return tr_drive(h, T, L, nb, st, args);
}

// Launches n_blk consecutive sample blocks of ns samples each (block b: ins[b] -> outs[b]) the way route() decides.  A time-split
// (stateless) program runs up to MAX_FUSED_BLOCKS of them in ONE launch — its work items are (block, time segment, instance group)
// and all are independent; everything else runs block after block.  `own_prev`: the operation right before this one on
// `st` is known to be this handle's own launch (or nothing that signals programmatic completion early).
int launch_blocks(fx8010_gpu* h, const float* const* ins, float* const* outs, int n_blk, size_t in_cs, size_t out_cs, int ns, cudaStream_t st, bool own_prev) {
    if (ns == 0 || n_blk == 0) return FX8010_OK;
    {
        const int rc = order_on(h, st);
        if (rc) return rc;
    }
    const Route r = route(h, ins, outs, n_blk, in_cs, out_cs, ns, nullptr);
    if (r.path == PATH_SPLIT)
        return split_periods(h, ins, outs, n_blk, ns, r.len, own_prev, [&](const float* in, float* out, int k, int, bool own) {
            return launch_blocks(h, &in, &out, 1, in_cs, out_cs, k, st, own);
        });
    if (r.path == PATH_TR_SERIAL) {
        for (int b = 0; b < n_blk; ++b) {
            Launch L = {};
            const int rc = tr_launch(h, h->tr, ins[b], outs[b], in_cs, out_cs, ns, st, nullptr, L);
            if (rc) return rc;
            record_launch(h, r.path, L, 1, ns, 0, 0, false, nullptr, st);
        }
        return FX8010_OK;
    }
    const bool tr_sl = r.path == PATH_TR_STREAM, tsplit = r.tsplit;
    for (int b0 = 0; b0 < n_blk;) {
        const int nb = std::min(n_blk - b0, r.fuse);
        if (h->encode_dirty && !tr_sl) { select_tables(h); h->plan_key.ns = -1; }
        Launch L = {};
        // the plan depends on the batch length and on how far the buffers are aligned
        unsigned align = 0;
        for (int b = b0; b < b0 + nb; ++b) align |= (unsigned)(((uintptr_t)ins[b] | (uintptr_t)outs[b]) & 15u);
        const bool any_in = ins[b0] != nullptr;                   // (fx8010_gpu_process_blocks refuses a list that mixes NULL and non-NULL inputs)
        align |= (unsigned)(((uintptr_t)(in_cs * 4) | (uintptr_t)(out_cs * 4)) & 15u) | (any_in ? 16u : 0u);
        const int deep = ((h->sl_ok && h->sl_tram) ? (known_tram_distance(h) > 2 * SL_MAX_M ? 1 : 0) : 0) | (tsplit ? 2 : 0);
        // a launch that may overlap its neighbours (late wait) is planned as half a wave; one that waits at its start fills the SMs
        const bool may_overlap = h->use_pdl && h->stateless && nb == 1 && (h->stream_exclusive || own_prev || b0 > 0);
        if (tr_sl) {}                                              // (its geometry is decided at the launch)
        else if (h->plan_key.ns == ns && h->plan_key.align == align && h->plan_key.deep == deep && h->plan_key.n_blk == nb && h->plan_key.wave == (int)may_overlap) L = h->plan;
        else {
            L.M = 0;
            const int rc = (h->sl_ok && h->use_sl && !h->trace_mode) ? plan_stateless(h, ins[b0], outs[b0], align, ns, nb, may_overlap, tsplit, L)
                                                                     : plan_launch(h, ins[b0], outs[b0], in_cs, out_cs, ns, L);
            if (rc) return rc;
            h->plan = L; h->plan_key.ns = ns; h->plan_key.align = align; h->plan_key.deep = deep; h->plan_key.n_blk = nb; h->plan_key.wave = (int)may_overlap;
        }
        // the kernel family that will run this launch (each keeps its own constant-memory copy of the program)
        const Family fam = L.M > 0 ? sl_family(L.K) : ((use_short_kernel(h)) ? FAM_SHORT : FAM_GENERIC);
        const bool reencode = !tr_sl && (h->encode_dirty || h->enc_K != L.K || h->enc_B != L.B || h->sl_M != L.M || (L.M == 0 && h->enc_chunk != L.chunk) || h->enc_family != (int)fam);
        if (reencode) {
            // the previous upload must have left the pinned buffer before it is rewritten
            FX_CUDA(h, cudaStreamSynchronize(st));
            if (L.M > 0) encode_stateless(h, L.K, L.B, L.M); else encode(h, L.K, L.B, L.chunk);
        }
        std::unique_lock<std::mutex> lk(g_dev_mutex[h->device], std::defer_lock);       // residency check -> launch
        bool fresh = false;
        if (!tr_sl) {
            lk.lock();
            const int rc = arena_acquire(h, (int)fam, (L.M > 0 ? 4 : 2) * (h->n_exec + 1), fresh);
            if (rc) return rc;
        }
        if (reencode || fresh) {
            FX_CUDA(h, cudaStreamSynchronize(st));                     // kernels still reading the old image of this range
            FX_CUDA(h, upload_program(fam, h->h_prog, sizeof(uint4) * (L.M > 0 ? 4 : 2) * (h->n_exec + 1), h->arena_off, st));
            h->enc_family = (int)fam;
            if (reencode) {
                if (L.M > 0) {
                    FX_CUDA(h, cudaMemcpyAsync(h->d_sl_load, h->sl_load.data(), sizeof(uint2) * h->sl_load.size(), cudaMemcpyHostToDevice, st));
                    FX_CUDA(h, cudaMemcpyAsync(h->d_sl_wb, h->sl_wb.data(), sizeof(uint2) * h->sl_wb.size(), cudaMemcpyHostToDevice, st));
                } else
                    FX_CUDA(h, cudaMemcpyAsync(h->d_latch_ch, h->latch_ch.data(), sizeof(uint32_t) * h->latch_ch.size(), cudaMemcpyHostToDevice, st));
            }
            FX_CUDA(h, cudaStreamSynchronize(st));
            h->encode_dirty = false;
            h->chain.clear();
        }
        // Programmatic dependent launch: the kernel may start while the previous launch on this stream drains.  It can
        // postpone its wait to the final state write-back when it reads nothing an earlier launch writes and writes
        // nothing an earlier launch reads or writes: a stateless program (its start-up reads only rows nobody writes)
        // whose I/O buffers are disjoint from those of EVERY launch that may still be running — all launches since the
        // last one that waited at its start (a launch starts once all blocks of its predecessor have started, so with
        // small grids several generations can be resident at once).  That reasoning covers this handle's own launches
        // only, so the operation right before this one on the stream must be known to be one of them: inside a
        // multi-block call, or when the caller set FX8010_OPT_STREAM_EXCLUSIVE.
        fx8010_gpu::Span sp;
        sp.out_lo = sp.out_hi = (const char*)outs[b0]; sp.in_lo = sp.in_hi = (const char*)ins[b0];
        bool disjoint = h->chain_stream == st && !h->chain.empty() && (int)h->chain.size() < MAX_CHAIN;
        auto overlap = [](const char* a0, const char* a1, const char* b0_, const char* b1) { return a0 < b1 && b0_ < a1; };
        for (int b = b0; b < b0 + nb; ++b) {
            const char* o_lo = (const char*)outs[b]; const char* o_hi = o_lo + sizeof(float) * ((size_t)(h->C - 1) * out_cs + (size_t)ns * h->N);
            const char* i_lo = (const char*)ins[b]; const char* i_hi = ins[b] ? i_lo + sizeof(float) * ((size_t)(h->C - 1) * in_cs + (size_t)ns * h->N) : i_lo;
            for (const fx8010_gpu::Span& q : h->chain)
                disjoint = disjoint && !overlap(o_lo, o_hi, q.out_lo, q.out_hi) && !overlap(i_lo, i_hi, q.out_lo, q.out_hi) && !overlap(o_lo, o_hi, q.in_lo, q.in_hi);
            sp.out_lo = std::min(sp.out_lo, o_lo); sp.out_hi = std::max(sp.out_hi, o_hi);
            if (ins[b]) { sp.in_lo = std::min(sp.in_lo, i_lo); sp.in_hi = std::max(sp.in_hi, i_hi); }
        }
        const int late_wait = (may_overlap && disjoint) ? 1 : 0;
        int tma = -1, rc;
        if (tr_sl) { rc = tr_sl_launch(h, h->tr, ins + b0, outs + b0, nb, in_cs, out_cs, ns, st, late_wait, L, nullptr); tma = 0; }
        else if (L.M > 0) rc = sl_launch(h, L, ins + b0, outs + b0, nb, in_cs, out_cs, ns, tsplit, late_wait, st, tma);
        else rc = generic_launch(h, L, ins[b0], outs[b0], in_cs, out_cs, ns, late_wait, st);
        if (rc) return rc;
        record_launch(h, r.path, L, nb, ns, late_wait, tma, false, &sp, st);
        b0 += nb;
    }
    return FX8010_OK;
}

int launch_block(fx8010_gpu* h, const float* d_in, float* d_out, size_t in_cs, size_t out_cs, int n_samples, cudaStream_t st, bool own_prev = false) {
    return launch_blocks(h, &d_in, &d_out, 1, in_cs, out_cs, n_samples, st, own_prev);
}

// ---- control curves (fx8010_gpu_process_batch_curves) ----
// A curve list the call accepts: registers in range, each named once, each a CONTROL or STATIC register.
bool curves_valid(const std::vector<fx8010_reg>& regs, const std::vector<int>& cv_reg, std::string& why) {
    for (size_t j = 0; j < cv_reg.size(); ++j) {
        const int r = cv_reg[j];
        if (r < 0 || r >= (int)regs.size()) { why = "control curve: register index out of range"; return false; }
        if (regs[r].type != FX_REG_CONTROL && regs[r].type != FX_REG_STATIC) { why = "control curve: the register is neither CONTROL nor STATIC"; return false; }
        for (size_t k = 0; k < j; ++k) if (cv_reg[k] == r) { why = "control curve: a register is named twice"; return false; }
    }
    return true;
}
// The curves from period s0 of the call on.
CurveBlock curves_from(const CurveBlock& cb, int n, size_t s0, size_t N) {
    CurveBlock r = cb;
    for (int j = 0; j < n; ++j) r.p[j] = cb.p[j] + (cb.bcast[j] ? s0 : s0 * N);
    return r;
}
struct CurveRows { CurveBlock cv; int reg[FX8010_MAX_CONTROL_CURVES]; int n; };

// While periods with curves on `regs` run, those registers hold no one value: nothing may fold them (interpreter encoding, plain
// translation — a folded STATIC voids it, once).  Afterwards they hold the last period's values, which the host does not know: still not uniform.
void curves_arm(fx8010_gpu* h, const std::vector<int>& regs) {
    for (int r : regs) {
        h->reg_uniform[r] = 0;
        if (h->enc_sensitive[r]) h->encode_dirty = true;
        tr_touch(h, r);
    }
}

// The preamble of both curve calls (device and host values): checks the list and copies it into rows — FX8010_ERR_ARG changes and
// queues nothing.  `arm`: the call will run periods (curves_arm).  h->tr_cv is keyed to this curve set.
template <class Curve>
int curves_begin(fx8010_gpu* h, const Curve* curves, int n_curves, const float* const Curve::*values, bool arm, CurveRows& rows) {
    if (n_curves < 0 || n_curves > FX8010_MAX_CONTROL_CURVES || (n_curves > 0 && !curves))
        return fail(h, FX8010_ERR_ARG, "the curve list is NULL or the curve count outside 0..8");
    std::vector<int> regs((size_t)n_curves);
    std::vector<uint8_t> bc((size_t)n_curves);
    rows = {};
    rows.n = n_curves;
    for (int j = 0; j < n_curves; ++j) {
        if (!(curves[j].*values)) return fail(h, FX8010_ERR_ARG, "control curve: the values pointer is NULL");
        regs[j] = rows.reg[j] = curves[j].reg_index;
        bc[j] = curves[j].broadcast ? 1 : 0;
        rows.cv.p[j] = curves[j].*values; rows.cv.bcast[j] = bc[j];
    }
    {
        std::string why;
        if (!curves_valid(h->regs, regs, why)) return fail(h, FX8010_ERR_ARG, why);
    }
    if (!arm || n_curves == 0) return FX8010_OK;
    curves_arm(h, regs);
    if (h->tr_cv.cv_reg != regs || h->tr_cv.cv_bcast != bc) {
        tr_reset(h, h->tr_cv);
        h->tr_cv.cv_reg = regs; h->tr_cv.cv_bcast = bc; h->tr_cv.serial = false;
    }
    return FX8010_OK;
}
// Period s of every curve into its register row: the per-period path of fx8010_gpu_process_batch_curves (grid.y = curve).
__global__ void fx_curve_rows_kernel(float* __restrict__ gpr, const CurveRows rows, int s, int N) {
    const int j = blockIdx.y;
    const float* p = rows.cv.p[j];
    float* dst = gpr + (size_t)rows.reg[j] * N;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x)
        dst[i] = rows.cv.bcast[j] ? p[s] : p[(size_t)s * N + i];
}

// ns periods of one block with the curves of `rows`, the way route() decides.
int launch_curves(fx8010_gpu* h, const float* d_in, float* d_out, size_t cs, int ns, const CurveRows& rows, cudaStream_t st) {
    const size_t N = (size_t)h->N;
    const Route r = route(h, &d_in, &d_out, 1, cs, cs, ns, &rows.cv);
    if (r.path == PATH_SPLIT)
        return split_periods(h, &d_in, &d_out, 1, ns, r.len, false, [&](const float* in, float* out, int k, int s0, bool) {
            CurveRows piece = rows;
            piece.cv = curves_from(rows.cv, rows.n, (size_t)s0, N);
            return launch_curves(h, in, out, cs, k, piece, st);
        });
    if (r.path == PATH_TR_SERIAL || r.path == PATH_TR_STREAM) {
        Launch L = {};
        const int rc = r.path == PATH_TR_SERIAL ? tr_launch(h, h->tr_cv, d_in, d_out, cs, cs, ns, st, &rows.cv, L)
                                                : tr_sl_launch(h, h->tr_cv, &d_in, &d_out, 1, cs, cs, ns, st, 0, L, &rows.cv);
        if (rc) return rc;
        record_launch(h, r.path, L, 1, ns, 0, 0, true, nullptr, st);
        return FX8010_OK;
    }
    // Per-period path (correctness, not speed): no translated kernel for this curve set, or the launch does not qualify.  Each period
    // is one copy of the curves' values into the register rows and one ordinary one-period launch.
    for (int s = 0; s < ns; ++s) {
        fx_curve_rows_kernel<<<dim3((unsigned)std::min<size_t>(1024, (N + 255) / 256), (unsigned)rows.n), 256, 0, st>>>(h->d_gpr, rows, s, (int)N);
        h->info.kernel_launches++;
        FX_CUDA(h, cudaGetLastError());
        h->chain.clear();
        const int rc = launch_block(h, d_in ? d_in + (size_t)s * N : nullptr, d_out + (size_t)s * N, cs, cs, 1, st);
        if (rc) return rc;
    }
    return FX8010_OK;
}

int sync_all(fx8010_gpu* h) {
    FX_CUDA(h, cudaSetDevice(h->device));
    if (h->has_last && cudaStreamSynchronize(h->last_stream) != cudaSuccess) {   // (a caller's stream that no longer exists: wait for the device instead)
        cudaGetLastError();
        FX_CUDA(h, cudaDeviceSynchronize());
        h->has_last = false;
    }
    h->chain.clear();
    FX_CUDA(h, cudaStreamSynchronize(h->s_comp));
    FX_CUDA(h, cudaStreamSynchronize(h->s_h2d));
    FX_CUDA(h, cudaStreamSynchronize(h->s_d2h));
    FX_CUDA(h, cudaStreamSynchronize(nullptr));
    return FX8010_OK;
}

// One fused kernel of a chain and what it was generated from.
struct ChainKernel {
    Translation tr;                                  // the fused kernel (kind 3) ...
    std::vector<ChainCurve> cvs;                     // ... reading these control curves (none: the plain kernel) ...
    std::vector<unsigned long long> epoch;           // ... generated while each stage had this tr_epoch ...
    std::vector<std::vector<uint8_t>> folded;        // ... folding these registers of each stage ...
    std::vector<std::vector<float>> fold_value;      // ... with these values
};

}  // namespace

// A chain of stages (fx8010_chain_*): handles of one device, instance count and channel count whose programs run one after another within
// every sample period.  Stateless stages run fused in one translated kernel (fx_translated_chain); anything else runs stage by stage through
// the chain's own intermediate blocks, which is the definition of a chain call.
struct fx8010_chain {
    std::vector<fx8010_gpu*> st;
    int device = 0;
    ChainKernel plain;                               // the fused kernel of fx8010_chain_process_batch
    ChainKernel cv;                                  // the one of fx8010_chain_process_batch_curves, for its most recent curve list
    float* d_mid[2] = {nullptr, nullptr};            // [C][S][N] intermediate blocks of the stage-by-stage path, used alternately
    size_t mid_floats = 0;
    cudaEvent_t ev = nullptr;                        // orders a stage-by-stage call after the previous one's use of d_mid on another stream
    cudaStream_t last_stream = nullptr; bool has_last = false;
    unsigned long long launches = 0;                 // fused launches (plain and with curves)
    int fused_last = 0;
    std::string why;                                 // why the last call (plain or with curves) did not run fused ("" when it did)
    std::string err;
};

namespace {

int chain_fail(fx8010_chain* c, int code, const std::string& msg) {
    c->err = msg;
    return code;
}

// Fused kernel K still computes what its stages would: no stage reloaded, every folded register still holds its folded value in every
// instance.  A register that no longer does is never folded again (as tr_touch decides for a handle's own translation).
bool chain_current(fx8010_chain* c, ChainKernel& K) {
    for (size_t j = 0; j < c->st.size(); ++j) {
        fx8010_gpu* h = c->st[j];
        if (h->tr_epoch != K.epoch[j]) return false;
        if (j >= K.folded.size()) continue;
        for (size_t r = 0; r < K.folded[j].size(); ++r) {
            if (!K.folded[j][r]) continue;
            uint32_t a, b;
            memcpy(&a, &K.fold_value[j][r], 4); memcpy(&b, &h->reg_value[r], 4);
            if (h->reg_uniform[r] && a == b) continue;
            h->tr_volatile[r] = 1;
            return false;
        }
    }
    return true;
}

// Whether fused kernel K is loaded for the chain's current stages (tr_obtain in stage 0's translation mode); `why` says why not.
bool chain_ready(fx8010_chain* c, ChainKernel& K, bool may_wait, std::string& why) {
    fx8010_gpu* h0 = c->st[0];
    if (!chain_current(c, K)) {
        tr_reset(c->device, K.tr);
        K.folded.clear(); K.fold_value.clear();
        for (size_t j = 0; j < c->st.size(); ++j) K.epoch[j] = c->st[j]->tr_epoch;
    }
    if (h0->use_translate == 0) { why = "translation is off on stage 0 (FX8010_OPT_TRANSLATE 0)"; return false; }
    if (K.tr.state == 0)
        for (size_t j = 0; j < c->st.size(); ++j)
            if (!c->st[j]->stateless) { K.tr.state = -1; K.tr.error = "stage " + std::to_string(j) + " carries state across sample periods"; break; }
    const bool ok = tr_obtain(c->device, h0->use_translate, h0->kc_env_dir, K.tr, [&](std::string& src, std::string&) {
        src = tr_generate_chain(std::vector<const fx8010_gpu*>(c->st.begin(), c->st.end()), K.folded, K.cvs);
        K.fold_value.clear();
        for (fx8010_gpu* h : c->st) K.fold_value.push_back(h->reg_value);
        return true;
    }, may_wait);
    why = ok ? "" : (K.tr.state == 1 ? "the chain kernel is compiling" : K.tr.error);
    return ok;
}

// One launch of fused kernel K (with the call's curves cv for the curve kernel): every stage's earlier work comes first (order_on), and the
// kernel waits at its start and never lets a later launch start early, so afterwards no stage has a late-waiting launch outstanding (each
// one's chain is empty).
int chain_launch(fx8010_chain* c, const ChainKernel& K, const float* d_in, float* d_out, int n, cudaStream_t stream, const CurveBlock* cv = nullptr) {
    for (fx8010_gpu* h : c->st) {
        const int rc = order_on(h, stream);
        if (rc) return chain_fail(c, rc, h->err);
    }
    fx8010_gpu* h0 = c->st[0];
    struct Stage { float* gpr; double* acc; float* latch; unsigned long long* counts; unsigned int* flags; const TableEntry* tabs; };
    struct { Stage s[FX8010_MAX_CHAIN_STAGES]; } stages = {};
    for (size_t j = 0; j < c->st.size(); ++j) {
        fx8010_gpu* h = c->st[j];
        stages.s[j] = Stage{h->d_gpr, h->d_acc, h->d_latch, h->d_counts, h->d_flags, h->d_tabs};
    }
    Launch L = {};
    L.K = 4; L.B = h0->tune_B ? h0->tune_B : 128; L.P = 1;
    L.grid_x = (h0->N / L.K + L.B - 1) / L.B;
    sl_segments(h0, L.grid_x, L.B, n, 1, L.seg_len, L.n_seg);
    size_t cs = (size_t)n * h0->N;
    const void* inp = d_in; void* outp = d_out;
    int n_ = n, N_ = h0->N;
    CurveBlock cvb = cv ? *cv : CurveBlock{};
    void* args[] = {&stages, &inp, &outp, &cs, &cs, &n_, &L.seg_len, &N_, &cvb};
    const int rc = tr_drive(h0, K.tr, L, 1, stream, args);
    if (rc) return chain_fail(c, rc, h0->err);
    for (fx8010_gpu* h : c->st) { h->chain.clear(); h->tram_periods += (unsigned long long)n; }
    c->launches++;
    return FX8010_OK;
}

// Stage by stage: fx8010_gpu_process_batch of every stage on `stream`, stage j writing the intermediate block stage j + 1 reads; a stage
// with curves in `cvs` (per stage, as the chain call lists them) takes fx8010_gpu_process_batch_curves and routes them itself.
int chain_sequential(fx8010_chain* c, const float* d_in, float* d_out, int n, cudaStream_t stream,
                     const std::vector<std::vector<fx8010_control_curve>>* cvs = nullptr) {
    const size_t ns = c->st.size(), need = (size_t)c->st[0]->C * n * c->st[0]->N;
    if (ns > 1 && need > c->mid_floats) {                 // (cudaFree waits for the device: no earlier call still uses the old blocks)
        cudaFree(c->d_mid[0]); cudaFree(c->d_mid[1]); c->d_mid[0] = c->d_mid[1] = nullptr; c->mid_floats = 0;
        for (int b = 0; b < 2; ++b) {
            const cudaError_t e = cudaMalloc(&c->d_mid[b], sizeof(float) * need);
            if (e != cudaSuccess) return chain_fail(c, FX8010_ERR_CUDA, std::string("chain intermediate blocks: ") + cudaGetErrorString(e));
        }
        c->mid_floats = need;
    }
    if (ns > 1 && c->has_last && c->last_stream != stream) {
        if (cudaEventRecord(c->ev, c->last_stream) == cudaSuccess) {
            const cudaError_t e = cudaStreamWaitEvent(stream, c->ev, 0);
            if (e != cudaSuccess) return chain_fail(c, FX8010_ERR_CUDA, std::string("cudaStreamWaitEvent: ") + cudaGetErrorString(e));
        } else {
            cudaGetLastError();                              // that stream no longer exists: everything on the device comes first
            const cudaError_t e = cudaDeviceSynchronize();
            if (e != cudaSuccess) return chain_fail(c, FX8010_ERR_CUDA, std::string("cudaDeviceSynchronize: ") + cudaGetErrorString(e));
        }
    }
    for (size_t j = 0; j < ns; ++j) {
        const float* in = j ? c->d_mid[(j - 1) & 1] : d_in;
        float* out = j + 1 == ns ? d_out : c->d_mid[j & 1];
        // A stage's launch may postpone its wait only when it follows that handle's own launches (launch_blocks); here it follows the
        // previous stage, which writes its input, so every stage launch waits at its start (STREAM_EXCLUSIVE set on a stage included).
        c->st[j]->chain.clear();
        const int rc = cvs && !(*cvs)[j].empty()
                           ? fx8010_gpu_process_batch_curves(c->st[j], in, out, n, (*cvs)[j].data(), (int)(*cvs)[j].size(), stream)
                           : fx8010_gpu_process_batch(c->st[j], in, out, n, stream);
        if (rc) return chain_fail(c, rc, "stage " + std::to_string(j) + ": " + c->st[j]->err);
    }
    c->last_stream = stream; c->has_last = true;
    return FX8010_OK;
}

// Some instruction of h's program preloads an INPUT register (reads the call's input).
bool reads_input(const fx8010_gpu* h) {
    for (const fx8010_instr& in : h->instrs) {
        bool pa, px, py; int nz;
        pre_targets(h, in, pa, px, py, nz);
        if (pa || px || py) return true;
    }
    return false;
}

// What every chain call checks before it queues anything (device buffers, io = "d_", or host buffers, io = ""): every stage has a program,
// `out` is given and the count not negative, `in` is given when stage 0 reads an input, and — with n_curves != 0 — the curve list: a count
// of 0..8, a list, and for every stage its own curves as fx8010_gpu_process_batch_curves checks them.  per_stage gets each stage's curves.
template <class Curve>
int chain_check(fx8010_chain* c, const char* io, const float* in, const float* out, int n_samples, const Curve* curves, int n_curves,
                const float* const Curve::*values, std::vector<std::vector<fx8010_control_curve>>& per_stage) {
    const int NS = (int)c->st.size();
    for (int j = 0; j < NS; ++j)
        if (!c->st[j]->loaded) return chain_fail(c, FX8010_ERR_NO_PROGRAM, "stage " + std::to_string(j) + " has no program");
    if (!out || n_samples < 0) return chain_fail(c, FX8010_ERR_ARG, std::string(io) + "out is NULL or n_samples negative");
    if (!in && reads_input(c->st[0])) return chain_fail(c, FX8010_ERR_ARG, std::string(io) + "in is NULL but stage 0 reads an input");
    per_stage.assign((size_t)NS, {});
    if (n_curves == 0) return FX8010_OK;
    // The whole list is checked, for every stage, before any stage runs (the stage-by-stage path must not run stage 0 and then refuse stage 2).
    if (n_curves < 0 || n_curves > FX8010_MAX_CONTROL_CURVES || !curves)
        return chain_fail(c, FX8010_ERR_ARG, "the curve list is NULL or the curve count outside 0..8");
    for (int q = 0; q < n_curves; ++q) {
        const Curve& cv = curves[q];
        if (cv.stage < 0 || cv.stage >= NS) return chain_fail(c, FX8010_ERR_ARG, "control curve " + std::to_string(q) + ": stage index out of range");
        per_stage[cv.stage].push_back(fx8010_control_curve{cv.reg_index, cv.broadcast ? 1 : 0, cv.*values});
    }
    for (int j = 0; j < NS; ++j) {
        CurveRows rows;
        if (curves_begin(c->st[j], per_stage[j].data(), (int)per_stage[j].size(), &fx8010_control_curve::d_values, false, rows))
            return chain_fail(c, FX8010_ERR_ARG, "stage " + std::to_string(j) + ": " + c->st[j]->err);
    }
    return FX8010_OK;
}

}  // namespace

extern "C" {

int fx8010_chain_create(fx8010_gpu* const* stages, int n_stages, fx8010_chain** out) {
    if (!out) return fail(nullptr, FX8010_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!stages || n_stages < 1 || n_stages > FX8010_MAX_CHAIN_STAGES) return fail(nullptr, FX8010_ERR_ARG, "the stage count must be 1..FX8010_MAX_CHAIN_STAGES");
    for (int j = 0; j < n_stages; ++j) {
        if (!stages[j]) return fail(nullptr, FX8010_ERR_ARG, "stage " + std::to_string(j) + " is NULL");
        for (int k = 0; k < j; ++k) if (stages[k] == stages[j]) return fail(nullptr, FX8010_ERR_ARG, "a handle appears twice in the chain");
        if (stages[j]->device != stages[0]->device || stages[j]->N != stages[0]->N || stages[j]->C != stages[0]->C)
            return fail(nullptr, FX8010_ERR_ARG, "the stages differ in device, instance count or channel count");
    }
    cudaError_t e = cudaSetDevice(stages[0]->device);
    fx8010_chain* c = new fx8010_chain();
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev, cudaEventDisableTiming);
    if (e != cudaSuccess) { delete c; return fail(nullptr, FX8010_ERR_CUDA, std::string("chain: ") + cudaGetErrorString(e)); }
    c->st.assign(stages, stages + n_stages);
    c->device = stages[0]->device;
    for (ChainKernel* K : {&c->plain, &c->cv}) {
        K->tr.kind = 3;
        for (fx8010_gpu* h : c->st) K->epoch.push_back(h->tr_epoch);
    }
    *out = c;
    return FX8010_OK;
}

void fx8010_chain_destroy(fx8010_chain* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    // A host-buffer call leaves every stage's latest work on stage 0's compute stream, which dies with stage 0: once it has drained, no
    // stage refers to it any more, so that the handles may be destroyed in any order.
    for (fx8010_gpu* h : c->st)
        if (h != c->st[0] && h->has_last && h->last_stream == c->st[0]->s_comp) {
            cudaStreamSynchronize(h->last_stream);
            h->has_last = false;
        }
    cudaFree(c->d_mid[0]); cudaFree(c->d_mid[1]);            // (waits for the device)
    if (c->ev) cudaEventDestroy(c->ev);
    tr_detach(c->device, c->plain.tr);
    tr_detach(c->device, c->cv.tr);
    delete c;
}

int fx8010_chain_process_batch(fx8010_chain* c, const float* d_in, float* d_out, int n_samples, void* stream) {
    if (!c) return FX8010_ERR_ARG;
    std::vector<std::vector<fx8010_control_curve>> per_stage;
    const int rc = chain_check(c, "d_", d_in, d_out, n_samples, (const fx8010_chain_curve*)nullptr, 0, &fx8010_chain_curve::d_values, per_stage);
    if (rc) return rc;
    if (cudaSetDevice(c->device) != cudaSuccess) return chain_fail(c, FX8010_ERR_CUDA, "cudaSetDevice failed");
    if (n_samples == 0) return FX8010_OK;
    cudaStream_t st = (cudaStream_t)stream;
    fx8010_gpu* h0 = c->st[0];
    const size_t cs = (size_t)n_samples * h0->N;
    bool fused = false;
    if (c->st.size() == 1) c->why = "a chain of one stage is that stage's process_batch";
    else if (h0->N % 4) c->why = "the instance count is not a multiple of 4";
    else if (!io_aligned(h0, 16, &d_in, &d_out, 1, cs, cs, n_samples)) c->why = "a buffer is not 16-byte aligned";
    else fused = chain_ready(c, c->plain, true, c->why);
    c->fused_last = fused ? 1 : 0;
    return fused ? chain_launch(c, c->plain, d_in, d_out, n_samples, st) : chain_sequential(c, d_in, d_out, n_samples, st);
}

int fx8010_chain_process_batch_curves(fx8010_chain* c, const float* d_in, float* d_out, int n_samples, const fx8010_chain_curve* curves,
                                      int n_curves, void* stream) {
    if (!c) return FX8010_ERR_ARG;
    if (n_curves == 0) return fx8010_chain_process_batch(c, d_in, d_out, n_samples, stream);
    std::vector<std::vector<fx8010_control_curve>> per_stage;
    const int rc = chain_check(c, "d_", d_in, d_out, n_samples, curves, n_curves, &fx8010_chain_curve::d_values, per_stage);
    if (rc) return rc;
    const int NS = (int)c->st.size();
    std::vector<ChainCurve> key;
    CurveBlock cb = {};
    for (int q = 0; q < n_curves; ++q) {
        const fx8010_chain_curve& cv = curves[q];
        key.push_back(ChainCurve{cv.stage, cv.reg_index, (uint8_t)(cv.broadcast ? 1 : 0)});
        cb.p[q] = cv.d_values; cb.bcast[q] = cv.broadcast ? 1 : 0;
    }
    if (cudaSetDevice(c->device) != cudaSuccess) return chain_fail(c, FX8010_ERR_CUDA, "cudaSetDevice failed");
    if (n_samples == 0) return FX8010_OK;
    for (int j = 0; j < NS; ++j) {                          // (as fx8010_gpu_process_batch_curves leaves each stage)
        std::vector<int> regs;
        for (const fx8010_control_curve& cv : per_stage[j]) regs.push_back(cv.reg_index);
        curves_arm(c->st[j], regs);
    }
    if (c->cv.cvs != key) {                                 // another curve list: another kernel
        tr_reset(c->device, c->cv.tr);
        c->cv.folded.clear(); c->cv.fold_value.clear();
        c->cv.cvs = key;
    }
    cudaStream_t st = (cudaStream_t)stream;
    fx8010_gpu* h0 = c->st[0];
    const size_t cs = (size_t)n_samples * h0->N;
    bool fused = false;
    if (NS == 1) c->why = "a chain of one stage is that stage's process_batch_curves";
    else if (h0->N % 4) c->why = "the instance count is not a multiple of 4";
    else if (!io_aligned(h0, 16, &d_in, &d_out, 1, cs, cs, n_samples)) c->why = "a buffer is not 16-byte aligned";
    else if (!io_aligned(h0, 16, &d_in, &d_out, 1, cs, cs, n_samples, &cb, n_curves)) c->why = "a curve buffer is not 16-byte aligned";
    else fused = chain_ready(c, c->cv, true, c->why);
    c->fused_last = fused ? 1 : 0;
    return fused ? chain_launch(c, c->cv, d_in, d_out, n_samples, st, &cb) : chain_sequential(c, d_in, d_out, n_samples, st, &per_stage);
}

int fx8010_chain_status(fx8010_chain* c, int* state, int* fused_last, unsigned long long* launches, int* regs_per_thread, int* local_bytes,
                        char* message, size_t message_cap) {
    if (!c) return FX8010_ERR_ARG;
    if (c->plain.tr.state == 1 && cudaSetDevice(c->device) == cudaSuccess) {     // pick up a finished background compilation
        bool loaded = true;
        for (fx8010_gpu* h : c->st) loaded = loaded && h->loaded;
        if (loaded) chain_ready(c, c->plain, false, c->why);
    }
    if (state) *state = c->plain.tr.state;
    if (fused_last) *fused_last = c->fused_last;
    if (launches) *launches = c->launches;
    if (regs_per_thread) *regs_per_thread = c->plain.tr.regs;
    if (local_bytes) *local_bytes = c->plain.tr.local;
    const std::string& m = c->fused_last ? std::string() : c->why;
    if (message && message_cap) { strncpy(message, m.c_str(), message_cap - 1); message[message_cap - 1] = 0; }
    return FX8010_OK;
}

int fx8010_chain_status_curves(fx8010_chain* c, int* state, int* regs_per_thread, int* local_bytes, char* message, size_t message_cap) {
    if (!c) return FX8010_ERR_ARG;
    std::string why = c->cv.tr.state == 1 ? "the chain kernel is compiling" : c->cv.tr.error;
    if (c->cv.tr.state == 1 && cudaSetDevice(c->device) == cudaSuccess) {        // pick up a finished background compilation
        bool loaded = true;
        for (fx8010_gpu* h : c->st) loaded = loaded && h->loaded;
        if (loaded) chain_ready(c, c->cv, false, why);
    }
    if (state) *state = c->cv.tr.state;
    if (regs_per_thread) *regs_per_thread = c->cv.tr.regs;
    if (local_bytes) *local_bytes = c->cv.tr.local;
    if (message && message_cap) { strncpy(message, why.c_str(), message_cap - 1); message[message_cap - 1] = 0; }
    return FX8010_OK;
}

const char* fx8010_chain_last_error(fx8010_chain* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int fx8010_gpu_create(int device, int n_instances, int n_channels, fx8010_gpu** out) {
    if (!out) return fail(nullptr, FX8010_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (n_instances <= 0 || n_channels <= 0 || n_channels > 255 || device < 0 || device >= MAX_DEVICES)
        return fail(nullptr, FX8010_ERR_ARG, "n_instances and n_channels (<= 255) must be positive, device in range");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, FX8010_ERR_CUDA, std::string("no usable CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (device >= count) return fail(nullptr, FX8010_ERR_ARG, "device ordinal out of range");
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(nullptr, FX8010_ERR_CUDA, cudaGetErrorString(e));
    fx8010_gpu* h = new fx8010_gpu();
    h->device = device; h->N = n_instances; h->C = n_channels;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
        h->num_sms = prop.multiProcessorCount;
        h->smem_optin = prop.sharedMemPerBlockOptin - 1024;   // the kernels keep a few hundred bytes of static shared memory
    }
    bool ok = cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < HOST_PIPE_BUFS && ok; ++i)
        ok = cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&h->ev_comp[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&h->ev_d2h[i], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->ev_events, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->ev_order, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaMallocHost(&h->h_prog, sizeof(uint4) * SLOT_WORDS) == cudaSuccess;
    ok = ok && cudaMalloc(&h->d_flags, sizeof(unsigned int)) == cudaSuccess;
    ok = ok && cudaMalloc(&h->d_tabs, sizeof(TableEntry) * 2 * FX8010_TABLE_COUNT * FX8010_TABLE_ENTRIES) == cudaSuccess;
    if (!ok) {
        const std::string msg = std::string("CUDA resource creation failed: ") + cudaGetErrorString(cudaGetLastError());
        fx8010_gpu_destroy(h);
        return fail(nullptr, FX8010_ERR_CUDA, msg);
    }
    h->tune_K = env_int("FX8010_TUNE_K"); h->tune_B = env_int("FX8010_TUNE_B");
    h->tune_seg = env_int("FX8010_TUNE_SEG"); h->tune_sub = env_int("FX8010_TUNE_SUB");
    if (getenv("FX8010_NO_PDL")) h->use_pdl = 0;
    if (getenv("FX8010_NO_FUSE")) h->use_fuse = 0;
    if (getenv("FX8010_NO_PAIRS")) h->use_pairs = 0;
    if (getenv("FX8010_NO_TSPLIT")) h->use_tsplit = 0;
    if (getenv("FX8010_USE_TMA")) h->use_tma = atoi(getenv("FX8010_USE_TMA"));
    if (getenv("FX8010_NO_STATELESS")) h->use_sl = 0;
    if (getenv("FX8010_NO_SHORT")) h->use_short = 0;
    if (getenv("FX8010_NO_CARRY")) h->use_carry = 0;
    if (getenv("FX8010_NO_TRAM_IM")) h->use_tram_im = 0;
    if (getenv("FX8010_NO_SPLIT")) h->use_split = 0;
    if (getenv("FX8010_TR_RECUR")) h->tr_recurrences = atoi(getenv("FX8010_TR_RECUR"));
    h->kc_env_dir = kc_env_dir();
    if (getenv("FX8010_TRANSLATE")) h->use_translate = std::min(2, std::max(0, atoi(getenv("FX8010_TRANSLATE"))));
    h->tune_P = env_int("FX8010_TUNE_P");
    h->tune_M = env_int("FX8010_TUNE_M");
    h->tune_chunk = env_int("FX8010_TUNE_CHUNK");
    if (h->tune_chunk & (h->tune_chunk - 1) || h->tune_chunk > MAX_CHUNK) h->tune_chunk = 0;
    if (h->tune_M != 1 && h->tune_M != 2 && h->tune_M != 4 && h->tune_M != 8 && h->tune_M != 16 && h->tune_M != 32 && h->tune_M != 64) h->tune_M = 0;
    if (h->tune_K != 1 && h->tune_K != 2 && h->tune_K != 4) h->tune_K = 0;
    if (h->tune_B != 32 && h->tune_B != 64 && h->tune_B != 128 && h->tune_B != 256) h->tune_B = 0;
    *out = h;
    return FX8010_OK;
}

void fx8010_gpu_destroy(fx8010_gpu* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    sync_all(h);
    tr_reset(h);
    free_state(h);
    cudaFree(h->d_flags); cudaFree(h->d_tabs); cudaFree(h->d_events); cudaFree(h->d_planar_in); cudaFree(h->d_planar_out);
    if (h->ev_events) cudaEventDestroy(h->ev_events);
    if (h->ev_order) cudaEventDestroy(h->ev_order);
    for (int i = 0; i < HOST_PIPE_BUFS; ++i) {
        cudaFree(h->d_stage_in[i]); cudaFree(h->d_stage_out[i]); cudaFree(h->d_bcast[i]); cudaFree(h->d_curve_stage[i]);
        if (h->ev_h2d[i]) cudaEventDestroy(h->ev_h2d[i]);
        if (h->ev_comp[i]) cudaEventDestroy(h->ev_comp[i]);
        if (h->ev_d2h[i]) cudaEventDestroy(h->ev_d2h[i]);
    }
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_comp) cudaStreamDestroy(h->s_comp);
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    if (h->h_prog) cudaFreeHost(h->h_prog);
    {
        std::lock_guard<std::mutex> lk(g_dev_mutex[h->device]);
        arena_release(h);
    }
    delete h;
}

int fx8010_gpu_load_program(fx8010_gpu* h, const fx8010_program_image* im) {
    if (!h) return FX8010_ERR_ARG;
    if (!im || !im->instrs || !im->regs || !im->log_tables || !im->exp_tables) return fail(h, FX8010_ERR_ARG, "image or one of its arrays is NULL");
    if (im->n_instrs <= 0 || im->n_regs <= 0) return fail(h, FX8010_ERR_PROGRAM, "empty program (the reference would spin forever, SURVEY U10)");
    if (im->n_instrs > MAX_INSTR) return fail(h, FX8010_ERR_CAPACITY, "more than FX8010_MAX_INSTRUCTIONS instructions");
    if (im->n_regs > 65535) return fail(h, FX8010_ERR_CAPACITY, "more than 65535 registers");
    bool has_end = false, use_i = false, use_x = false;
    for (int i = 0; i < im->n_instrs; ++i) {
        const fx8010_instr& in = im->instrs[i];
        if (in.opcode < 0 || in.opcode >= FX_NUM_OPCODES) return fail(h, FX8010_ERR_PROGRAM, "opcode out of range");
        if (in.r < 0 || in.r >= im->n_regs || in.a < 0 || in.a >= im->n_regs || in.x < 0 || in.x >= im->n_regs ||
            in.y < 0 || in.y >= im->n_regs) return fail(h, FX8010_ERR_PROGRAM, "operand register index out of range");
        if (in.opcode == FX_END) has_end = true;
        const int t = im->regs[in.r].type;
        if (in.opcode == FX_IDELAY && (t == FX_REG_READ || t == FX_REG_WRITE)) use_i = true;
        if (in.opcode == FX_XDELAY && (t == FX_REG_READ || t == FX_REG_WRITE)) use_x = true;
    }
    if (!has_end) return fail(h, FX8010_ERR_PROGRAM, "program has no END (the reference would spin forever)");
    for (int r = 0; r < im->n_regs; ++r)
        if (im->regs[r].io_index < 0 || im->regs[r].io_index >= h->C) return fail(h, FX8010_ERR_PROGRAM, "I/O index outside the channel count");
    if ((use_i && im->itram_size <= 0) || (use_x && im->xtram_size <= 0))
        return fail(h, FX8010_ERR_PROGRAM, "IDELAY/XDELAY without a declared TRAM size (SURVEY U4)");
    if (im->itram_size > (1 << 24) || im->xtram_size > (1 << 24)) return fail(h, FX8010_ERR_CAPACITY, "TRAM size above 2^24");

    FX_CUDA(h, cudaSetDevice(h->device));
    const int rc = sync_all(h);
    if (rc) return rc;
    {
        std::lock_guard<std::mutex> lk(g_dev_mutex[h->device]);
        arena_release(h);          // the new program gets its constant-memory range at its first launch
    }
    h->loaded = false;
    free_state(h);
    h->instrs.assign(im->instrs, im->instrs + im->n_instrs);
    h->regs.assign(im->regs, im->regs + im->n_regs);
    h->itram_size = use_i ? im->itram_size : 0;
    h->xtram_size = use_x ? im->xtram_size : 0;
    const size_t N = (size_t)h->N, nr = (size_t)im->n_regs;

    // LOG/EXP tables: T[i] and the interpolation quotient (T[i+1]-T[i])/(x2-x1), evaluated here with
    // the same IEEE double operations as linearInterpolate (source/FX8010.cpp:285-293); T[64] = 0 (U5).
    h->h_tabs.resize((size_t)2 * FX8010_TABLE_COUNT * FX8010_TABLE_ENTRIES);
    const double x_min = -1.0, x_max = 1.0;
    const double step = (x_max - x_min) / (double)(FX8010_TABLE_ENTRIES - 1);
    for (int op = 0; op < 2; ++op)
        for (int t = 0; t < FX8010_TABLE_COUNT; ++t) {
            const double* T = (op == 0 ? im->log_tables : im->exp_tables) + (size_t)t * FX8010_TABLE_ENTRIES;
            for (int i = 0; i < FX8010_TABLE_ENTRIES; ++i) {
                const volatile double x1 = x_min + i * step;
                const volatile double x2 = x_min + (i + 1) * step;
                const volatile double y1 = T[i];
                const volatile double y2 = (i + 1 < FX8010_TABLE_ENTRIES) ? T[i + 1] : 0.0;
                const volatile double num = y2 - y1, den = x2 - x1;
                TableEntry e; e.y1 = y1; e.slope = num / den;
                h->h_tabs[((size_t)op * FX8010_TABLE_COUNT + t) * FX8010_TABLE_ENTRIES + i] = e;
            }
        }
    FX_CUDA(h, cudaMemcpy(h->d_tabs, h->h_tabs.data(), sizeof(TableEntry) * h->h_tabs.size(), cudaMemcpyHostToDevice));

    // capacity check before allocating the rings
    size_t free_b = 0, total_b = 0;
    FX_CUDA(h, cudaMemGetInfo(&free_b, &total_b));
    const size_t need = N * (4 * nr + 8 + 8 + 4 * (size_t)h->C + 16 + 8) + 4 * N * ((size_t)h->itram_size + (size_t)h->xtram_size);
    if (need + (64u << 20) > free_b) return fail(h, FX8010_ERR_CAPACITY, "per-instance state (registers + TRAM rings) does not fit in device memory");

    FX_CUDA(h, cudaMalloc(&h->d_gpr, sizeof(float) * nr * N));
    FX_CUDA(h, cudaMalloc(&h->d_acc, sizeof(double) * N));
    FX_CUDA(h, cudaMalloc(&h->d_lfsr, sizeof(uint32_t) * 2 * N));
    FX_CUDA(h, cudaMalloc(&h->d_latch, sizeof(float) * (size_t)h->C * N));
    FX_CUDA(h, cudaMalloc(&h->d_ptrs, sizeof(int32_t) * 4 * N));
    FX_CUDA(h, cudaMalloc(&h->d_counts, sizeof(unsigned long long) * N));
    if (h->itram_size) { FX_CUDA(h, cudaMalloc(&h->d_itram, sizeof(float) * (size_t)h->itram_size * N)); FX_CUDA(h, cudaMemset(h->d_itram, 0, sizeof(float) * (size_t)h->itram_size * N)); }
    if (h->xtram_size) { FX_CUDA(h, cudaMalloc(&h->d_xtram, sizeof(float) * (size_t)h->xtram_size * N)); FX_CUDA(h, cudaMemset(h->d_xtram, 0, sizeof(float) * (size_t)h->xtram_size * N)); }
    // state of a freshly constructed + loaded reference object
    for (size_t r = 0; r < nr; ++r) {
        fx_fill_kernel<<<(unsigned)((N + 255) / 256), 256>>>(h->d_gpr + r * N, im->regs[r].init_value, (int)N);
        h->info.kernel_launches++;
    }
    FX_CUDA(h, cudaGetLastError());
    FX_CUDA(h, cudaMemset(h->d_acc, 0, sizeof(double) * N));
    FX_CUDA(h, cudaMemset(h->d_latch, 0, sizeof(float) * (size_t)h->C * N));
    FX_CUDA(h, cudaMemset(h->d_ptrs, 0, sizeof(int32_t) * 4 * N));
    FX_CUDA(h, cudaMemset(h->d_counts, 0, sizeof(unsigned long long) * N));
    FX_CUDA(h, cudaMemset(h->d_flags, 0, sizeof(unsigned int)));
    {
        std::vector<uint32_t> seeds(2 * N);
        for (size_t i = 0; i < N; ++i) { seeds[i] = FX8010_LFSR_SEED1; seeds[N + i] = FX8010_LFSR_SEED2; }
        FX_CUDA(h, cudaMemcpy(h->d_lfsr, seeds.data(), sizeof(uint32_t) * 2 * N, cudaMemcpyHostToDevice));
    }
    h->reg_uniform.assign(nr, 1);
    h->reg_value.resize(nr);
    for (size_t r = 0; r < nr; ++r) h->reg_value[r] = im->regs[r].init_value;
    h->tr_volatile.assign(nr, 0);
    tr_reset(h);
    analyse(h);
    FX_CUDA(h, cudaMalloc(&h->d_wb, sizeof(uint32_t) * std::max<size_t>(1, h->wb.size())));
    FX_CUDA(h, cudaMalloc(&h->d_latch_ch, sizeof(uint32_t) * 256));
    FX_CUDA(h, cudaMalloc(&h->d_sl_load, sizeof(uint2) * std::max<size_t>(1, nr)));
    FX_CUDA(h, cudaMalloc(&h->d_sl_wb, sizeof(uint2) * std::max<size_t>(1, nr)));
    FX_CUDA(h, cudaMalloc(&h->d_reg_map, sizeof(uint32_t) * h->reg_map.size()));
    FX_CUDA(h, cudaMalloc(&h->d_load_rows, sizeof(uint32_t) * std::max<size_t>(1, h->load_rows.size())));
    if (!h->load_rows.empty()) FX_CUDA(h, cudaMemcpy(h->d_load_rows, h->load_rows.data(), sizeof(uint32_t) * h->load_rows.size(), cudaMemcpyHostToDevice));
    FX_CUDA(h, cudaMemcpy(h->d_reg_map, h->reg_map.data(), sizeof(uint32_t) * h->reg_map.size(), cudaMemcpyHostToDevice));
    if (!h->wb.empty()) FX_CUDA(h, cudaMemcpy(h->d_wb, h->wb.data(), sizeof(uint32_t) * h->wb.size(), cudaMemcpyHostToDevice));
    FX_CUDA(h, cudaDeviceSynchronize());
    h->encode_dirty = true;
    h->loaded = true; h->tram_ptrs_pristine = true; h->tram_periods = 0; h->plan_key = PlanKey();
    return FX8010_OK;
}

#define FX_NEED_PROGRAM(h)                                                                  \
    if (!h) return FX8010_ERR_ARG;                                                         \
    if (!h->loaded) return fail(h, FX8010_ERR_NO_PROGRAM, "no program loaded (SURVEY U10)"); \
    FX_CUDA(h, cudaSetDevice(h->device));

int fx8010_gpu_set_controls(fx8010_gpu* h, int reg, const float* values, int broadcast) {
    FX_NEED_PROGRAM(h);
    if (!values || reg < 0 || reg >= (int)h->regs.size()) return fail(h, FX8010_ERR_ARG, "bad register index or NULL values");
    const int rc = sync_all(h);
    if (rc) return rc;
    float* dst = h->d_gpr + (size_t)reg * h->N;
    if (broadcast) {
        fx_fill_kernel<<<(h->N + 255) / 256, 256>>>(dst, values[0], h->N);
        h->info.kernel_launches++;
        FX_CUDA(h, cudaGetLastError());
        FX_CUDA(h, cudaStreamSynchronize(nullptr));
        h->reg_uniform[reg] = 1; h->reg_value[reg] = values[0];
    } else {
        FX_CUDA(h, cudaMemcpy(dst, values, sizeof(float) * h->N, cudaMemcpyHostToDevice));
        h->reg_uniform[reg] = 0;
    }
    if (h->enc_sensitive[reg]) h->encode_dirty = true;
    tr_touch(h, reg);
    return FX8010_OK;
}

int fx8010_gpu_set_controls_device(fx8010_gpu* h, int reg, const float* d_values, void* stream) {
    FX_NEED_PROGRAM(h);
    if (!d_values || reg < 0 || reg >= (int)h->regs.size()) return fail(h, FX8010_ERR_ARG, "bad register index or NULL values");
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = order_on(h, st);
    if (rc) return rc;
    FX_CUDA(h, cudaMemcpyAsync(h->d_gpr + (size_t)reg * h->N, d_values, sizeof(float) * h->N, cudaMemcpyDeviceToDevice, st));
    h->reg_uniform[reg] = 0;
    if (h->enc_sensitive[reg]) h->encode_dirty = true;
    tr_touch(h, reg);
    return FX8010_OK;
}

int fx8010_gpu_get_register(fx8010_gpu* h, int reg, float* out) {
    FX_NEED_PROGRAM(h);
    if (!out || reg < 0 || reg >= (int)h->regs.size()) return fail(h, FX8010_ERR_ARG, "bad register index or NULL out");
    const int rc = sync_all(h);
    if (rc) return rc;
    FX_CUDA(h, cudaMemcpy(out, h->d_gpr + (size_t)reg * h->N, sizeof(float) * h->N, cudaMemcpyDeviceToHost));
    return FX8010_OK;
}

int fx8010_gpu_process_batch(fx8010_gpu* h, const float* d_in, float* d_out, int n_samples, void* stream) {
    FX_NEED_PROGRAM(h);
    if (!d_out || n_samples < 0) return fail(h, FX8010_ERR_ARG, "d_out is NULL or n_samples negative");
    const size_t cs = (size_t)n_samples * h->N;
    // (work this handle queued on another stream — host-buffer batches run on an internal one — comes first: launch_blocks orders it)
    return launch_block(h, d_in, d_out, cs, cs, n_samples, (cudaStream_t)stream);
}

int fx8010_gpu_process_blocks(fx8010_gpu* h, const float* const* d_in, float* const* d_out, int n_blocks, int n_samples, void* stream) {
    FX_NEED_PROGRAM(h);
    if (!d_out || n_samples < 0 || n_blocks < 0) return fail(h, FX8010_ERR_ARG, "d_out is NULL or a count is negative");
    for (int b = 0; b < n_blocks; ++b) if (!d_out[b]) return fail(h, FX8010_ERR_ARG, "d_out holds a NULL block");
    for (int b = 1; d_in && b < n_blocks; ++b)
        if (!d_in[b] != !d_in[0]) return fail(h, FX8010_ERR_ARG, "either every block of a call has an input buffer or none has");
    const size_t cs = (size_t)n_samples * h->N;
    std::vector<const float*> no_in;
    if (!d_in) { no_in.assign((size_t)std::max(1, n_blocks), nullptr); d_in = no_in.data(); }
    return launch_blocks(h, d_in, d_out, n_blocks, cs, cs, n_samples, (cudaStream_t)stream, false);
}

int fx8010_gpu_set_option(fx8010_gpu* h, int option, int value) {
    if (!h) return FX8010_ERR_ARG;
    if (option == FX8010_OPT_STREAM_EXCLUSIVE) { h->stream_exclusive = value ? 1 : 0; h->chain.clear(); return FX8010_OK; }
    if (option == FX8010_OPT_TRANSLATE) {
        if (value < 0 || value > 2) return fail(h, FX8010_ERR_ARG, "FX8010_OPT_TRANSLATE takes 0, 1 or 2");
        h->use_translate = value;
        for (Translation* T : {&h->tr, &h->tr_cv}) if (T->state < 0) tr_reset(h, *T);      // look again (e.g. after FX8010_NVRTC was set)
        return FX8010_OK;
    }
    return fail(h, FX8010_ERR_ARG, "unknown option");
}

int fx8010_gpu_process_batch_events(fx8010_gpu* h, const float* d_in, float* d_out, int n_samples,
                                    const fx8010_control_event* events, int n_events, void* stream) {
    FX_NEED_PROGRAM(h);
    if (!d_out || n_samples < 0 || n_events < 0 || (n_events > 0 && !events)) return fail(h, FX8010_ERR_ARG, "bad buffer, count or event list");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t N = (size_t)h->N, cs = (size_t)n_samples * N;
    size_t per_instance = 0;
    for (int e = 0; e < n_events; ++e) {
        const fx8010_control_event& ev = events[e];
        if (!ev.values || ev.reg_index < 0 || ev.reg_index >= (int)h->regs.size() || ev.sample < 0 || ev.sample >= std::max(1, n_samples) ||
            (e > 0 && ev.sample < events[e - 1].sample))
            return fail(h, FX8010_ERR_ARG, "control event: bad register, sample out of range or list not sorted by sample");
        if (!ev.broadcast) ++per_instance;
    }
    {
        const int rc = order_on(h, st);
        if (rc) return rc;
    }
    // per-instance value arrays go to the device up front (the caller may reuse them when this call returns)
    if (per_instance * N > h->events_floats) {
        const int rc = sync_all(h);
        if (rc) return rc;
        cudaFree(h->d_events); h->d_events = nullptr; h->events_floats = 0;
        FX_CUDA(h, cudaMalloc(&h->d_events, sizeof(float) * per_instance * N));
        h->events_floats = per_instance * N;
    } else if (per_instance) {                           // an earlier call's copies out of d_events must have been consumed
        FX_CUDA(h, cudaStreamSynchronize(st));
    }
    size_t slot = 0;
    if (per_instance) {                                  // on the copy stream: `st` may be busy with earlier batches
        for (int e = 0; e < n_events; ++e)
            if (!events[e].broadcast)
                FX_CUDA(h, cudaMemcpyAsync(h->d_events + (slot++) * N, events[e].values, sizeof(float) * N, cudaMemcpyHostToDevice, h->s_h2d));
        FX_CUDA(h, cudaEventRecord(h->ev_events, h->s_h2d));
        FX_CUDA(h, cudaStreamWaitEvent(st, h->ev_events, 0));
        FX_CUDA(h, cudaEventSynchronize(h->ev_events)); // the caller's arrays are free again when this call returns
    }
    int e = 0, s0 = 0;
    slot = 0;
    while (true) {
        // changes that take effect before sample s0 (source/main.cpp:109-113: setRegisterValue, then process)
        for (; e < n_events && events[e].sample <= s0; ++e) {
            const fx8010_control_event& ev = events[e];
            float* dst = h->d_gpr + (size_t)ev.reg_index * N;
            if (ev.broadcast) {
                fx_fill_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(dst, ev.values[0], (int)N);
                h->info.kernel_launches++;
                FX_CUDA(h, cudaGetLastError());
                h->reg_uniform[ev.reg_index] = 1; h->reg_value[ev.reg_index] = ev.values[0];
            } else {
                FX_CUDA(h, cudaMemcpyAsync(dst, h->d_events + (slot++) * N, sizeof(float) * N, cudaMemcpyDeviceToDevice, st));
                h->reg_uniform[ev.reg_index] = 0;
            }
            if (h->enc_sensitive[ev.reg_index]) h->encode_dirty = true;
            tr_touch(h, ev.reg_index);
        }
        if (s0 >= n_samples) break;
        const int s1 = (e < n_events) ? std::min(n_samples, (int)events[e].sample) : n_samples;
        const int rc = launch_block(h, d_in ? d_in + (size_t)s0 * N : nullptr, d_out + (size_t)s0 * N, cs, cs, s1 - s0, st);
        if (rc) return rc;
        s0 = s1;
        if (e >= n_events && s0 >= n_samples) break;
    }
    return FX8010_OK;
}

int fx8010_gpu_process_batch_curves(fx8010_gpu* h, const float* d_in, float* d_out, int n_samples,
                                    const fx8010_control_curve* curves, int n_curves, void* stream) {
    FX_NEED_PROGRAM(h);
    if (!d_out || n_samples < 0) return fail(h, FX8010_ERR_ARG, "d_out is NULL or n_samples negative");
    CurveRows rows;
    {
        const int rc = curves_begin(h, curves, n_curves, &fx8010_control_curve::d_values, n_samples > 0, rows);
        if (rc) return rc;
    }
    if (n_samples == 0) return FX8010_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t N = (size_t)h->N, cs = (size_t)n_samples * N;
    if (n_curves == 0) return launch_block(h, d_in, d_out, cs, cs, n_samples, st);
    {
        const int rc = order_on(h, st);
        if (rc) return rc;
    }
    h->chain.clear();                 // every launch of the call waits for its predecessor at its start: a curve may be earlier work's output
    return launch_curves(h, d_in, d_out, cs, n_samples, rows, st);
}

// [C][rows][cols] -> [C][cols][rows], 32 x 32 tiles through shared memory (coalesced on both sides)
static __global__ void fx_transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols) {
    __shared__ float tile[32][33];
    const size_t plane = (size_t)rows * cols * blockIdx.z;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        if (r < rows && c < cols) tile[j][threadIdx.x] = src[plane + (size_t)r * cols + c];
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int c = c0 + j, r = r0 + threadIdx.x;
        if (r < rows && c < cols) dst[plane + (size_t)c * rows + r] = tile[threadIdx.x][j];
    }
}

int fx8010_gpu_process_batch_planar(fx8010_gpu* h, const float* d_in, float* d_out, int n_samples, void* stream) {
    FX_NEED_PROGRAM(h);
    if (!d_out || n_samples < 0) return fail(h, FX8010_ERR_ARG, "d_out is NULL or n_samples negative");
    if (n_samples == 0) return FX8010_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t N = (size_t)h->N, C = (size_t)h->C, S = (size_t)n_samples, need = C * S * N;
    if (need > h->planar_floats) {
        const int rc = sync_all(h);
        if (rc) return rc;
        FX_CUDA(h, cudaStreamSynchronize(st));
        cudaFree(h->d_planar_in); cudaFree(h->d_planar_out); h->d_planar_in = h->d_planar_out = nullptr; h->planar_floats = 0;
        FX_CUDA(h, cudaMalloc(&h->d_planar_in, sizeof(float) * need));
        FX_CUDA(h, cudaMalloc(&h->d_planar_out, sizeof(float) * need));
        h->planar_floats = need;
    }
    {
        const int rc = order_on(h, st);
        if (rc) return rc;
    }
    const dim3 blk(32, 8);
    if (d_in) {     // [C][N][S] -> [C][S][N]
        fx_transpose_kernel<<<dim3((unsigned)((S + 31) / 32), (unsigned)((N + 31) / 32), (unsigned)C), blk, 0, st>>>(d_in, h->d_planar_in, (int)N, (int)S);
        h->info.kernel_launches++;
        FX_CUDA(h, cudaGetLastError());
    }
    const int rc = launch_block(h, d_in ? h->d_planar_in : nullptr, h->d_planar_out, S * N, S * N, n_samples, st);
    if (rc) return rc;
    fx_transpose_kernel<<<dim3((unsigned)((N + 31) / 32), (unsigned)((S + 31) / 32), (unsigned)C), blk, 0, st>>>(h->d_planar_out, d_out, (int)S, (int)N);
    h->info.kernel_launches++;
    FX_CUDA(h, cudaGetLastError());
    return FX8010_OK;
}

// One input value per channel and sample period for ALL instances (a parameter sweep driven by one signal): [rows] -> [rows][N]
static __global__ void fx_broadcast_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int N) {
    const int row = blockIdx.y;
    const float v = src[row];
    float* d = dst + (size_t)row * N;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) d[i] = v;
}

// The compute step of one sub-block of the host pipeline, queued on h->s_comp: `len` periods from d_in (NULL without input) to d_out, channel
// stride cs, with `staged` (NULL without curves) pointing at this sub-block's rows of every curve.
using HostStep = std::function<int(const float* d_in, float* d_out, size_t cs, int len, const CurveRows* staged)>;

// host_n: instances per row of the HOST buffers (>= N: this handle's columns are a slice of a wider [channel][sample][instance] block)
// bcast: `in` holds ONE value per channel and sample period ([channel][sample]); it is copied as it is and spread over the instances on the device
// cv: control curves in HOST memory (checked and armed by the caller): a per-instance curve is [n_samples][host_n] from this handle's first
// column, a broadcast one [n_samples]; each sub-block's rows are staged like its inputs and handed to `step`
// packed: a sub-block's staged channels are len * N floats apart ([channel][len][instance], the layout of a device call on len periods);
// otherwise sub * N
static int process_host_impl(fx8010_gpu* h, const float* in, float* out, int n_samples, bool wait, size_t host_n, bool bcast, const CurveRows* cv,
                             bool packed, const HostStep& step) {
    FX_NEED_PROGRAM(h);
    if (!out || n_samples < 0) return fail(h, FX8010_ERR_ARG, "out is NULL or n_samples negative");
    if (n_samples == 0) return FX8010_OK;
    const size_t N = (size_t)h->N, C = (size_t)h->C;
    if (host_n == 0) host_n = N;
    if (host_n < N) return fail(h, FX8010_ERR_ARG, "host row length below the instance count");
    size_t n_pi = 0, n_bc = 0;                   // per-instance and broadcast curves
    for (int j = 0; cv && j < cv->n; ++j) ++(cv->cv.bcast[j] ? n_bc : n_pi);
    // sub-block: ~16 MiB of samples and per-instance curve values per buffer set
    long sub = h->tune_sub ? h->tune_sub : (long)((16u << 20) / (4 * N * (C + n_pi)));     // (cfg2 end to end: 256-sample sub-blocks 0.446 ms per block, 512 0.396, 1 024 0.380)
    sub = std::max<long>(8, sub / 8 * 8);
    sub = std::min<long>(sub, n_samples);
    const size_t need = C * (size_t)sub * N;
    if (need > h->stage_floats) {
        const int rc = sync_all(h);
        if (rc) return rc;
        for (int i = 0; i < HOST_PIPE_BUFS; ++i) {
            cudaFree(h->d_stage_in[i]); cudaFree(h->d_stage_out[i]);
            h->d_stage_in[i] = h->d_stage_out[i] = nullptr;
        }
        h->stage_floats = 0; h->pipe_seq = 0;
        for (int i = 0; i < HOST_PIPE_BUFS; ++i) {
            FX_CUDA(h, cudaMalloc(&h->d_stage_in[i], sizeof(float) * need));
            FX_CUDA(h, cudaMalloc(&h->d_stage_out[i], sizeof(float) * need));
        }
        h->stage_floats = need;
    }
    if (bcast && in && (size_t)(C * sub) > h->bcast_floats) {
        const int rc = sync_all(h);
        if (rc) return rc;
        for (int i = 0; i < HOST_PIPE_BUFS; ++i) { cudaFree(h->d_bcast[i]); h->d_bcast[i] = nullptr; }
        for (int i = 0; i < HOST_PIPE_BUFS; ++i) FX_CUDA(h, cudaMalloc(&h->d_bcast[i], sizeof(float) * C * sub));
        h->bcast_floats = (size_t)(C * sub);
    }
    // Curve j's staging in each buffer set: the per-instance curves at k * sub * N floats (16-byte aligned whenever N % 4 == 0, as the
    // streaming kernels need; route() takes any other launch to the serial kernel or period by period), then the broadcast ones.
    size_t cv_off[FX8010_MAX_CONTROL_CURVES] = {};
    if (cv) {
        size_t k_pi = 0, k_bc = 0;
        for (int j = 0; j < cv->n; ++j) cv_off[j] = cv->cv.bcast[j] ? n_pi * sub * N + (k_bc++) * sub : (k_pi++) * sub * N;
        const size_t cv_need = (size_t)sub * (n_pi * N + n_bc);
        if (cv_need > h->curve_floats) {
            const int rc = sync_all(h);
            if (rc) return rc;
            for (int i = 0; i < HOST_PIPE_BUFS; ++i) { cudaFree(h->d_curve_stage[i]); h->d_curve_stage[i] = nullptr; }
            h->curve_floats = 0;
            for (int i = 0; i < HOST_PIPE_BUFS; ++i) FX_CUDA(h, cudaMalloc(&h->d_curve_stage[i], sizeof(float) * cv_need));
            h->curve_floats = cv_need;
        }
    }
    {   // earlier device-side batches come first
        const int rc = order_on(h, h->s_comp);
        if (rc) return rc;
    }
    if (cv) h->chain.clear();       // every curve launch waits for its predecessor at its start (as in fx8010_gpu_process_batch_curves)
    // pipe_seq counts sub-blocks over the life of the staging buffers, so that asynchronous calls chain:
    // sub-block q reuses the buffers of sub-block q - HOST_PIPE_BUFS once those have been consumed / drained
    for (long s0 = 0; s0 < n_samples; s0 += sub, ++h->pipe_seq) {
        const int buf = (int)(h->pipe_seq % HOST_PIPE_BUFS);
        const long len = std::min<long>(sub, n_samples - s0);
        const size_t cs = (size_t)(packed ? len : sub) * N;
        if (h->pipe_seq >= HOST_PIPE_BUFS) FX_CUDA(h, cudaStreamWaitEvent(h->s_h2d, h->ev_comp[buf], 0));     // stage_in[buf] consumed
        if (in && bcast)
            for (size_t c = 0; c < C; ++c)
                FX_CUDA(h, cudaMemcpyAsync(h->d_bcast[buf] + c * (size_t)sub, in + c * (size_t)n_samples + s0, sizeof(float) * len, cudaMemcpyHostToDevice, h->s_h2d));
        else if (in)
            for (size_t c = 0; c < C; ++c) {
                if (host_n == N)
                    FX_CUDA(h, cudaMemcpyAsync(h->d_stage_in[buf] + c * cs, in + (c * (size_t)n_samples + s0) * N,
                                               sizeof(float) * len * N, cudaMemcpyHostToDevice, h->s_h2d));
                else
                    FX_CUDA(h, cudaMemcpy2DAsync(h->d_stage_in[buf] + c * cs, sizeof(float) * N, in + (c * (size_t)n_samples + s0) * host_n,
                                                 sizeof(float) * host_n, sizeof(float) * N, (size_t)len, cudaMemcpyHostToDevice, h->s_h2d));
            }
        CurveRows staged = {};
        if (cv) {                   // this sub-block's rows of every curve, on the stream and behind the same events as its inputs
            staged = *cv;
            for (int j = 0; j < cv->n; ++j) {
                float* dst = h->d_curve_stage[buf] + cv_off[j];
                const float* src = cv->cv.p[j];
                staged.cv.p[j] = dst;
                if (cv->cv.bcast[j])
                    FX_CUDA(h, cudaMemcpyAsync(dst, src + s0, sizeof(float) * len, cudaMemcpyHostToDevice, h->s_h2d));
                else if (host_n == N)
                    FX_CUDA(h, cudaMemcpyAsync(dst, src + (size_t)s0 * N, sizeof(float) * len * N, cudaMemcpyHostToDevice, h->s_h2d));
                else
                    FX_CUDA(h, cudaMemcpy2DAsync(dst, sizeof(float) * N, src + (size_t)s0 * host_n, sizeof(float) * host_n, sizeof(float) * N, (size_t)len,
                                                 cudaMemcpyHostToDevice, h->s_h2d));
            }
        }
        FX_CUDA(h, cudaEventRecord(h->ev_h2d[buf], h->s_h2d));
        FX_CUDA(h, cudaStreamWaitEvent(h->s_comp, h->ev_h2d[buf], 0));
        if (h->pipe_seq >= HOST_PIPE_BUFS) FX_CUDA(h, cudaStreamWaitEvent(h->s_comp, h->ev_d2h[buf], 0));    // stage_out[buf] drained
        if (in && bcast) {
            for (size_t c = 0; c < C; ++c) {
                fx_broadcast_kernel<<<dim3((unsigned)std::min<size_t>(64, (N + 255) / 256), (unsigned)len), 256, 0, h->s_comp>>>(
                    h->d_bcast[buf] + c * (size_t)sub, h->d_stage_in[buf] + c * cs, (int)len, (int)N);
                h->info.kernel_launches++;
            }
            FX_CUDA(h, cudaGetLastError());
        }
        const float* d_in = in ? h->d_stage_in[buf] : nullptr;
        const int rc = step(d_in, h->d_stage_out[buf], cs, (int)len, cv ? &staged : nullptr);
        if (rc) return rc;
        FX_CUDA(h, cudaEventRecord(h->ev_comp[buf], h->s_comp));
        FX_CUDA(h, cudaStreamWaitEvent(h->s_d2h, h->ev_comp[buf], 0));
        for (size_t c = 0; c < C; ++c) {
            if (host_n == N)
                FX_CUDA(h, cudaMemcpyAsync(out + (c * (size_t)n_samples + s0) * N, h->d_stage_out[buf] + c * cs,
                                           sizeof(float) * len * N, cudaMemcpyDeviceToHost, h->s_d2h));
            else
                FX_CUDA(h, cudaMemcpy2DAsync(out + (c * (size_t)n_samples + s0) * host_n, sizeof(float) * host_n, h->d_stage_out[buf] + c * cs,
                                             sizeof(float) * N, sizeof(float) * N, (size_t)len, cudaMemcpyDeviceToHost, h->s_d2h));
        }
        FX_CUDA(h, cudaEventRecord(h->ev_d2h[buf], h->s_d2h));
    }
    if (wait) FX_CUDA(h, cudaStreamSynchronize(h->s_d2h));
    return FX8010_OK;
}

// The single-handle host calls: each sub-block runs launch_block, or launch_curves with the call's curves.
static int process_host_handle(fx8010_gpu* h, const float* in, float* out, int n_samples, bool wait, size_t host_n = 0, bool bcast = false,
                               const CurveRows* cv = nullptr) {
    return process_host_impl(h, in, out, n_samples, wait, host_n, bcast, cv, false,
                             [h](const float* d_in, float* d_out, size_t cs, int len, const CurveRows* staged) {
        return staged ? launch_curves(h, d_in, d_out, cs, len, *staged, h->s_comp)
                      : launch_block(h, d_in, d_out, cs, cs, len, h->s_comp, true);   // (the internal stream carries this handle's launches only)
    });
}

int fx8010_gpu_process_batch_host(fx8010_gpu* h, const float* in, float* out, int n_samples) {
    return process_host_handle(h, in, out, n_samples, true);
}
int fx8010_gpu_process_batch_host_async(fx8010_gpu* h, const float* in, float* out, int n_samples) {
    return process_host_handle(h, in, out, n_samples, false);
}
int fx8010_gpu_process_batch_host_slice(fx8010_gpu* h, const float* in, float* out, int n_samples, size_t host_instances, int wait) {
    return process_host_handle(h, in, out, n_samples, wait != 0, host_instances);
}
int fx8010_gpu_process_batch_host_broadcast(fx8010_gpu* h, const float* in, float* out, int n_samples, size_t host_instances, int wait) {
    return process_host_handle(h, in, out, n_samples, wait != 0, host_instances, true);
}
int fx8010_gpu_process_batch_host_curves(fx8010_gpu* h, const float* in, float* out, int n_samples, const fx8010_host_curve* curves, int n_curves,
                                         size_t host_instances, int wait) {
    FX_NEED_PROGRAM(h);
    if (!out || n_samples < 0) return fail(h, FX8010_ERR_ARG, "out is NULL or n_samples negative");
    if (host_instances != 0 && host_instances < (size_t)h->N) return fail(h, FX8010_ERR_ARG, "host row length below the instance count");
    CurveRows rows;
    const int rc = curves_begin(h, curves, n_curves, &fx8010_host_curve::values, n_samples > 0, rows);
    if (rc) return rc;
    return process_host_handle(h, in, out, n_samples, wait != 0, host_instances, false, n_curves > 0 ? &rows : nullptr);
}

// fx8010_chain_process_batch_host(_curves): stage 0's host pipeline, each sub-block running the device chain call on its staging buffers
// (packed, so that they are laid out as the device call's buffers) on stage 0's compute stream.
static int chain_host(fx8010_chain* c, const float* in, float* out, int n_samples, const fx8010_chain_host_curve* curves, int n_curves,
                      size_t host_n, bool wait) {
    if (!c) return FX8010_ERR_ARG;
    std::vector<std::vector<fx8010_control_curve>> per_stage;
    int rc = chain_check(c, "", in, out, n_samples, curves, n_curves, &fx8010_chain_host_curve::values, per_stage);
    if (rc) return rc;
    fx8010_gpu* h0 = c->st[0];
    if (host_n != 0 && host_n < (size_t)h0->N) return chain_fail(c, FX8010_ERR_ARG, "host row length below the instance count");
    if (cudaSetDevice(c->device) != cudaSuccess) return chain_fail(c, FX8010_ERR_CUDA, "cudaSetDevice failed");
    if (n_samples == 0) return FX8010_OK;
    for (fx8010_gpu* h : c->st) {                            // every stage's earlier work, on any stream, comes first
        rc = order_on(h, h0->s_comp);
        if (rc) return chain_fail(c, rc, h->err);
    }
    CurveRows rows = {};
    rows.n = n_curves;
    for (int q = 0; q < n_curves; ++q) {
        rows.reg[q] = curves[q].reg_index;
        rows.cv.p[q] = curves[q].values; rows.cv.bcast[q] = curves[q].broadcast ? 1 : 0;
    }
    bool all_fused = true, step_failed = false;
    std::string why;
    rc = process_host_impl(h0, in, out, n_samples, wait, host_n, false, n_curves > 0 ? &rows : nullptr, true,
                           [&](const float* d_in, float* d_out, size_t, int len, const CurveRows* staged) {
        int r;
        if (staged) {
            fx8010_chain_curve cv[FX8010_MAX_CONTROL_CURVES];
            for (int q = 0; q < n_curves; ++q) cv[q] = fx8010_chain_curve{curves[q].stage, curves[q].reg_index, rows.cv.bcast[q], 0, staged->cv.p[q]};
            r = fx8010_chain_process_batch_curves(c, d_in, d_out, len, cv, n_curves, h0->s_comp);
        } else
            r = fx8010_chain_process_batch(c, d_in, d_out, len, h0->s_comp);
        if (r) { step_failed = true; return r; }
        if (!c->fused_last && all_fused) { all_fused = false; why = c->why; }
        return (int)FX8010_OK;
    });
    if (rc) return step_failed ? rc : chain_fail(c, rc, h0->err);
    c->fused_last = all_fused ? 1 : 0;
    c->why = all_fused ? std::string() : why;
    // Stage 0's compute stream now carries other handles' launches: none of its later launches may count on following its own.
    for (fx8010_gpu* h : c->st) h->chain.clear();
    return FX8010_OK;
}

int fx8010_chain_process_batch_host(fx8010_chain* c, const float* in, float* out, int n_samples, size_t host_instances, int wait) {
    return chain_host(c, in, out, n_samples, nullptr, 0, host_instances, wait != 0);
}
int fx8010_chain_process_batch_host_curves(fx8010_chain* c, const float* in, float* out, int n_samples, const fx8010_chain_host_curve* curves,
                                           int n_curves, size_t host_instances, int wait) {
    return chain_host(c, in, out, n_samples, curves, n_curves, host_instances, wait != 0);
}

int fx8010_chain_synchronize(fx8010_chain* c) {
    if (!c) return FX8010_ERR_ARG;
    for (fx8010_gpu* h : c->st) {
        const int rc = sync_all(h);
        if (rc) return chain_fail(c, rc, h->err);
    }
    return FX8010_OK;
}

int fx8010_gpu_synchronize(fx8010_gpu* h, void* stream) {
    if (!h) return FX8010_ERR_ARG;
    FX_CUDA(h, cudaSetDevice(h->device));
    if (stream) FX_CUDA(h, cudaStreamSynchronize((cudaStream_t)stream));
    return sync_all(h);
}

void* fx8010_gpu_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
    return p;
}
void fx8010_gpu_host_free(void* p) { if (p) cudaFreeHost(p); }

int fx8010_gpu_get_instruction_counts(fx8010_gpu* h, unsigned long long* out) {
    FX_NEED_PROGRAM(h);
    if (!out) return fail(h, FX8010_ERR_ARG, "out is NULL");
    const int rc = sync_all(h);
    if (rc) return rc;
    FX_CUDA(h, cudaMemcpy(out, h->d_counts, sizeof(unsigned long long) * h->N, cudaMemcpyDeviceToHost));
    return FX8010_OK;
}

int fx8010_gpu_get_instruction_count(fx8010_gpu* h, unsigned long long* total) {
    FX_NEED_PROGRAM(h);
    if (!total) return fail(h, FX8010_ERR_ARG, "total is NULL");
    std::vector<unsigned long long> c(h->N);
    const int rc = fx8010_gpu_get_instruction_counts(h, c.data());
    if (rc) return rc;
    unsigned long long s = 0;
    for (unsigned long long v : c) s += v;
    *total = s;
    return FX8010_OK;
}

int fx8010_gpu_get_dims(fx8010_gpu* h, fx8010_state_dims* out) {
    if (!h || !out) return FX8010_ERR_ARG;
    out->n_instances = h->N; out->n_channels = h->C;
    out->n_regs = (int)h->regs.size(); out->n_instrs = (int)h->instrs.size();
    out->itram_size = h->itram_size; out->xtram_size = h->xtram_size;
    out->itram_alloc = h->itram_size; out->xtram_alloc = h->xtram_size;
    return FX8010_OK;
}

int fx8010_gpu_get_registers(fx8010_gpu* h, float* out) {
    FX_NEED_PROGRAM(h);
    if (!out) return fail(h, FX8010_ERR_ARG, "out is NULL");
    const int rc = sync_all(h);
    if (rc) return rc;
    FX_CUDA(h, cudaMemcpy(out, h->d_gpr, sizeof(float) * h->regs.size() * h->N, cudaMemcpyDeviceToHost));
    return FX8010_OK;
}

int fx8010_gpu_set_registers(fx8010_gpu* h, const float* in) {
    FX_NEED_PROGRAM(h);
    if (!in) return fail(h, FX8010_ERR_ARG, "in is NULL");
    const int rc = sync_all(h);
    if (rc) return rc;
    FX_CUDA(h, cudaMemcpy(h->d_gpr, in, sizeof(float) * h->regs.size() * h->N, cudaMemcpyHostToDevice));
    for (size_t r = 0; r < h->regs.size(); ++r) {            // rows holding one bit pattern in every instance stay load-time constants
        const uint32_t* row = reinterpret_cast<const uint32_t*>(in) + r * (size_t)h->N;
        bool same = true;
        for (int i = 1; i < h->N && same; ++i) same = row[i] == row[0];
        h->reg_uniform[r] = same ? 1 : 0;
        if (same) memcpy(&h->reg_value[r], row, 4);
        tr_touch(h, (int)r);
    }
    h->encode_dirty = true;
    return FX8010_OK;
}

int fx8010_gpu_get_scalars(fx8010_gpu* h, double* acc, uint32_t* lfsr, float* out_latch, int32_t* tram_ptrs) {
    FX_NEED_PROGRAM(h);
    const int rc = sync_all(h);
    if (rc) return rc;
    const size_t N = (size_t)h->N;
    if (acc) FX_CUDA(h, cudaMemcpy(acc, h->d_acc, sizeof(double) * N, cudaMemcpyDeviceToHost));
    if (lfsr) FX_CUDA(h, cudaMemcpy(lfsr, h->d_lfsr, sizeof(uint32_t) * 2 * N, cudaMemcpyDeviceToHost));
    if (out_latch) FX_CUDA(h, cudaMemcpy(out_latch, h->d_latch, sizeof(float) * h->C * N, cudaMemcpyDeviceToHost));
    if (tram_ptrs) FX_CUDA(h, cudaMemcpy(tram_ptrs, h->d_ptrs, sizeof(int32_t) * 4 * N, cudaMemcpyDeviceToHost));
    return FX8010_OK;
}

int fx8010_gpu_set_scalars(fx8010_gpu* h, const double* acc, const uint32_t* lfsr, const float* out_latch, const int32_t* tram_ptrs) {
    FX_NEED_PROGRAM(h);
    const int rc = sync_all(h);
    if (rc) return rc;
    const size_t N = (size_t)h->N;
    if (tram_ptrs) {                                  // pointers index the rings: keep them inside
        const int sizes[4] = {h->itram_size, h->itram_size, h->xtram_size, h->xtram_size};
        for (int q = 0; q < 4; ++q)
            for (size_t i = 0; i < N; ++i) {
                const int32_t v = tram_ptrs[q * N + i];
                if (v < 0 || (sizes[q] > 0 && v >= sizes[q]) || (sizes[q] == 0 && v != 0))
                    return fail(h, FX8010_ERR_ARG, "TRAM pointer outside its ring");
            }
    }
    if (acc) FX_CUDA(h, cudaMemcpy(h->d_acc, acc, sizeof(double) * N, cudaMemcpyHostToDevice));
    if (lfsr) FX_CUDA(h, cudaMemcpy(h->d_lfsr, lfsr, sizeof(uint32_t) * 2 * N, cudaMemcpyHostToDevice));
    if (out_latch) FX_CUDA(h, cudaMemcpy(h->d_latch, out_latch, sizeof(float) * h->C * N, cudaMemcpyHostToDevice));
    if (tram_ptrs) { FX_CUDA(h, cudaMemcpy(h->d_ptrs, tram_ptrs, sizeof(int32_t) * 4 * N, cudaMemcpyHostToDevice)); h->tram_ptrs_pristine = false; }
    return FX8010_OK;
}

int fx8010_gpu_get_tram(fx8010_gpu* h, int which, int instance, float* out) {
    FX_NEED_PROGRAM(h);
    const int size = which == 0 ? h->itram_size : h->xtram_size;
    const float* ring = which == 0 ? h->d_itram : h->d_xtram;
    if (!out || (which != 0 && which != 1) || instance < 0 || instance >= h->N || !ring) return fail(h, FX8010_ERR_ARG, "bad TRAM selector / instance, or that TRAM is unused");
    const int rc = sync_all(h);
    if (rc) return rc;
    FX_CUDA(h, cudaMemcpy2D(out, sizeof(float), ring + instance, sizeof(float) * h->N, sizeof(float), size, cudaMemcpyDeviceToHost));
    return FX8010_OK;
}

int fx8010_gpu_set_tram(fx8010_gpu* h, int which, int instance, const float* in) {
    FX_NEED_PROGRAM(h);
    const int size = which == 0 ? h->itram_size : h->xtram_size;
    float* ring = which == 0 ? h->d_itram : h->d_xtram;
    if (!in || (which != 0 && which != 1) || instance < 0 || instance >= h->N || !ring) return fail(h, FX8010_ERR_ARG, "bad TRAM selector / instance, or that TRAM is unused");
    const int rc = sync_all(h);
    if (rc) return rc;
    FX_CUDA(h, cudaMemcpy2D(ring + instance, sizeof(float) * h->N, in, sizeof(float), sizeof(float), size, cudaMemcpyHostToDevice));
    return FX8010_OK;
}

int fx8010_gpu_get_runtime_flags(fx8010_gpu* h, unsigned int* flags, int clear) {
    if (!h || !flags) return FX8010_ERR_ARG;
    FX_CUDA(h, cudaSetDevice(h->device));
    const int rc = sync_all(h);
    if (rc) return rc;
    FX_CUDA(h, cudaMemcpy(flags, h->d_flags, sizeof(unsigned int), cudaMemcpyDeviceToHost));
    if (clear) FX_CUDA(h, cudaMemset(h->d_flags, 0, sizeof(unsigned int)));
    return FX8010_OK;
}

int fx8010_gpu_trace(fx8010_gpu* h, const float* in, float* out, int n_samples, int instance, fx8010_trace_entry* entries) {
    FX_NEED_PROGRAM(h);
    if (!entries || n_samples <= 0 || instance < 0 || instance >= h->N) return fail(h, FX8010_ERR_ARG, "bad instance / n_samples or NULL entries");
    int rc = sync_all(h);
    if (rc) return rc;
    const size_t n_rec = (size_t)n_samples * h->instrs.size(), io = (size_t)h->C * n_samples * h->N;
    float* d_in = nullptr; float* d_out = nullptr;
    auto cleanup = [&]() {
        cudaFree(h->d_trace); h->d_trace = nullptr; cudaFree(d_in); cudaFree(d_out);
        h->trace_mode = false; h->encode_dirty = true; h->plan_key.ns = -1;
    };
    h->trace_mode = true; h->trace_inst = instance; h->encode_dirty = true; h->plan_key.ns = -1;
    cudaError_t e = cudaMalloc(&h->d_trace, sizeof(fx8010_trace_entry) * n_rec);
    if (e == cudaSuccess) e = cudaMemset(h->d_trace, 0, sizeof(fx8010_trace_entry) * n_rec);
    if (e == cudaSuccess) e = cudaMalloc(&d_out, sizeof(float) * io);
    if (e == cudaSuccess && in) { e = cudaMalloc(&d_in, sizeof(float) * io); if (e == cudaSuccess) e = cudaMemcpy(d_in, in, sizeof(float) * io, cudaMemcpyHostToDevice); }
    if (e != cudaSuccess) { cleanup(); return fail(h, FX8010_ERR_CUDA, std::string("trace buffers: ") + cudaGetErrorString(e)); }
    const size_t cs = (size_t)n_samples * h->N;
    rc = launch_block(h, d_in, d_out, cs, cs, n_samples, h->s_comp);
    if (!rc) {
        e = cudaStreamSynchronize(h->s_comp);
        if (e == cudaSuccess) e = cudaMemcpy(entries, h->d_trace, sizeof(fx8010_trace_entry) * n_rec, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && out) e = cudaMemcpy(out, d_out, sizeof(float) * io, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(h, FX8010_ERR_CUDA, std::string("trace: ") + cudaGetErrorString(e));
    }
    cleanup();
    return rc;
}

// ---- program translator: status and the host-only source generator (tests/test_translate.py) ----
static int translate_status(fx8010_gpu* h, Translation& T, int* state, int* regs_per_thread, int* local_bytes, char* message, size_t message_cap) {
    if (T.state == 1 && h->loaded && cudaSetDevice(h->device) == cudaSuccess) tr_ready(h, T, false);   // pick up a finished background compilation (the kernel loads into this device's context)
    if (state) *state = T.state;
    if (regs_per_thread) *regs_per_thread = T.regs;
    if (local_bytes) *local_bytes = T.local;
    if (message && message_cap) { strncpy(message, T.error.c_str(), message_cap - 1); message[message_cap - 1] = 0; }
    return FX8010_OK;
}
int fx8010_gpu_translate_status(fx8010_gpu* h, int* state, int* regs_per_thread, int* local_bytes, char* message, size_t message_cap) {
    if (!h) return FX8010_ERR_ARG;
    return translate_status(h, h->tr, state, regs_per_thread, local_bytes, message, message_cap);
}
int fx8010_gpu_translate_status_curves(fx8010_gpu* h, int* state, int* regs_per_thread, int* local_bytes, int* kind, char* message, size_t message_cap) {
    if (!h) return FX8010_ERR_ARG;
    if (kind) *kind = h->tr_cv.state == 2 ? h->tr_cv.kind : -1;
    return translate_status(h, h->tr_cv, state, regs_per_thread, local_bytes, message, message_cap);
}

// Needs no device: analyses the image as load_program would and generates the CUDA source of its translated kernel (for control curves
// on cregs[n_curves] when n_curves > 0) into `src`.  0, -1 for a bad image or curve list, -2 when the program is not eligible.
// For a freshly loaded image this is the source a handle generates at its first launch on a B200 (148 SMs), except that the developer
// switches a handle reads when it is created (FX8010_NO_STATELESS, FX8010_NO_TSPLIT, FX8010_TR_RECUR) are not applied.
// The host-side analysis of image `im` as load_program would leave it (the registers of cv_reg automated, hence not uniform) in tmp.
// 0, or -1 for a bad image or curve list.
static int image_handle(const fx8010_program_image* im, int n_instances, int n_channels, const std::vector<int>& cv_reg, fx8010_gpu& tmp) {
    if (!im || !im->instrs || !im->regs || im->n_instrs <= 0 || im->n_regs <= 0 || n_channels <= 0 || n_instances <= 0) return -1;
    tmp.C = n_channels; tmp.N = n_instances;
    tmp.instrs.assign(im->instrs, im->instrs + im->n_instrs);
    tmp.regs.assign(im->regs, im->regs + im->n_regs);
    for (const fx8010_instr& in : tmp.instrs)
        if (in.opcode < 0 || in.opcode >= FX_NUM_OPCODES || in.r < 0 || in.r >= im->n_regs || in.a < 0 || in.a >= im->n_regs ||
            in.x < 0 || in.x >= im->n_regs || in.y < 0 || in.y >= im->n_regs) return -1;
    for (const fx8010_reg& r : tmp.regs) if (r.io_index < 0 || r.io_index >= n_channels) return -1;
    std::string why;
    if (!curves_valid(tmp.regs, cv_reg, why)) return -1;
    tmp.itram_size = im->itram_size; tmp.xtram_size = im->xtram_size;
    tmp.reg_uniform.assign(im->n_regs, 1);
    tmp.reg_value.resize(im->n_regs);
    for (int r = 0; r < im->n_regs; ++r) tmp.reg_value[r] = im->regs[r].init_value;
    for (int r : cv_reg) tmp.reg_uniform[r] = 0;              // (as fx8010_gpu_process_batch_curves leaves them)
    tmp.tr_volatile.assign(im->n_regs, 0);
    analyse(&tmp);
    return 0;
}

// Needs no device: analyses the image as load_program would and generates the CUDA source of its translated kernel (for control curves
// on cregs[n_curves] when n_curves > 0) into `src`.  0, -1 for a bad image or curve list, -2 when the program is not eligible.
// For a freshly loaded image this is the source a handle generates at its first launch on a B200 (148 SMs), except that the developer
// switches a handle reads when it is created (FX8010_NO_STATELESS, FX8010_NO_TSPLIT, FX8010_TR_RECUR) are not applied.
static int translate_source_gen(const fx8010_program_image* im, int n_instances, int n_channels, const int32_t* cregs, const int32_t* cbcast,
                                int n_curves, std::string& src) {
    if (n_curves < 0 || n_curves > FX8010_MAX_CONTROL_CURVES || (n_curves > 0 && (!cregs || !cbcast))) return -1;
    Translation T;
    for (int j = 0; j < n_curves; ++j) { T.cv_reg.push_back(cregs[j]); T.cv_bcast.push_back(cbcast[j] ? 1 : 0); }
    fx8010_gpu tmp;
    if (image_handle(im, n_instances, n_channels, T.cv_reg, tmp)) return -1;
    const int kind = tr_kind(&tmp, T);
    tmp.tr_gen = n_curves ? &T : nullptr;
    if (kind == 0 && !tr_eligible(&tmp)) return -2;
    std::vector<uint8_t> folded;
    src = kind ? tr_generate_sl(&tmp, folded, kind == 2) : tr_generate(&tmp, folded);
    tmp.tr_gen = nullptr;
    return 0;
}
// Writes `src` to buf (cap bytes with the terminator) and, with compile_check, compiles it with NVRTC: *cubin_bytes = the CUBIN size or -1.
static long long translate_source_out(const std::string& src, char* buf, size_t cap, int compile_check, int* cubin_bytes) {
    if (buf && cap) { strncpy(buf, src.c_str(), cap - 1); buf[cap - 1] = 0; }
    if (compile_check) {                                     // NVRTC -> sm_100a CUBIN (works without a GPU)
        std::vector<char> cubin; std::string log;
        const bool ok = translate_compile(src, cubin, log);
        if (cubin_bytes) *cubin_bytes = ok ? (int)cubin.size() : -1;
        if (!ok) fprintf(stderr, "fx8010_translate_source: %s\n", log.c_str());
    }
    return (long long)src.size();
}
static long long translate_source_impl(const fx8010_program_image* im, int n_instances, int n_channels, const int32_t* cregs, const int32_t* cbcast,
                                       int n_curves, char* buf, size_t cap, int compile_check, int* regs_or_status) {
    std::string src;
    const int g = translate_source_gen(im, n_instances, n_channels, cregs, cbcast, n_curves, src);
    return g ? g : translate_source_out(src, buf, cap, compile_check, regs_or_status);
}
long long fx8010_translate_source(const fx8010_program_image* im, int n_instances, int n_channels, char* buf, size_t cap, int compile_check, int* regs_or_status) {
    return translate_source_impl(im, n_instances, n_channels, nullptr, nullptr, 0, buf, cap, compile_check, regs_or_status);
}
long long fx8010_translate_source_curves(const fx8010_program_image* im, int n_instances, int n_channels, const int32_t* regs, const int32_t* broadcast,
                                         int n_curves, char* buf, size_t cap, int compile_check, int* cubin_bytes) {
    return translate_source_impl(im, n_instances, n_channels, regs, broadcast, n_curves, buf, cap, compile_check, cubin_bytes);
}

// The chain's fused kernel, with control curves q on register regs[q] of stage stage[q] when n_curves > 0: -1 for a bad image or a curve
// list fx8010_chain_process_batch_curves refuses, -2 when some stage is not stateless (a program with SKIP never is, so no curve can make a
// stateless stage ineligible).
static long long translate_source_chain_impl(const fx8010_program_image* const* images, int n_stages, int n_instances, int n_channels,
                                             const int32_t* stage, const int32_t* regs, const int32_t* broadcast, int n_curves, char* buf,
                                             size_t cap, int compile_check, int* cubin_bytes) {
    if (!images || n_stages < 1 || n_stages > FX8010_MAX_CHAIN_STAGES) return -1;
    if (n_curves < 0 || n_curves > FX8010_MAX_CONTROL_CURVES || (n_curves > 0 && (!stage || !regs || !broadcast))) return -1;
    std::vector<ChainCurve> cvs;
    std::vector<std::vector<int>> per_stage((size_t)n_stages);
    for (int q = 0; q < n_curves; ++q) {
        if (stage[q] < 0 || stage[q] >= n_stages) return -1;
        per_stage[stage[q]].push_back(regs[q]);
        cvs.push_back(ChainCurve{stage[q], regs[q], (uint8_t)(broadcast[q] ? 1 : 0)});
    }
    std::vector<fx8010_gpu> tmp((size_t)n_stages);
    for (int j = 0; j < n_stages; ++j)
        if (image_handle(images[j], n_instances, n_channels, per_stage[j], tmp[j])) return -1;
    for (const fx8010_gpu& h : tmp) if (!h.stateless) return -2;
    std::vector<const fx8010_gpu*> hs;
    for (const fx8010_gpu& h : tmp) hs.push_back(&h);
    std::vector<std::vector<uint8_t>> folded;
    return translate_source_out(tr_generate_chain(hs, folded, cvs), buf, cap, compile_check, cubin_bytes);
}
long long fx8010_translate_source_chain(const fx8010_program_image* const* images, int n_stages, int n_instances, int n_channels, char* buf,
                                        size_t cap, int compile_check, int* cubin_bytes) {
    return translate_source_chain_impl(images, n_stages, n_instances, n_channels, nullptr, nullptr, nullptr, 0, buf, cap, compile_check, cubin_bytes);
}
long long fx8010_translate_source_chain_curves(const fx8010_program_image* const* images, int n_stages, int n_instances, int n_channels,
                                               const int32_t* stage, const int32_t* regs, const int32_t* broadcast, int n_curves, char* buf,
                                               size_t cap, int compile_check, int* cubin_bytes) {
    return translate_source_chain_impl(images, n_stages, n_instances, n_channels, stage, regs, broadcast, n_curves, buf, cap, compile_check,
                                       cubin_bytes);
}

int fx8010_kernel_cache_set_dir(const char* dir) {
    std::lock_guard<std::mutex> lk(g_kc_dir_mutex);
    g_kc_dir_set = true;
    g_kc_dir = dir ? dir : "";
    return FX8010_OK;
}
int fx8010_kernel_cache_precompile(const fx8010_program_image* im, int n_instances, int n_channels, const int32_t* regs, const int32_t* broadcast,
                                   int n_curves) {
    std::string src;
    const int g = translate_source_gen(im, n_instances, n_channels, regs, broadcast, n_curves, src);
    return g ? g : kc_precompile(src);
}
int fx8010_kernel_cache_get_stats(fx8010_kernel_cache_stats* out) {
    if (!out) return FX8010_ERR_ARG;
    out->nvrtc_compiles = g_kc.nvrtc_compiles; out->memory_hits = g_kc.memory_hits; out->store_hits = g_kc.store_hits;
    out->joined_compiles = g_kc.joined_compiles; out->disk_hits = g_kc.disk_hits; out->disk_writes = g_kc.disk_writes;
    out->disk_rejected = g_kc.disk_rejected; out->disk_write_failures = g_kc.disk_write_failures;
    return FX8010_OK;
}

const char* fx8010_gpu_last_error(fx8010_gpu* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int fx8010_gpu_get_launch_info(fx8010_gpu* h, fx8010_launch_info* out) {
    if (!h || !out) return FX8010_ERR_ARG;
    *out = h->info;
    return FX8010_OK;
}

}  // extern "C"
