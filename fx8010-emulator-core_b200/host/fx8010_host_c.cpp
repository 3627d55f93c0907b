// fx8010_host_c.cpp — the plain-C view of Klangraum::FX8010 declared in include/fx8010_host.h.
#include <cstring>
#include <exception>
#include <string>
#include <vector>

#include "FX8010.h"
#include "fx8010_host.h"

struct fx8010_host {
    Klangraum::FX8010 fx;
    std::string err;
    fx8010_host(int c, int n, int d) : fx(c, n, d) {}
    fx8010_host(int c, int n, const std::vector<int>& devs) : fx(c, n, devs) {}
};

struct fx8010_host_chain {
    Klangraum::FX8010Chain chain;
    std::string err;
    explicit fx8010_host_chain(const std::vector<Klangraum::FX8010*>& stages) : chain(stages) {}
};

namespace {
thread_local std::string g_chain_create_error;
void copy_out(const std::string& s, char* buf, int cap) {
    if (!buf || cap <= 0) return;
    std::strncpy(buf, s.c_str(), (size_t)cap - 1);
    buf[cap - 1] = 0;
}
template <typename F> int guarded(fx8010_host* h, F f) {
    try { f(); return 0; }
    catch (const std::exception& e) { h->err = e.what(); return 1; }
}
}  // namespace

extern "C" {

fx8010_host* fx8010_host_create(int c, int n, int d) {
    if (c <= 0 || n <= 0) return nullptr;
    return new fx8010_host(c, n, d);
}
fx8010_host* fx8010_host_create_multi(int c, int n, const int* devices, int n_devices) {
    if (c <= 0 || n <= 0 || !devices || n_devices <= 0) return nullptr;
    return new fx8010_host(c, n, std::vector<int>(devices, devices + n_devices));
}
void fx8010_host_destroy(fx8010_host* h) { delete h; }
const char* fx8010_host_last_error(fx8010_host* h) { return h ? h->err.c_str() : ""; }

int fx8010_host_load_file(fx8010_host* h, const char* path) { return h->fx.loadFile(path) ? 1 : 0; }
int fx8010_host_load_text(fx8010_host* h, const char* text, size_t len) { return h->fx.loadText(std::string(text, len)) ? 1 : 0; }
void fx8010_host_set_relaxed(fx8010_host* h, int on) { h->fx.setRelaxedSyntax(on != 0); }
int fx8010_host_set_translation(fx8010_host* h, int mode) {
    try { h->fx.setTranslation(mode); return 0; } catch (...) { return 1; }
}
void fx8010_host_set_kernel_cache_dir(const char* dir) { Klangraum::FX8010::setKernelCacheDir(dir ? dir : ""); }
int fx8010_host_ready(fx8010_host* h) { return h->fx.getReadyStatus() ? 1 : 0; }

int fx8010_host_num_registers(fx8010_host* h) { return (int)h->fx.frontend().registers().size(); }
void fx8010_host_register_info(fx8010_host* h, int i, int* type, float* value, int* io, char* name, int cap) {
    const fx8010::Register& r = h->fx.frontend().registers()[(size_t)i];
    *type = r.type; *value = r.value; *io = r.io_index;
    copy_out(r.name, name, cap);
}
int fx8010_host_num_instructions(fx8010_host* h) { return (int)h->fx.frontend().instructions().size(); }
void fx8010_host_instruction_info(fx8010_host* h, int i, int* f) {
    const fx8010_instr& in = h->fx.frontend().instructions()[(size_t)i];
    f[0] = in.opcode; f[1] = in.r; f[2] = in.a; f[3] = in.x; f[4] = in.y;
    f[5] = in.has_input; f[6] = in.has_output; f[7] = in.has_noise;
}
int fx8010_host_itram_size(fx8010_host* h) { return h->fx.frontend().itramSize(); }
int fx8010_host_xtram_size(fx8010_host* h) { return h->fx.frontend().xtramSize(); }
void fx8010_host_tables(fx8010_host* h, double* out) {
    const size_t n = (size_t)FX8010_TABLE_COUNT * FX8010_TABLE_ENTRIES;
    std::memcpy(out, h->fx.frontend().logTables().data(), n * sizeof(double));
    std::memcpy(out + n, h->fx.frontend().expTables().data(), n * sizeof(double));
}
const fx8010_program_image* fx8010_host_image(fx8010_host* h) { return h->fx.frontend().image(); }

int fx8010_host_num_errors(fx8010_host* h) { return (int)h->fx.getErrorList().size(); }
int fx8010_host_error_info(fx8010_host* h, int i, char* buf, int cap) {
    const auto l = h->fx.getErrorList();
    copy_out(l[(size_t)i].errorDescription, buf, cap);
    return l[(size_t)i].errorRow;
}
int fx8010_host_num_controls(fx8010_host* h) { return (int)h->fx.getControlRegisters().size(); }
void fx8010_host_control_name(fx8010_host* h, int i, char* buf, int cap) { copy_out(h->fx.getControlRegisters()[(size_t)i], buf, cap); }
int fx8010_host_metadata(fx8010_host* h, const char* key, char* buf, int cap) {
    const auto m = h->fx.getMetaData();
    const auto it = m.find(key);
    if (it == m.end()) { copy_out("", buf, cap); return 0; }
    copy_out(it->second, buf, cap);
    return 1;
}

int fx8010_host_set_register(fx8010_host* h, const char* name, float v) {
    int r = 1;
    if (guarded(h, [&] { r = h->fx.setRegisterValue(name, v); })) return -1;
    return r;
}
float fx8010_host_get_register(fx8010_host* h, const char* name) {
    float v = 0.0f;
    guarded(h, [&] { v = h->fx.getRegisterValue(name); });
    return v;
}
int fx8010_host_set_register_values(fx8010_host* h, const char* name, const float* values) {
    int r = 1;
    if (guarded(h, [&] { r = h->fx.setRegisterValues(name, values); })) return -1;
    return r;
}
int fx8010_host_get_register_values(fx8010_host* h, const char* name, float* out) {
    int r = 1;
    if (guarded(h, [&] { r = h->fx.getRegisterValues(name, out); })) return -1;
    return r;
}

int fx8010_host_process(fx8010_host* h, const float* in, float* out, int n_samples) {
    return guarded(h, [&] {
        const int c = h->fx.getChannels();
        std::vector<float> ibuf((size_t)c, 0.0f);
        for (int s = 0; s < n_samples; ++s) {
            for (int j = 0; j < c; ++j) ibuf[(size_t)j] = in ? in[(size_t)s * c + j] : 0.0f;
            const std::vector<float> o = h->fx.process(ibuf);
            for (int j = 0; j < c; ++j) out[(size_t)s * c + j] = o[(size_t)j];
        }
    });
}
int fx8010_host_process_block(fx8010_host* h, const float* in, float* out, int n_samples) {
    return guarded(h, [&] { h->fx.processBlock(in, out, n_samples); });
}
int fx8010_host_process_block_device_curves(fx8010_host* h, const float* d_in, float* d_out, int n_samples, const char* const* names,
                                            const float* const* d_values, const int* broadcast, int n_curves, void* stream) {
    return guarded(h, [&] {
        std::vector<Klangraum::FX8010::Curve> cv;
        for (int j = 0; j < n_curves; ++j) cv.push_back(Klangraum::FX8010::Curve{names[j], d_values[j], broadcast[j] != 0});
        h->fx.processBlockDeviceWithCurves(d_in, d_out, n_samples, cv, stream);
    });
}
int fx8010_host_process_block_curves(fx8010_host* h, const float* in, float* out, int n_samples, const char* const* names, const float* const* values,
                                     const int* broadcast, int n_curves) {
    return guarded(h, [&] {
        std::vector<Klangraum::FX8010::HostCurve> cv;
        for (int j = 0; j < n_curves; ++j) cv.push_back(Klangraum::FX8010::HostCurve{names[j], values[j], broadcast[j] != 0});
        h->fx.processBlockWithCurves(in, out, n_samples, cv);
    });
}
int fx8010_host_instruction_counter(fx8010_host* h) {
    int v = 0;
    guarded(h, [&] { v = h->fx.getInstructionCounter(); });
    return v;
}
unsigned long long fx8010_host_instruction_counter_total(fx8010_host* h) {
    unsigned long long v = 0;
    guarded(h, [&] { v = h->fx.getInstructionCounterTotal(); });
    return v;
}
fx8010_gpu* fx8010_host_gpu(fx8010_host* h) {
    fx8010_gpu* g = nullptr;
    guarded(h, [&] { g = h->fx.gpuHandle(); });
    return g;
}

fx8010_host_chain* fx8010_host_chain_create(fx8010_host* const* stages, int n_stages) {
    if (!stages || n_stages <= 0) { g_chain_create_error = "no stages"; return nullptr; }
    std::vector<Klangraum::FX8010*> v;
    for (int j = 0; j < n_stages; ++j) v.push_back(stages[j] ? &stages[j]->fx : nullptr);
    try { return new fx8010_host_chain(v); }
    catch (const std::exception& e) { g_chain_create_error = e.what(); return nullptr; }
}
void fx8010_host_chain_destroy(fx8010_host_chain* c) { delete c; }
int fx8010_host_chain_process_block_device(fx8010_host_chain* c, const float* d_in, float* d_out, int n_samples, void* stream) {
    try { c->chain.processBlockDevice(d_in, d_out, n_samples, stream); return 0; }
    catch (const std::exception& e) { c->err = e.what(); return 1; }
}
int fx8010_host_chain_process_block_device_curves(fx8010_host_chain* c, const float* d_in, float* d_out, int n_samples, const int* stages,
                                                  const char* const* names, const float* const* d_values, const int* broadcast, int n_curves,
                                                  void* stream) {
    try {
        std::vector<Klangraum::FX8010Chain::Curve> cv;
        for (int j = 0; j < n_curves; ++j) cv.push_back(Klangraum::FX8010Chain::Curve{stages[j], names[j], d_values[j], broadcast[j] != 0});
        c->chain.processBlockDeviceWithCurves(d_in, d_out, n_samples, cv, stream);
        return 0;
    } catch (const std::exception& e) { c->err = e.what(); return 1; }
}
int fx8010_host_chain_process_block(fx8010_host_chain* c, const float* in, float* out, int n_samples) {
    try { c->chain.processBlock(in, out, n_samples); return 0; }
    catch (const std::exception& e) { c->err = e.what(); return 1; }
}
int fx8010_host_chain_process_block_curves(fx8010_host_chain* c, const float* in, float* out, int n_samples, const int* stages,
                                           const char* const* names, const float* const* values, const int* broadcast, int n_curves) {
    try {
        std::vector<Klangraum::FX8010Chain::HostCurve> cv;
        for (int j = 0; j < n_curves; ++j) cv.push_back(Klangraum::FX8010Chain::HostCurve{stages[j], names[j], values[j], broadcast[j] != 0});
        c->chain.processBlockWithCurves(in, out, n_samples, cv);
        return 0;
    } catch (const std::exception& e) { c->err = e.what(); return 1; }
}
const char* fx8010_host_chain_last_error(fx8010_host_chain* c) { return c ? c->err.c_str() : g_chain_create_error.c_str(); }

}  // extern "C"
