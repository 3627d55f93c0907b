// FX8010.cpp — the Klangraum::FX8010 facade (see FX8010.h).  Parsing is host C++ (fx8010_frontend);
// every sample is computed by the CUDA interpreter behind the C ABI.
#include "FX8010.h"

#include <stdexcept>

namespace Klangraum {

FX8010::FX8010(int numChannels) : front_(numChannels) {}
FX8010::FX8010(int numChannels, int numInstances, int device)
    : front_(numChannels), instances_(numInstances), device_(device) {}

FX8010::FX8010(int numChannels, int numInstances, const std::vector<int>& devices)
    : front_(numChannels), instances_(numInstances), device_(devices.empty() ? 0 : devices[0]), devices_(devices) {}

FX8010::~FX8010() {
    if (gpu_) fx8010_gpu_destroy(gpu_);
    if (multi_) fx8010_multi_destroy(multi_);
}

void FX8010::initialize() { front_.initialize(); }

void FX8010::check(int rc, const char* what) {
    if (rc == FX8010_OK) return;
    std::string msg = std::string("FX8010 (B200): ") + what + " failed: " + (multi_ ? fx8010_multi_last_error(multi_) : fx8010_gpu_last_error(gpu_));
    throw std::runtime_error(msg);
}

bool FX8010::loadFile(const std::string& path) { return front_.loadFile(path); }
bool FX8010::loadText(const std::string& source) { return front_.loadText(source); }

void FX8010::ensureUploaded() {
    if (!front_.ready()) throw std::runtime_error("FX8010 (B200): process() before a successful loadFile()");
    if (devices_.size() > 1) {                                 // instances sharded over several GPUs
        if (!multi_) {
            const int rc = fx8010_multi_create(devices_.data(), (int)devices_.size(), instances_, front_.channels(), &multi_);
            if (rc != FX8010_OK) {
                std::string msg = std::string("FX8010 (B200): no multi-GPU executor: ") + fx8010_multi_last_error(nullptr);
                multi_ = nullptr;
                throw std::runtime_error(msg);
            }
        }
        if (translate_mode_ >= 0) check(fx8010_multi_set_option(multi_, FX8010_OPT_TRANSLATE, translate_mode_), "set_option");
        if (!uploaded_ || uploaded_generation_ != front_.generation()) {
            check(fx8010_multi_load_program(multi_, front_.image()), "load_program");
            uploaded_ = true;
            uploaded_generation_ = front_.generation();
        }
        return;
    }
    if (!gpu_) {
        const int rc = fx8010_gpu_create(device_, instances_, front_.channels(), &gpu_);
        if (rc != FX8010_OK) {
            std::string msg = std::string("FX8010 (B200): no GPU executor: ") + fx8010_gpu_last_error(nullptr);
            gpu_ = nullptr;
            throw std::runtime_error(msg);
        }
    }
    // The image the device holds is stale after ANY later loadFile/loadText/initialize (they append, like the
    // reference, source/FX8010.cpp:777-875 — but an edit that keeps the counts equal must be noticed too).  A reload
    // puts every instance back into the state of a freshly loaded object (see FX8010.h).
    if (translate_mode_ >= 0) check(fx8010_gpu_set_option(gpu_, FX8010_OPT_TRANSLATE, translate_mode_), "set_option");
    if (!uploaded_ || uploaded_generation_ != front_.generation()) {
        check(fx8010_gpu_load_program(gpu_, front_.image()), "load_program");
        uploaded_ = true;
        uploaded_generation_ = front_.generation();
    }
}

FX8010Chain::FX8010Chain(const std::vector<FX8010*>& stages) : stages_(stages) {
    for (FX8010* s : stages_)
        if (!s) throw std::runtime_error("FX8010Chain (B200): a stage is NULL");
    if (stages_.empty() || !stages_[0]->multiHandle()) {
        std::vector<fx8010_gpu*> h;
        for (FX8010* s : stages_) {
            if (s->multiHandle()) throw std::runtime_error("FX8010Chain (B200): objects on one device and on several cannot be mixed");
            h.push_back(s->gpuHandle());
        }
        if (fx8010_chain_create(h.data(), (int)h.size(), &chain_) != FX8010_OK)
            throw std::runtime_error(std::string("FX8010Chain (B200): ") + fx8010_chain_last_error(nullptr));
        return;
    }
    std::vector<fx8010_multi*> m;
    for (FX8010* s : stages_) {
        fx8010_multi* e = s->multiHandle();
        if (!e) throw std::runtime_error("FX8010Chain (B200): objects on one device and on several cannot be mixed");
        m.push_back(e);
    }
    if (fx8010_multi_chain_create(m.data(), (int)m.size(), &multi_) != FX8010_OK)
        throw std::runtime_error(std::string("FX8010Chain (B200): ") + fx8010_multi_chain_last_error(nullptr));
}

FX8010Chain::~FX8010Chain() {
    fx8010_chain_destroy(chain_);
    fx8010_multi_chain_destroy(multi_);
}

void FX8010Chain::upload() {
    for (FX8010* s : stages_) s->multiHandle();                // (ensures the upload on one device and on several)
}

int FX8010Chain::registerOf(int stage, const std::string& key) {
    if (stage < 0 || stage >= (int)stages_.size())
        throw std::runtime_error("FX8010Chain (B200): curve stage " + std::to_string(stage) + " out of range");
    const int reg = stages_[stage]->frontend().findRegister(key);
    if (reg < 0) throw std::runtime_error("FX8010Chain: unknown register '" + key + "' of stage " + std::to_string(stage));
    return reg;
}

void FX8010Chain::processBlock(const float* in, float* out, int n_samples) {
    upload();
    const int rc = multi_ ? fx8010_multi_chain_process_batch_host(multi_, in, out, n_samples, 1)
                          : fx8010_chain_process_batch_host(chain_, in, out, n_samples, 0, 1);
    if (rc != FX8010_OK)
        throw std::runtime_error(std::string("FX8010Chain (B200): process_batch_host failed: ") +
                                 (multi_ ? fx8010_multi_chain_last_error(multi_) : fx8010_chain_last_error(chain_)));
}

void FX8010Chain::processBlockWithCurves(const float* in, float* out, int n_samples, const std::vector<HostCurve>& curves) {
    upload();
    std::vector<fx8010_chain_host_curve> cv;
    for (const HostCurve& c : curves) cv.push_back(fx8010_chain_host_curve{c.stage, registerOf(c.stage, c.key), c.broadcast ? 1 : 0, 0, c.values});
    const int rc = multi_ ? fx8010_multi_chain_process_batch_host_curves(multi_, in, out, n_samples, cv.data(), (int)cv.size(), 1)
                          : fx8010_chain_process_batch_host_curves(chain_, in, out, n_samples, cv.data(), (int)cv.size(), 0, 1);
    if (rc != FX8010_OK)
        throw std::runtime_error(std::string("FX8010Chain (B200): process_batch_host_curves failed: ") +
                                 (multi_ ? fx8010_multi_chain_last_error(multi_) : fx8010_chain_last_error(chain_)));
}

void FX8010Chain::processBlockDevice(const float* d_in, float* d_out, int n_samples, void* stream) {
    if (multi_) throw std::runtime_error("FX8010Chain (B200): device-pointer members need a single device");
    upload();
    if (fx8010_chain_process_batch(chain_, d_in, d_out, n_samples, stream) != FX8010_OK)
        throw std::runtime_error(std::string("FX8010Chain (B200): process_batch failed: ") + fx8010_chain_last_error(chain_));
}

void FX8010Chain::processBlockDeviceWithCurves(const float* d_in, float* d_out, int n_samples, const std::vector<Curve>& curves, void* stream) {
    if (multi_) throw std::runtime_error("FX8010Chain (B200): device-pointer members need a single device");
    upload();
    std::vector<fx8010_chain_curve> cv;
    for (const Curve& c : curves) cv.push_back(fx8010_chain_curve{c.stage, registerOf(c.stage, c.key), c.broadcast ? 1 : 0, 0, c.d_values});
    if (fx8010_chain_process_batch_curves(chain_, d_in, d_out, n_samples, cv.data(), (int)cv.size(), stream) != FX8010_OK)
        throw std::runtime_error(std::string("FX8010Chain (B200): process_batch_curves failed: ") + fx8010_chain_last_error(chain_));
}

fx8010_gpu* FX8010::gpuHandle() {
    ensureUploaded();
    if (multi_) throw std::runtime_error("FX8010 (B200): this object drives several GPUs; there is no single device handle");
    return gpu_;
}

fx8010_multi* FX8010::multiHandle() {
    ensureUploaded();
    return multi_;
}

void FX8010::setTranslation(int mode) {
    if (mode < 0 || mode > 2) throw std::invalid_argument("FX8010 (B200): setTranslation takes 0, 1 or 2");
    translate_mode_ = mode;                                     // applied by the next process* call (ensureUploaded)
}

void FX8010::setKernelCacheDir(const std::string& dir) { fx8010_kernel_cache_set_dir(dir.c_str()); }

std::vector<float> FX8010::process(const std::vector<float>& inputSamples) {
    ensureUploaded();
    const size_t C = (size_t)front_.channels(), N = (size_t)instances_;
    in_block_.assign(C * N, 0.0f);
    out_block_.assign(C * N, 0.0f);
    for (size_t c = 0; c < C && c < inputSamples.size(); ++c)
        for (size_t i = 0; i < N; ++i) in_block_[c * N + i] = inputSamples[c];
    if (multi_) check(fx8010_multi_process_batch_host(multi_, in_block_.data(), out_block_.data(), 1), "process_batch_host");
    else check(fx8010_gpu_process_batch_host(gpu_, in_block_.data(), out_block_.data(), 1), "process_batch_host");
    std::vector<float> out(C);
    for (size_t c = 0; c < C; ++c) out[c] = out_block_[c * N];
    return out;
}

void FX8010::processBlock(const float* in, float* out, int n_samples) {
    ensureUploaded();
    if (multi_) check(fx8010_multi_process_batch_host(multi_, in, out, n_samples), "process_batch_host");
    else check(fx8010_gpu_process_batch_host(gpu_, in, out, n_samples), "process_batch_host");
}

void FX8010::processBlockDevice(const float* d_in, float* d_out, int n_samples, void* stream) {
    ensureUploaded();
    if (multi_) throw std::runtime_error("FX8010 (B200): device-pointer members need a single device");
    check(fx8010_gpu_process_batch(gpu_, d_in, d_out, n_samples, stream), "process_batch");
}

void FX8010::processBlockDeviceWithControls(const float* d_in, float* d_out, int n_samples,
                                            const std::vector<ControlChange>& changes, void* stream) {
    ensureUploaded();
    if (multi_) throw std::runtime_error("FX8010 (B200): device-pointer members need a single device");
    std::vector<fx8010_control_event> ev;
    std::vector<float> vals(changes.size());
    for (size_t i = 0; i < changes.size(); ++i) {
        const int reg = front_.findRegister(changes[i].key);
        if (reg < 0) throw std::runtime_error("FX8010: unknown register '" + changes[i].key + "'");
        vals[i] = changes[i].value;
        ev.push_back(fx8010_control_event{changes[i].sample, reg, 1, 0, &vals[i]});
        front_.registers()[reg].value = changes[i].value;    // initial value of a later upload, as setRegisterValue keeps it
    }
    check(fx8010_gpu_process_batch_events(gpu_, d_in, d_out, n_samples, ev.data(), (int)ev.size(), stream), "process_batch_events");
}

void FX8010::processBlockDeviceWithCurves(const float* d_in, float* d_out, int n_samples, const std::vector<Curve>& curves, void* stream) {
    ensureUploaded();
    if (multi_) throw std::runtime_error("FX8010 (B200): device-pointer members need a single device");
    std::vector<fx8010_control_curve> cv;
    for (const Curve& c : curves) {
        const int reg = front_.findRegister(c.key);
        if (reg < 0) throw std::runtime_error("FX8010: unknown register '" + c.key + "'");
        cv.push_back(fx8010_control_curve{reg, c.broadcast ? 1 : 0, c.d_values});
    }
    check(fx8010_gpu_process_batch_curves(gpu_, d_in, d_out, n_samples, cv.data(), (int)cv.size(), stream), "process_batch_curves");
}

void FX8010::processBlockWithCurves(const float* in, float* out, int n_samples, const std::vector<HostCurve>& curves) {
    ensureUploaded();
    std::vector<fx8010_host_curve> cv;
    for (const HostCurve& c : curves) {
        const int reg = front_.findRegister(c.key);
        if (reg < 0) throw std::runtime_error("FX8010: unknown register '" + c.key + "'");
        cv.push_back(fx8010_host_curve{reg, c.broadcast ? 1 : 0, c.values});
    }
    if (multi_) check(fx8010_multi_process_batch_host_curves(multi_, in, out, n_samples, cv.data(), (int)cv.size(), 1), "process_batch_host_curves");
    else check(fx8010_gpu_process_batch_host_curves(gpu_, in, out, n_samples, cv.data(), (int)cv.size(), 0, 1), "process_batch_host_curves");
}

void FX8010::processBlockDevicePlanar(const float* d_in, float* d_out, int n_samples, void* stream) {
    ensureUploaded();
    if (multi_) throw std::runtime_error("FX8010 (B200): device-pointer members need a single device");
    check(fx8010_gpu_process_batch_planar(gpu_, d_in, d_out, n_samples, stream), "process_batch_planar");
}

int FX8010::getInstructionCounter() {
    if (multi_ && uploaded_) {                                  // instance 0 lives on the first shard
        int lo = 0, hi = 0;
        fx8010_gpu* g0 = fx8010_multi_shard(multi_, 0, &lo, &hi);
        std::vector<unsigned long long> c((size_t)(hi - lo));
        if (fx8010_gpu_get_instruction_counts(g0, c.data()) != FX8010_OK) throw std::runtime_error("FX8010 (B200): get_instruction_counts failed");
        return (int)(unsigned int)c[0];
    }
    if (!gpu_ || !uploaded_) return 0;
    std::vector<unsigned long long> c((size_t)instances_);
    check(fx8010_gpu_get_instruction_counts(gpu_, c.data()), "get_instruction_counts");
    return (int)(unsigned int)c[0];                             // the reference counter is a 32-bit int
}

unsigned long long FX8010::getInstructionCounterTotal() {
    if (multi_ && uploaded_) {
        unsigned long long t = 0;
        check(fx8010_multi_get_instruction_count(multi_, &t), "get_instruction_count");
        return t;
    }
    if (!gpu_ || !uploaded_) return 0;
    unsigned long long t = 0;
    check(fx8010_gpu_get_instruction_count(gpu_, &t), "get_instruction_count");
    return t;
}

std::vector<FX8010::MyError> FX8010::getErrorList() {
    std::vector<MyError> out;
    for (const fx8010::Diagnostic& d : front_.errors()) {
        MyError e;
        e.errorDescription = d.description;
        e.errorRow = d.row;
        out.push_back(e);
    }
    return out;
}

// Any register can be written by name, first match wins (source/FX8010.cpp:236-253).
int FX8010::setRegisterValue(const std::string& key, float value) {
    const int idx = front_.findRegister(key);
    if (idx < 0) return 1;
    front_.registers()[idx].value = value;                      // initial value of a later upload
    if (multi_ && uploaded_ && uploaded_generation_ == front_.generation())
        check(fx8010_multi_set_controls(multi_, idx, &value, 1), "set_controls");
    else if (gpu_ && uploaded_ && uploaded_generation_ == front_.generation())
        check(fx8010_gpu_set_controls(gpu_, idx, &value, 1), "set_controls");
    return 0;
}

int FX8010::setRegisterValues(const std::string& key, const float* values) {
    const int idx = front_.findRegister(key);
    if (idx < 0) return 1;
    ensureUploaded();
    if (multi_) check(fx8010_multi_set_controls(multi_, idx, values, 0), "set_controls");
    else check(fx8010_gpu_set_controls(gpu_, idx, values, 0), "set_controls");
    return 0;
}

float FX8010::getRegisterValue(const std::string& key) {
    const int idx = front_.findRegister(key);
    if (idx < 0) return 1;                                      // the reference's "not found" value (:265)
    if ((gpu_ || multi_) && uploaded_ && uploaded_generation_ == front_.generation()) {
        std::vector<float> v((size_t)instances_);
        if (multi_) check(fx8010_multi_get_register(multi_, idx, v.data()), "get_register");
        else check(fx8010_gpu_get_register(gpu_, idx, v.data()), "get_register");
        return v[0];
    }
    return front_.registers()[idx].value;
}

int FX8010::getRegisterValues(const std::string& key, float* out) {
    const int idx = front_.findRegister(key);
    if (idx < 0) return 1;
    ensureUploaded();
    if (multi_) check(fx8010_multi_get_register(multi_, idx, out), "get_register");
    else check(fx8010_gpu_get_register(gpu_, idx, out), "get_register");
    return 0;
}

std::vector<std::string> FX8010::getControlRegisters() { return front_.controls(); }
std::unordered_map<std::string, std::string> FX8010::getMetaData() { return front_.metadata(); }

}  // namespace Klangraum
