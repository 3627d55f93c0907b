// FX8010.h — drop-in for the reference's class Klangraum::FX8010 (reference include/FX8010.h:47-302)
// on top of the B200 executor.  The public members of the reference keep their names, arguments
// and return conventions; the batched members below them are the reason this library exists: one
// parsed program executed over N independent DSP instances on one GPU.
//
// There is no CPU interpreter behind this class: process*/ need a CUDA device and throw
// std::runtime_error when the C ABI (include/fx8010_gpu.h) reports an error.
#ifndef FX8010_B200_FACADE_H
#define FX8010_B200_FACADE_H

#include <string>
#include <unordered_map>
#include <vector>

#include "fx8010_frontend.h"
#include "fx8010_gpu.h"
#include "fx8010_multi.h"

#if defined(__GNUC__)
#define FX8010_CLASS __attribute__((visibility("default")))
#else
#define FX8010_CLASS
#endif

namespace Klangraum {

class FX8010_CLASS FX8010 {
public:
    // ---- the reference's surface (include/FX8010.h:49-75) --------------------------------------
    FX8010(int numChannels);                                   // one instance on device 0
    ~FX8010();
    void initialize();                                         // re-runs the constructor's set-up (appends, like the reference)
    std::vector<float> process(const std::vector<float>& inputSamples);   // one sample period (:57)
    int getInstructionCounter();                               // executed instructions of instance 0 (:60)
    bool loadFile(const std::string& path);                    // (:62) appends to what is loaded, like the reference; the next process*
                                                               // call uploads the new image, which RESETS the run-time state of every
                                                               // instance (registers, TRAM, accumulator, LFSR, counters) — the reference
                                                               // object keeps its state across an appending load
    struct MyError {
        std::string errorDescription = "";
        int errorRow = 1;
    };
    std::vector<FX8010::MyError> getErrorList();               // (:68)
    int setRegisterValue(const std::string& key, float value); // 0 ok / 1 unknown name; every instance (:69)
    float getRegisterValue(const std::string& key);            // instance 0; 1 when unknown (:70)
    std::vector<std::string> getControlRegisters();            // (:71)
    std::unordered_map<std::string, std::string> getMetaData();// (:72)
    inline void setChannels(int numChannels_) { front_.setChannels(numChannels_); }
    inline int getChannels() { return front_.channels(); }
    bool getReadyStatus() { return front_.ready(); }

    // ---- batched extension ------------------------------------------------------------------------
    FX8010(int numChannels, int numInstances, int device);
    // numInstances spread over several GPUs of one box (contiguous instance ranges, include/fx8010_multi.h): the host-buffer
    // members (process, processBlock, processBlockWithCurves, set/getRegisterValue(s), the counters) work as on one device and
    // gather into the caller's buffers; the device-pointer members have no single device to refer to and throw
    FX8010(int numChannels, int numInstances, const std::vector<int>& devices);
    bool loadText(const std::string& source);
    void setRelaxedSyntax(bool on) { front_.setRelaxed(on); }   // accept the README's forms too (see fx8010_frontend.h)
    int getInstances() const { return instances_; }
    // per-instance control values, values[numInstances]; 0 ok / 1 unknown name
    int setRegisterValues(const std::string& key, const float* values);
    // reads one register of every instance into out[numInstances]; 0 ok / 1 unknown name
    int getRegisterValues(const std::string& key, float* out);
    // n_samples sample periods for all instances; HOST buffers laid out [channel][sample][instance]
    void processBlock(const float* in, float* out, int n_samples);
    // same with DEVICE buffers, asynchronous on `stream` (a cudaStream_t)
    void processBlockDevice(const float* d_in, float* d_out, int n_samples, void* stream);
    // the driver's slider pattern (source/main.cpp:107-114) inside one block: `key` takes `value` for every instance
    // right before sample period `sample`; DEVICE buffers, asynchronous on `stream`
    struct ControlChange { int sample; std::string key; float value; };
    void processBlockDeviceWithControls(const float* d_in, float* d_out, int n_samples,
                                        const std::vector<ControlChange>& changes, void* stream);
    // sample-accurate automation (include/fx8010_gpu.h, fx8010_gpu_process_batch_curves): register `key` takes d_values[s] (broadcast: one
    // value for every instance, d_values[n_samples]) or d_values[s * numInstances + i] (d_values[n_samples][numInstances]) right before
    // sample period s; DEVICE buffers, asynchronous on `stream`; throws on an unknown name
    struct Curve { std::string key; const float* d_values; bool broadcast; };
    void processBlockDeviceWithCurves(const float* d_in, float* d_out, int n_samples, const std::vector<Curve>& curves, void* stream);
    // the same automation with HOST buffers, on one device or several: `key` takes values[s] (broadcast, values[n_samples]) or
    // values[s * numInstances + i] (values[n_samples][numInstances]) right before sample period s; in / out as in processBlock; each
    // pipelined sub-block copies its rows of the curves to the device with its inputs (include/fx8010_gpu.h,
    // fx8010_gpu_process_batch_host_curves); returns when `out` is complete; throws on an unknown name
    struct HostCurve { std::string key; const float* values; bool broadcast; };
    void processBlockWithCurves(const float* in, float* out, int n_samples, const std::vector<HostCurve>& curves);
    // DEVICE buffers laid out [channel][instance][sample] (planar audio), asynchronous on `stream`
    void processBlockDevicePlanar(const float* d_in, float* d_out, int n_samples, void* stream);
    // program translator (include/fx8010_gpu.h, FX8010_OPT_TRANSLATE): 0 interpreter kernels only, 1 compile in the background and switch
    // over when the kernel is loaded (default), 2 compile before the first block
    void setTranslation(int mode);
    // the translator's disk kernel cache for the whole process (include/fx8010_gpu.h, fx8010_kernel_cache_set_dir): translated kernels
    // compiled once are reused by later processes; "" turns it off (it is off unless FX8010_KERNEL_CACHE names a directory)
    static void setKernelCacheDir(const std::string& dir);
    unsigned long long getInstructionCounterTotal();           // summed over instances
    fx8010_gpu* gpuHandle();                                   // creates the handle / uploads the program if needed
    fx8010::Frontend& frontend() { return front_; }

private:
    void ensureUploaded();
    void check(int rc, const char* what);

    fx8010::Frontend front_;
    int instances_ = 1;
    int device_ = 0;
    fx8010_gpu* gpu_ = nullptr;
    std::vector<int> devices_;                                 // more than one entry: the multi-GPU executor below is used instead of gpu_
    fx8010_multi* multi_ = nullptr;
    int translate_mode_ = -1;                                  // -1: the library's default
    bool uploaded_ = false;                                    // the device holds the image of generation uploaded_generation_
    unsigned long uploaded_generation_ = 0;
    std::vector<float> in_block_, out_block_;
};

}  // namespace Klangraum

#endif
