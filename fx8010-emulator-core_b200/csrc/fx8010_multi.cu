// fx8010_multi.cu — the multi-GPU executor of include/fx8010_multi.h: one fx8010_gpu handle per shard, one persistent
// host thread per shard (SURVEY.md §7 step 8 / §8e: contiguous instance ranges, one host thread + streams per GPU,
// outputs gathered into one host buffer, no collective on the data path).
//
// Every entry point hands a job to all shard threads and waits for them; the threads call the single-device C ABI
// (fx8010_gpu.cu) with pointers into the caller's buffers, so scatter and gather ARE the per-device strided copies.
#include <cuda_runtime.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "fx8010_multi.h"

namespace {

struct Shard {
    int g = 0, device = 0, lo = 0, hi = 0;
    fx8010_gpu* h = nullptr;
    std::thread th;
    // job hand-off
    std::function<int(Shard&)> job;
    bool has_job = false, stop = false;
    int rc = 0;
    std::string err;
};

}  // namespace

struct fx8010_multi {
    int N = 0, C = 0;
    std::vector<Shard*> shards;
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    int pending = 0;
    std::string err;
};

namespace {

void worker(fx8010_multi* m, Shard* s) {
    cudaSetDevice(s->device);
    while (true) {
        std::function<int(Shard&)> job;
        {
            std::unique_lock<std::mutex> lk(m->mu);
            m->cv_job.wait(lk, [&] { return s->has_job || s->stop; });
            if (s->stop) return;
            job = s->job;
        }
        const int rc = job(*s);
        {
            std::lock_guard<std::mutex> lk(m->mu);
            s->rc = rc;
            if (rc) s->err = s->h ? fx8010_gpu_last_error(s->h) : fx8010_gpu_last_error(nullptr);
            s->has_job = false;
            if (--m->pending == 0) m->cv_done.notify_all();
        }
    }
}

// Runs `job` on every shard thread and waits; the first failure is reported.
int run_all(fx8010_multi* m, const std::function<int(Shard&)>& job) {
    {
        std::lock_guard<std::mutex> lk(m->mu);
        for (Shard* s : m->shards) { s->job = job; s->has_job = true; s->rc = 0; }
        m->pending = (int)m->shards.size();
    }
    m->cv_job.notify_all();
    std::unique_lock<std::mutex> lk(m->mu);
    m->cv_done.wait(lk, [&] { return m->pending == 0; });
    for (Shard* s : m->shards)
        if (s->rc) { m->err = "device " + std::to_string(s->device) + " (instances " + std::to_string(s->lo) + ".." + std::to_string(s->hi) + "): " + s->err; return s->rc; }
    return FX8010_OK;
}

thread_local std::string g_multi_create_error;

}  // namespace

extern "C" {

void fx8010_multi_shard_range(int n_total, int g, int G, int* lo, int* hi) {
    if (G <= 0) G = 1;
    if (lo) *lo = (int)(((long long)n_total * g) / G);
    if (hi) *hi = (int)(((long long)n_total * (g + 1)) / G);
}

int fx8010_multi_create(const int* devices, int n_devices, int n_instances, int n_channels, fx8010_multi** out) {
    if (!out) return FX8010_ERR_ARG;
    *out = nullptr;
    if (!devices || n_devices <= 0 || n_instances < n_devices || n_channels <= 0) {
        g_multi_create_error = "need at least one device, one instance per device and one channel";
        return FX8010_ERR_ARG;
    }
    fx8010_multi* m = new fx8010_multi();
    m->N = n_instances; m->C = n_channels;
    for (int g = 0; g < n_devices; ++g) {
        Shard* s = new Shard();
        s->g = g; s->device = devices[g];
        fx8010_multi_shard_range(n_instances, g, n_devices, &s->lo, &s->hi);
        const int rc = fx8010_gpu_create(s->device, s->hi - s->lo, n_channels, &s->h);
        if (rc) {
            g_multi_create_error = std::string("shard ") + std::to_string(g) + ": " + fx8010_gpu_last_error(nullptr);
            delete s;
            fx8010_multi_destroy(m);
            return rc;
        }
        m->shards.push_back(s);
    }
    for (Shard* s : m->shards) s->th = std::thread(worker, m, s);
    *out = m;
    return FX8010_OK;
}

void fx8010_multi_destroy(fx8010_multi* m) {
    if (!m) return;
    {
        std::lock_guard<std::mutex> lk(m->mu);
        for (Shard* s : m->shards) s->stop = true;
    }
    m->cv_job.notify_all();
    for (Shard* s : m->shards) {
        if (s->th.joinable()) s->th.join();
        if (s->h) fx8010_gpu_destroy(s->h);
        delete s;
    }
    delete m;
}

int fx8010_multi_num_shards(fx8010_multi* m) { return m ? (int)m->shards.size() : 0; }

fx8010_gpu* fx8010_multi_shard(fx8010_multi* m, int g, int* lo, int* hi) {
    if (!m || g < 0 || g >= (int)m->shards.size()) return nullptr;
    if (lo) *lo = m->shards[g]->lo;
    if (hi) *hi = m->shards[g]->hi;
    return m->shards[g]->h;
}

int fx8010_multi_load_program(fx8010_multi* m, const fx8010_program_image* image) {
    if (!m) return FX8010_ERR_ARG;
    return run_all(m, [image](Shard& s) { return fx8010_gpu_load_program(s.h, image); });
}

int fx8010_multi_set_controls(fx8010_multi* m, int reg_index, const float* values, int broadcast) {
    if (!m || !values) return FX8010_ERR_ARG;
    return run_all(m, [=](Shard& s) { return fx8010_gpu_set_controls(s.h, reg_index, broadcast ? values : values + s.lo, broadcast); });
}

int fx8010_multi_get_register(fx8010_multi* m, int reg_index, float* out) {
    if (!m || !out) return FX8010_ERR_ARG;
    return run_all(m, [=](Shard& s) { return fx8010_gpu_get_register(s.h, reg_index, out + s.lo); });
}

static int multi_process(fx8010_multi* m, const float* in, float* out, int n_samples, int wait) {
    if (!m || !out || n_samples < 0) return FX8010_ERR_ARG;
    const size_t N = (size_t)m->N;
    return run_all(m, [=](Shard& s) {
        return fx8010_gpu_process_batch_host_slice(s.h, in ? in + s.lo : nullptr, out + s.lo, n_samples, N, wait);
    });
}
int fx8010_multi_process_batch_host(fx8010_multi* m, const float* in, float* out, int n_samples) { return multi_process(m, in, out, n_samples, 1); }
int fx8010_multi_process_batch_host_async(fx8010_multi* m, const float* in, float* out, int n_samples) { return multi_process(m, in, out, n_samples, 0); }

int fx8010_multi_process_batch_host_broadcast(fx8010_multi* m, const float* in, float* out, int n_samples, int wait) {
    if (!m || !out || n_samples < 0) return FX8010_ERR_ARG;
    const size_t N = (size_t)m->N;
    return run_all(m, [=](Shard& s) { return fx8010_gpu_process_batch_host_broadcast(s.h, in, out + s.lo, n_samples, N, wait); });
}

void fx8010_multi_shard_curves(const fx8010_host_curve* curves, int n_curves, int n_total, int g, int G, fx8010_host_curve* out) {
    int lo = 0;
    fx8010_multi_shard_range(n_total, g, G, &lo, nullptr);
    for (int j = 0; j < n_curves; ++j) {
        out[j] = curves[j];
        if (!curves[j].broadcast && curves[j].values) out[j].values = curves[j].values + lo;
    }
}

int fx8010_multi_process_batch_host_curves(fx8010_multi* m, const float* in, float* out, int n_samples, const fx8010_host_curve* curves, int n_curves,
                                           int wait) {
    if (!m || !out || n_samples < 0 || n_curves < 0 || n_curves > FX8010_MAX_CONTROL_CURVES || (n_curves > 0 && !curves)) return FX8010_ERR_ARG;
    const size_t N = (size_t)m->N;
    const int G = (int)m->shards.size();
    // Every shard checks the list before it queues anything, against the same program: a list one shard refuses, all refuse.
    return run_all(m, [=](Shard& s) {
        fx8010_host_curve mine[FX8010_MAX_CONTROL_CURVES];
        fx8010_multi_shard_curves(curves, n_curves, m->N, s.g, G, mine);
        return fx8010_gpu_process_batch_host_curves(s.h, in ? in + s.lo : nullptr, out + s.lo, n_samples, mine, n_curves, N, wait);
    });
}

int fx8010_multi_set_option(fx8010_multi* m, int option, int value) {
    if (!m) return FX8010_ERR_ARG;
    return run_all(m, [option, value](Shard& s) { return fx8010_gpu_set_option(s.h, option, value); });
}

int fx8010_multi_synchronize(fx8010_multi* m) {
    if (!m) return FX8010_ERR_ARG;
    return run_all(m, [](Shard& s) { return fx8010_gpu_synchronize(s.h, nullptr); });
}

int fx8010_multi_get_instruction_count(fx8010_multi* m, unsigned long long* total) {
    if (!m || !total) return FX8010_ERR_ARG;
    std::vector<unsigned long long> part(m->shards.size(), 0);
    Shard* const* base = m->shards.data();
    const int rc = run_all(m, [&part, base](Shard& s) {
        size_t g = 0;
        while (base[g] != &s) ++g;
        return fx8010_gpu_get_instruction_count(s.h, &part[g]);
    });
    if (rc) return rc;
    *total = 0;
    for (unsigned long long v : part) *total += v;
    return FX8010_OK;
}

int fx8010_multi_get_registers(fx8010_multi* m, float* out) {
    if (!m || !out) return FX8010_ERR_ARG;
    const size_t N = (size_t)m->N;
    return run_all(m, [=](Shard& s) {
        fx8010_state_dims d;
        int rc = fx8010_gpu_get_dims(s.h, &d);
        if (rc) return rc;
        const size_t n = (size_t)(s.hi - s.lo);
        std::vector<float> tmp((size_t)d.n_regs * n);
        rc = fx8010_gpu_get_registers(s.h, tmp.data());
        if (rc) return rc;
        for (int r = 0; r < d.n_regs; ++r) std::copy(tmp.begin() + (size_t)r * n, tmp.begin() + (size_t)(r + 1) * n, out + (size_t)r * N + s.lo);
        return (int)FX8010_OK;
    });
}

int fx8010_multi_get_runtime_flags(fx8010_multi* m, unsigned int* flags, int clear) {
    if (!m || !flags) return FX8010_ERR_ARG;
    std::vector<unsigned int> part(m->shards.size(), 0);
    Shard* const* base = m->shards.data();
    const int rc = run_all(m, [&part, base, clear](Shard& s) {
        size_t g = 0;
        while (base[g] != &s) ++g;
        return fx8010_gpu_get_runtime_flags(s.h, &part[g], clear);
    });
    if (rc) return rc;
    *flags = 0;
    for (unsigned int v : part) *flags |= v;
    return FX8010_OK;
}

const char* fx8010_multi_last_error(fx8010_multi* m) { return m ? m->err.c_str() : g_multi_create_error.c_str(); }

void fx8010_multi_shard_chain_curves(const fx8010_chain_host_curve* curves, int n_curves, int n_total, int g, int G, fx8010_chain_host_curve* out) {
    int lo = 0;
    fx8010_multi_shard_range(n_total, g, G, &lo, nullptr);
    for (int j = 0; j < n_curves; ++j) {
        out[j] = curves[j];
        if (!curves[j].broadcast && curves[j].values) out[j].values = curves[j].values + lo;
    }
}

}  // extern "C"

// A chain of executors (fx8010_multi_chain_*): one fx8010_chain per shard over the stages' handles of that shard, driven by the shard
// threads of stage 0's executor.
struct fx8010_multi_chain {
    fx8010_multi* m = nullptr;                       // stage 0's executor (its threads run the calls)
    std::vector<fx8010_chain*> chains;               // per shard
    std::string err;
};

namespace {

thread_local std::string g_multi_chain_create_error;

int multi_chain_fail(const std::string& msg) {
    g_multi_chain_create_error = msg;
    return FX8010_ERR_ARG;
}

// Runs `job` (shard g's chain) on every shard thread of the chain; a failure is reported with the chain's own error text.
int multi_chain_run(fx8010_multi_chain* mc, const std::function<int(Shard&, fx8010_chain*)>& job) {
    const int rc = run_all(mc->m, [&](Shard& s) { return job(s, mc->chains[(size_t)s.g]); });
    if (rc == FX8010_OK) return rc;
    for (Shard* s : mc->m->shards) {
        if (!s->rc) continue;
        mc->err = "device " + std::to_string(s->device) + " (instances " + std::to_string(s->lo) + ".." + std::to_string(s->hi) + "): " +
                  fx8010_chain_last_error(mc->chains[(size_t)s->g]);
        break;
    }
    return rc;
}

int multi_chain_process(fx8010_multi_chain* mc, const float* in, float* out, int n_samples, const fx8010_chain_host_curve* curves, int n_curves,
                        int wait) {
    if (!mc) return FX8010_ERR_ARG;
    if (!out || n_samples < 0) {
        mc->err = "out is NULL or n_samples negative";
        return FX8010_ERR_ARG;
    }
    if (n_curves < 0 || n_curves > FX8010_MAX_CONTROL_CURVES || (n_curves > 0 && !curves)) {
        mc->err = "the curve list is NULL or the curve count outside 0..8";
        return FX8010_ERR_ARG;
    }
    fx8010_multi* m = mc->m;
    const size_t N = (size_t)m->N;
    const int G = (int)m->shards.size();
    // Every shard checks the list before it queues anything, against the same programs: a list one shard refuses, all refuse.
    return multi_chain_run(mc, [=](Shard& s, fx8010_chain* c) {
        fx8010_chain_host_curve mine[FX8010_MAX_CONTROL_CURVES];
        fx8010_multi_shard_chain_curves(curves, n_curves, m->N, s.g, G, mine);
        return fx8010_chain_process_batch_host_curves(c, in ? in + s.lo : nullptr, out + s.lo, n_samples, mine, n_curves, N, wait);
    });
}

}  // namespace

extern "C" {

int fx8010_multi_chain_create(fx8010_multi* const* stages, int n_stages, fx8010_multi_chain** out) {
    if (!out) return multi_chain_fail("out is NULL");
    *out = nullptr;
    if (!stages || n_stages < 1 || n_stages > FX8010_MAX_CHAIN_STAGES) return multi_chain_fail("the stage count must be 1..FX8010_MAX_CHAIN_STAGES");
    for (int j = 0; j < n_stages; ++j) {
        if (!stages[j]) return multi_chain_fail("stage " + std::to_string(j) + " is NULL");
        for (int k = 0; k < j; ++k) if (stages[k] == stages[j]) return multi_chain_fail("an executor appears twice in the chain");
        if (stages[j]->N != stages[0]->N || stages[j]->C != stages[0]->C)
            return multi_chain_fail("stage " + std::to_string(j) + " differs in instance count or channel count");
        if (stages[j]->shards.size() != stages[0]->shards.size())
            return multi_chain_fail("stage " + std::to_string(j) + " differs in shard count");
        for (size_t g = 0; g < stages[0]->shards.size(); ++g)
            if (stages[j]->shards[g]->device != stages[0]->shards[g]->device)
                return multi_chain_fail("stage " + std::to_string(j) + ": shard " + std::to_string(g) + " is on another device");
    }
    fx8010_multi_chain* mc = new fx8010_multi_chain();
    mc->m = stages[0];
    for (size_t g = 0; g < stages[0]->shards.size(); ++g) {
        std::vector<fx8010_gpu*> h;
        for (int j = 0; j < n_stages; ++j) h.push_back(stages[j]->shards[g]->h);
        fx8010_chain* c = nullptr;
        const int rc = fx8010_chain_create(h.data(), n_stages, &c);
        if (rc) {
            g_multi_chain_create_error = "shard " + std::to_string(g) + ": " + fx8010_chain_last_error(nullptr);
            fx8010_multi_chain_destroy(mc);
            return rc;
        }
        mc->chains.push_back(c);
    }
    *out = mc;
    return FX8010_OK;
}

void fx8010_multi_chain_destroy(fx8010_multi_chain* mc) {
    if (!mc) return;
    for (fx8010_chain* c : mc->chains) fx8010_chain_destroy(c);
    delete mc;
}

int fx8010_multi_chain_process_batch_host(fx8010_multi_chain* mc, const float* in, float* out, int n_samples, int wait) {
    return multi_chain_process(mc, in, out, n_samples, nullptr, 0, wait);
}

int fx8010_multi_chain_process_batch_host_curves(fx8010_multi_chain* mc, const float* in, float* out, int n_samples,
                                                 const fx8010_chain_host_curve* curves, int n_curves, int wait) {
    return multi_chain_process(mc, in, out, n_samples, curves, n_curves, wait);
}

int fx8010_multi_chain_synchronize(fx8010_multi_chain* mc) {
    if (!mc) return FX8010_ERR_ARG;
    return multi_chain_run(mc, [](Shard&, fx8010_chain* c) { return fx8010_chain_synchronize(c); });
}

fx8010_chain* fx8010_multi_chain_shard(fx8010_multi_chain* mc, int g) {
    if (!mc || g < 0 || g >= (int)mc->chains.size()) return nullptr;
    return mc->chains[(size_t)g];
}

const char* fx8010_multi_chain_last_error(fx8010_multi_chain* mc) { return mc ? mc->err.c_str() : g_multi_chain_create_error.c_str(); }

}  // extern "C"
