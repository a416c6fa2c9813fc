// Process-wide state of the octm library: error string, launch counter, device properties, host-mapped report cells.
#include "common.cuh"

#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

namespace octm {

std::atomic<int> g_profile{0};
namespace {
struct ProfRec {
    const char* name;
    cudaEvent_t a, b;
};
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof_recs;
}  // namespace

void ProfScope::begin(const char* name) {
    ProfRec r{name, nullptr, nullptr};
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    cudaEventRecord(r.a, stream);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    slot = static_cast<int>(g_prof_recs.size());
    g_prof_recs.push_back(r);
}

void ProfScope::end() {
    cudaEvent_t b;
    {
        std::lock_guard<std::mutex> lk(g_prof_mu);
        b = g_prof_recs[slot].b;
    }
    cudaEventRecord(b, stream);
}

thread_local char g_last_error[512] = "";
std::atomic<uint64_t> g_launches{0};

int sm_count() {
    static thread_local int cached_dev = -1, cached = 148;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) cached = v;
        cached_dev = dev;
    }
    return cached;
}

int max_optin_smem() {
    static thread_local int cached_dev = -1, cached = 227 * 1024;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) == cudaSuccess && v > 0) cached = v;
        cached_dev = dev;
    }
    return cached;
}

HostReport* host_report(int slot) {
    static HostReport cells[64][2];
    static std::mutex mu;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return nullptr; }
    std::lock_guard<std::mutex> lk(mu);
    HostReport& r = cells[dev][slot];
    if (r.host == nullptr) {
        void* h = nullptr;
        void* d = nullptr;
        if (cudaHostAlloc(&h, 2 * sizeof(uint32_t), cudaHostAllocMapped) != cudaSuccess || cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        r.host = static_cast<uint32_t*>(h);
        r.dev = static_cast<uint32_t*>(d);
        r.host[0] = r.host[1] = 0;
    }
    return &r;
}

}  // namespace octm

extern "C" int octm_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(octm::g_prof_mu);
    for (auto& r : octm::g_prof_recs) {
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    octm::g_prof_recs.clear();
    octm::g_profile.store(on ? 1 : 0);
    return OCTM_OK;
}

extern "C" size_t octm_profile_report(char* buf, size_t cap) {
    std::map<std::string, std::pair<long long, double>> agg;       // name -> (launches, ms)
    std::vector<std::string> order;
    {
        std::lock_guard<std::mutex> lk(octm::g_prof_mu);
        for (auto& r : octm::g_prof_recs) {
            float ms = 0.f;
            if (cudaEventSynchronize(r.b) != cudaSuccess || cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) {
                cudaGetLastError();
                continue;
            }
            auto it = agg.find(r.name);
            if (it == agg.end()) {
                order.push_back(r.name);
                agg[r.name] = {1, ms};
            } else {
                it->second.first += 1;
                it->second.second += ms;
            }
        }
    }
    std::string out;
    char line[160];
    for (auto& n : order) {
        snprintf(line, sizeof(line), "%s %lld %.6f\n", n.c_str(), agg[n].first, agg[n].second);
        out += line;
    }
    if (buf != nullptr && cap > 0) {
        const size_t m = out.size() < cap - 1 ? out.size() : cap - 1;
        memcpy(buf, out.data(), m);
        buf[m] = 0;
    }
    return out.size() + 1;
}

extern "C" int octm_abi_version(void) { return OCTM_ABI_VERSION; }
extern "C" const char* octm_last_error(void) { return octm::g_last_error; }
extern "C" uint64_t octm_launch_count(void) { return octm::g_launches.load(std::memory_order_relaxed); }
