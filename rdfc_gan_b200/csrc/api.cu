// Library-wide state of librdfc_b200.so: error string, launch counter, device queries.
#include <atomic>
#include <map>
#include <mutex>
#include <stdlib.h>
#include <string>

#include "common.cuh"

namespace rdfc {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

char *err_buf() { return g_err; }

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

void count_launch(unsigned n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
    }
    return n;
}

TmapEncodeFn tmap_encoder() {
    static const TmapEncodeFn fn = [] {
        cudaDriverEntryPointQueryResult q;
        void *p = nullptr;
        const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                        q == cudaDriverEntryPointSuccess;
        (void)cudaGetLastError();
        return ok ? (TmapEncodeFn)p : nullptr;
    }();
    return fn;
}

// Development knobs (RDFC_* environment variables): read ONCE per name, then served from a table, so no launch path calls
// getenv; rdfc_dev_set_knob overrides a value at run time (tests sweep the NLSPN band halo that way).
static std::mutex g_knob_mu;
static std::map<std::string, long long> g_knobs;

long long knob(const char *name, long long dflt) {
    std::lock_guard<std::mutex> lk(g_knob_mu);
    auto it = g_knobs.find(name);
    if (it != g_knobs.end()) return it->second == KNOB_UNSET ? dflt : it->second;
    const char *e = getenv(name);
    g_knobs[name] = e ? atoll(e) : KNOB_UNSET;
    return e ? atoll(e) : dflt;
}

}  // namespace rdfc

extern "C" int rdfc_dev_set_knob(const char *name, long long value) {
    if (!name) return RDFC_ERR_INVALID;
    std::lock_guard<std::mutex> lk(rdfc::g_knob_mu);
    rdfc::g_knobs[name] = value;
    return 0;
}

extern "C" int rdfc_abi_version(void) { return RDFC_ABI_VERSION; }
extern "C" const char *rdfc_last_error(void) { return rdfc::err_buf(); }
extern "C" uint64_t rdfc_launch_count(void) { return rdfc::g_launches.load(); }
