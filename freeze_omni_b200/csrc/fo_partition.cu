// SM groups of a device for fo_create_on_sms: CUDA green contexts, reached through cudaGetDriverEntryPoint (no -lcuda).
//
// A split (device, sm_split) is made once per process and kept in a registry, so that contexts created with the same split get
// disjoint groups.  Each group's green context is created at its first use and lives as long as the process: the contexts that
// run on it may be destroyed and created again in any order.  Work reaches a group only through streams created in its green
// context (sm_group_stream); kernels launched there run on the group's SMs, graphs captured and replayed there too (DESIGN §5).
#include <cuda.h>
#include <string.h>

#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "fo_common.cuh"

namespace fo {

namespace {

#define FO_DRV_FN(name) decltype(&::name) p_##name = nullptr;
struct Driver {
    FO_DRV_FN(cuDeviceGet)
    FO_DRV_FN(cuDeviceGetDevResource)
    FO_DRV_FN(cuDevSmResourceSplitByCount)
    FO_DRV_FN(cuDevResourceGenerateDesc)
    FO_DRV_FN(cuGreenCtxCreate)
    FO_DRV_FN(cuGreenCtxStreamCreate)
};
#undef FO_DRV_FN

struct Split {
    std::vector<CUdevResource> res;           // one SM resource per group
    std::vector<CUgreenCtx> green;            // created at the group's first use
};

std::mutex g_mu;                              // guards everything below
Driver g_drv;
bool g_drv_loaded = false;
std::map<std::pair<int, int>, Split> g_splits;

template <class F>
int entry(const char* name, F* fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const cudaError_t e = cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q);
    FO_CHECK(e == cudaSuccess && q == cudaDriverEntryPointSuccess && p,
             "fo_create_on_sms: the CUDA driver has no green contexts (%s not found; driver 12.4 or later needed)", name);
    *fn = reinterpret_cast<F>(p);
    return 0;
}

int load_driver() {
    if (g_drv_loaded) return 0;
    FO_TRY(entry("cuDeviceGet", &g_drv.p_cuDeviceGet));
    FO_TRY(entry("cuDeviceGetDevResource", &g_drv.p_cuDeviceGetDevResource));
    FO_TRY(entry("cuDevSmResourceSplitByCount", &g_drv.p_cuDevSmResourceSplitByCount));
    FO_TRY(entry("cuDevResourceGenerateDesc", &g_drv.p_cuDevResourceGenerateDesc));
    FO_TRY(entry("cuGreenCtxCreate", &g_drv.p_cuGreenCtxCreate));
    FO_TRY(entry("cuGreenCtxStreamCreate", &g_drv.p_cuGreenCtxStreamCreate));
    g_drv_loaded = true;
    return 0;
}

__global__ void sm_ids_kernel(int32_t* out, int n) {
    unsigned s;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(s));
    // ~20 us of residency per CTA, so that the CTAs of one launch spread over every SM the stream can reach
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    do { asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); } while (t - t0 < 20000ull);
    if (threadIdx.x == 0 && (int)blockIdx.x < n) out[blockIdx.x] = (int32_t)s;
}

}  // namespace

int sm_group_acquire(int device, int split, int group, void** green, int* sms) {
    std::lock_guard<std::mutex> lk(g_mu);
    FO_TRY(load_driver());
    CUdevice dev;
    FO_CHECK(g_drv.p_cuDeviceGet(&dev, device) == CUDA_SUCCESS, "fo_create_on_sms: cuDeviceGet(%d) failed", device);
    const auto key = std::make_pair(device, split);
    if (!g_splits.count(key)) {
        CUdevResource all;
        memset(&all, 0, sizeof(all));
        CUresult r = g_drv.p_cuDeviceGetDevResource(dev, &all, CU_DEV_RESOURCE_TYPE_SM);
        FO_CHECK(r == CUDA_SUCCESS, "fo_create_on_sms: cuDeviceGetDevResource failed (%d)", (int)r);
        // equal groups at the architecture's granularity: at least 8 SMs, a multiple of 8 (sm_90 and later)
        const int per = (int)all.sm.smCount / split / SM_GROUP_GRANULE * SM_GROUP_GRANULE;
        FO_CHECK(per >= SM_GROUP_GRANULE,
                 "fo_create_on_sms: %u SMs split %d ways gives groups below the %d-SM granularity of green contexts",
                 all.sm.smCount, split, SM_GROUP_GRANULE);
        Split made;
        made.res.resize(split);
        CUdevResource rem;
        memset(&rem, 0, sizeof(rem));
        unsigned nb = (unsigned)split;
        r = g_drv.p_cuDevSmResourceSplitByCount(made.res.data(), &nb, &all, &rem, 0, (unsigned)per);
        bool ok = r == CUDA_SUCCESS && nb == (unsigned)split;
        for (unsigned i = 0; ok && i < nb; ++i) ok = made.res[i].sm.smCount >= (unsigned)per;
        FO_CHECK(ok, "fo_create_on_sms: cuDevSmResourceSplitByCount could not make %d groups of %d SMs (%d, %u groups)", split, per,
                 (int)r, nb);
        made.green.assign(split, nullptr);
        g_splits[key] = made;
    }
    Split& sp = g_splits[key];
    if (!sp.green[group]) {
        CUdevResourceDesc desc;
        CUresult r = g_drv.p_cuDevResourceGenerateDesc(&desc, &sp.res[group], 1);
        FO_CHECK(r == CUDA_SUCCESS, "fo_create_on_sms: cuDevResourceGenerateDesc failed (%d)", (int)r);
        r = g_drv.p_cuGreenCtxCreate(&sp.green[group], desc, dev, CU_GREEN_CTX_DEFAULT_STREAM);
        if (r != CUDA_SUCCESS) sp.green[group] = nullptr;
        FO_CHECK(r == CUDA_SUCCESS, "fo_create_on_sms: cuGreenCtxCreate failed (%d)", (int)r);
    }
    *green = sp.green[group];
    *sms = (int)sp.res[group].sm.smCount;
    return 0;
}

int sm_group_stream(void* green, cudaStream_t* st) {
    CUstream s = nullptr;
    const CUresult r = g_drv.p_cuGreenCtxStreamCreate(&s, (CUgreenCtx)green, CU_STREAM_NON_BLOCKING, 0);
    FO_CHECK(r == CUDA_SUCCESS, "cuGreenCtxStreamCreate failed (%d)", (int)r);
    *st = (cudaStream_t)s;
    return 0;
}

int sm_ids(int32_t* out, int n, cudaStream_t st) {
    sm_ids_kernel<<<n, 32, 0, st>>>(out, n);
    FO_LAUNCHED();
    FO_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace fo
