// pe_partition.cu -- SM partitions of one device (CUDA green contexts) and grid sizing by the launching stream.
//
// A partition splits the SMs of a device into two disjoint sets with one stream on each.  Two kernels limited by different
// resources (the blob path by HBM and grid barriers, the sphere kernel by issue slots) then run side by side, each at its full
// per-SM occupancy; on shared SMs the block scheduler can only run them one after the other, because neither leaves room for a
// block of the other.  The driver is reached through cudaGetDriverEntryPointByVersion, so the library still links cudart only,
// and a driver without green contexts is reported as an error the caller can fall back from.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <mutex>
#include <utility>
#include <vector>
#include "pe_common.cuh"

namespace pe {
namespace {

struct Driver {
    PFN_cuDeviceGet_v2000 deviceGet = nullptr;
    PFN_cuDeviceGetDevResource_v12040 deviceGetDevResource = nullptr;
    PFN_cuDevSmResourceSplitByCount_v12040 smResourceSplitByCount = nullptr;
    PFN_cuDevResourceGenerateDesc_v12040 resourceGenerateDesc = nullptr;
    PFN_cuGreenCtxCreate_v12040 greenCtxCreate = nullptr;
    PFN_cuGreenCtxDestroy_v12040 greenCtxDestroy = nullptr;
    PFN_cuGreenCtxGetDevResource_v12040 greenCtxGetDevResource = nullptr;
    PFN_cuGreenCtxStreamCreate_v12050 greenCtxStreamCreate = nullptr;
    PFN_cuStreamGetGreenCtx_v12040 streamGetGreenCtx = nullptr;
    PFN_cuStreamSynchronize_v2000 streamSynchronize = nullptr;
    PFN_cuStreamDestroy_v4000 streamDestroy = nullptr;
    bool ok = false;
};

template <class F>
bool entry(const char *name, unsigned version, F &fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPointByVersion(name, &p, version, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !p) {
        cudaGetLastError();
        return false;
    }
    fn = reinterpret_cast<F>(p);
    return true;
}

// The driver's green-context entry points, resolved once; nullptr when the driver lacks any of them.
const Driver *driver() {
    static Driver d;
    static std::once_flag once;
    std::call_once(once, [] {
        d.ok = entry("cuDeviceGet", 2000, d.deviceGet) && entry("cuDeviceGetDevResource", 12040, d.deviceGetDevResource) &&
               entry("cuDevSmResourceSplitByCount", 12040, d.smResourceSplitByCount) &&
               entry("cuDevResourceGenerateDesc", 12040, d.resourceGenerateDesc) && entry("cuGreenCtxCreate", 12040, d.greenCtxCreate) &&
               entry("cuGreenCtxDestroy", 12040, d.greenCtxDestroy) && entry("cuGreenCtxGetDevResource", 12040, d.greenCtxGetDevResource) &&
               entry("cuGreenCtxStreamCreate", 12050, d.greenCtxStreamCreate) && entry("cuStreamGetGreenCtx", 12040, d.streamGetGreenCtx) &&
               entry("cuStreamSynchronize", 2000, d.streamSynchronize) && entry("cuStreamDestroy", 4000, d.streamDestroy);
    });
    return d.ok ? &d : nullptr;
}

struct Partition {
    CUgreenCtx ctx[2] = {nullptr, nullptr};  // [0] the blob SMs, [1] the rest
    CUstream stream[2] = {nullptr, nullptr};
};

std::mutex g_mutex;                                      // guards both tables
std::vector<Partition> g_partitions;                     // live partitions of this library
std::vector<std::pair<cudaStream_t, int>> g_stream_sms;  // SMs a launching stream can use, by stream handle

// Destroys what exists of p.  With report, the first failure is the library's error; the rest is released in any case.
int release(const Driver *d, Partition &p, bool report) {
    int rc = PE_OK;
    for (int i = 0; i < 2; ++i) {
        if (p.stream[i]) {
            const CUresult s = d->streamSynchronize(p.stream[i]);
            const CUresult r = d->streamDestroy(p.stream[i]);
            if (s != CUDA_SUCCESS || r != CUDA_SUCCESS) {
                if (report && rc == PE_OK) set_error("pe_sm_partition_destroy: stream %d: cuStreamSynchronize %d, cuStreamDestroy %d", i, (int)s, (int)r);
                rc = PE_ERR_CUDA;
            }
            p.stream[i] = nullptr;
        }
    }
    for (int i = 0; i < 2; ++i) {
        if (p.ctx[i]) {
            const CUresult r = d->greenCtxDestroy(p.ctx[i]);
            if (r != CUDA_SUCCESS) {
                if (report && rc == PE_OK) set_error("pe_sm_partition_destroy: cuGreenCtxDestroy failed (%d)", (int)r);
                rc = PE_ERR_CUDA;
            }
            p.ctx[i] = nullptr;
        }
    }
    return rc;
}

#define PE_DRV(call)                                                                   \
    do {                                                                               \
        const CUresult r__ = (call);                                                   \
        if (r__ != CUDA_SUCCESS) {                                                     \
            pe::set_error("pe_sm_partition_create: %s failed (CUresult %d)", #call, (int)r__); \
            return PE_ERR_CUDA;                                                        \
        }                                                                              \
    } while (0)

int create(const Driver *d, int device, int blob_sms, Partition &p, int sms[2]) {
    PE_CUDA(cudaInitDevice(device, 0, 0));  // green contexts retain the primary context: have it exist first
    CUdevice dev = 0;
    PE_DRV(d->deviceGet(&dev, device));
    CUdevResource all{};
    PE_DRV(d->deviceGetDevResource(dev, &all, CU_DEV_RESOURCE_TYPE_SM));
    PE_CHECK_ARG(blob_sms < (int)all.sm.smCount, "pe_sm_partition_create: blob_sms %d leaves none of the device's %u SMs", blob_sms,
                 all.sm.smCount);
    CUdevResource res[2] = {};
    unsigned groups = 1;
    PE_DRV(d->smResourceSplitByCount(&res[0], &groups, &all, &res[1], 0, (unsigned)blob_sms));
    // the driver rounds a count up to its granularity (8 SMs from compute capability 9.0 on); a different partition than the one
    // asked for is refused rather than silently used
    PE_CHECK_ARG(groups == 1 && (int)res[0].sm.smCount == blob_sms && res[1].sm.smCount > 0,
                 "pe_sm_partition_create: the driver splits %d SMs as %u group(s) of %u and %u left (device of %u SMs)", blob_sms, groups,
                 groups ? res[0].sm.smCount : 0u, res[1].sm.smCount, all.sm.smCount);
    for (int i = 0; i < 2; ++i) {
        CUdevResourceDesc desc = nullptr;
        PE_DRV(d->resourceGenerateDesc(&desc, &res[i], 1));
        PE_DRV(d->greenCtxCreate(&p.ctx[i], desc, dev, CU_GREEN_CTX_DEFAULT_STREAM));
        PE_DRV(d->greenCtxStreamCreate(&p.stream[i], p.ctx[i], CU_STREAM_NON_BLOCKING, 0));
        CUdevResource got{};
        PE_DRV(d->greenCtxGetDevResource(p.ctx[i], &got, CU_DEV_RESOURCE_TYPE_SM));
        sms[i] = (int)got.sm.smCount;
    }
    return PE_OK;
}

}  // namespace

int stream_sm_count(cudaStream_t st) {
    std::lock_guard<std::mutex> lock(g_mutex);
    for (const auto &e : g_stream_sms)
        if (e.first == st) return e.second;
    int n = sm_count();
    if (const Driver *d = driver()) {
        CUgreenCtx g = nullptr;
        CUdevResource r{};
        if (d->streamGetGreenCtx((CUstream)st, &g) == CUDA_SUCCESS && g &&
            d->greenCtxGetDevResource(g, &r, CU_DEV_RESOURCE_TYPE_SM) == CUDA_SUCCESS && r.sm.smCount > 0)
            n = (int)r.sm.smCount;
    }
    if (g_stream_sms.size() >= 64) g_stream_sms.clear();
    g_stream_sms.emplace_back(st, n);
    return n;
}

}  // namespace pe

extern "C" {

int pe_sm_partition_create(int32_t device, int32_t blob_sms, void **stream_blob, void **stream_rest, int32_t *sms_blob,
                           int32_t *sms_rest) {
    PE_CHECK_ARG(stream_blob && stream_rest && sms_blob && sms_rest, "pe_sm_partition_create: null pointer");
    *stream_blob = *stream_rest = nullptr;
    *sms_blob = *sms_rest = 0;
    PE_CHECK_ARG(blob_sms > 0, "pe_sm_partition_create: blob_sms must be positive (got %d)", blob_sms);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        pe::set_error("no CUDA device is visible");
        return PE_ERR_NO_DEVICE;
    }
    PE_CHECK_ARG(device >= 0 && device < ndev, "pe_sm_partition_create: device %d of %d", device, ndev);
    const pe::Driver *d = pe::driver();
    if (!d) {
        pe::set_error("pe_sm_partition_create: the CUDA driver has no green-context entry points");
        return PE_ERR_CUDA;
    }
    std::lock_guard<std::mutex> lock(pe::g_mutex);
    pe::Partition p;
    int sms[2] = {0, 0};
    const int rc = pe::create(d, device, blob_sms, p, sms);
    if (rc != PE_OK) {
        pe::release(d, p, false);  // the error stays that of the step that failed
        return rc;
    }
    pe::g_partitions.push_back(p);
    pe::g_stream_sms.clear();  // a handle seen before may now name one of these streams
    *stream_blob = (void *)p.stream[0];
    *stream_rest = (void *)p.stream[1];
    *sms_blob = sms[0];
    *sms_rest = sms[1];
    return PE_OK;
}

int pe_sm_partition_destroy(void *stream_blob, void *stream_rest) {
    std::lock_guard<std::mutex> lock(pe::g_mutex);
    for (size_t i = 0; i < pe::g_partitions.size(); ++i) {
        pe::Partition &p = pe::g_partitions[i];
        if ((void *)p.stream[0] == stream_blob && (void *)p.stream[1] == stream_rest) {
            const int rc = pe::release(pe::driver(), p, true);
            pe::g_partitions.erase(pe::g_partitions.begin() + i);
            pe::g_stream_sms.clear();
            return rc;
        }
    }
    pe::set_error("pe_sm_partition_destroy: the streams are not a live partition of this library");
    return PE_ERR_ARG;
}

}  // extern "C"
