// ABI bookkeeping: version, status names, last CUDA error (thread-local, diagnostics only); the DWT kernel-family
// switches.
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include "dwt_levels.cuh"
#include "tma.cuh"

namespace b200w {
constexpr int kLaunchLog = 64;
static thread_local int g_last_cuda_error = 0;
int set_last_cuda_error(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return B200W_ERR_LAUNCH;
}
const DwtPolicy& dwt_policy() {
    static const DwtPolicy pol = [] {
        auto flag = [](const char* name) { const char* e = getenv(name); return e && e[0] == '1'; };
        auto count = [](const char* name) { const char* e = getenv(name); return e ? std::max(1, atoi(e)) : 0; };
        const char* owner = getenv("B200W_OWNER");
        const char* tma = getenv("B200W_TMA");
        DwtPolicy p;
        p.force_direct = flag("B200W_FORCE_DIRECT");
        p.owner = (owner && owner[0] >= '0' && owner[0] <= '2') ? owner[0] - '0' : 1;
        p.tma = !(tma && tma[0] == '0');
        p.tma_noboxes = getenv("B200W_TMA_NOBOXES") != nullptr;
        p.tma_G = count("B200W_TMA_G");
        p.tma_D = count("B200W_TMA_D");
        return p;
    }();
    return pol;
}
EncodeTiledFn tma_encode_fn() {
    static std::atomic<void*> fn{nullptr};
    static std::atomic<int> state{0};   // 0 = not looked up, 1 = found, 2 = unavailable
    if (state.load(std::memory_order_acquire) == 0) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres = cudaDriverEntryPointSymbolNotFound;
        const cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
        if (e != cudaSuccess) (void)cudaGetLastError();
        const bool ok = e == cudaSuccess && qres == cudaDriverEntryPointSuccess && p != nullptr;
        fn.store(ok ? p : nullptr, std::memory_order_relaxed);
        state.store(ok ? 1 : 2, std::memory_order_release);
    }
    return reinterpret_cast<EncodeTiledFn>(fn.load(std::memory_order_relaxed));
}

bool tma_make_map_f32(CUtensorMap* map, const float* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box) {
    EncodeTiledFn enc = tma_encode_fn();
    if (!enc || rank < 1 || rank > 4) return false;
    cuuint64_t gdim[4], gstr[4];
    cuuint32_t bdim[4], estr[4];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bdim[i] = box[i];
        estr[i] = 1;
        if (box[i] < 1 || box[i] > 256 || dims[i] < 1) return false;
    }
    for (int i = 0; i + 1 < rank; ++i) {
        gstr[i] = strides_bytes[i];
        if ((gstr[i] & 15) != 0 || gstr[i] == 0) return false;
    }
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || ((size_t)box[0] * 4) % 16 != 0) return false;
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<float*>(base), gdim, gstr,
                           bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

static std::atomic<unsigned long long> g_launches{0};
static const char* g_log[kLaunchLog] = {nullptr};
void note_launch(const char* kernel) {
    const unsigned long long n = g_launches.fetch_add(1, std::memory_order_relaxed);
    g_log[n % kLaunchLog] = kernel;
}
}  // namespace b200w

extern "C" unsigned long long b200w_kernel_launches(void) { return b200w::g_launches.load(std::memory_order_relaxed); }

extern "C" const char* b200w_kernel_log(int back) {
    const unsigned long long n = b200w::g_launches.load(std::memory_order_relaxed);
    if (back < 0 || back >= b200w::kLaunchLog || (unsigned long long)back >= n) return "";
    const char* s = b200w::g_log[(n - 1 - (unsigned long long)back) % b200w::kLaunchLog];
    return s ? s : "";
}

#ifndef B200W_BUILD_HASH
#define B200W_BUILD_HASH "unknown"
#endif
extern "C" const char* b200w_build_hash(void) { return B200W_BUILD_HASH; }

extern "C" int b200w_abi_version(void) { return B200W_ABI_VERSION; }

extern "C" int b200w_last_cuda_error(void) { return b200w::g_last_cuda_error; }

extern "C" const char* b200w_status_string(int status) {
    switch (status) {
        case B200W_OK: return "ok";
        case B200W_ERR_BAD_MODE: return "Unkown pad type";
        case B200W_ERR_BAD_TAPS: return "bad filter taps (null, empty or more than B200W_MAX_TAPS)";
        case B200W_ERR_NULL_POINTER: return "null pointer";
        case B200W_ERR_BAD_SHAPE: return "bad shape";
        case B200W_ERR_REFLECT_PAD: return "reflect padding must be smaller than the padded dimension";
        case B200W_ERR_PER_TOO_SHORT: return "periodization needs a signal at least as long as the filter";
        case B200W_ERR_LAUNCH: return "CUDA launch failed";
        case B200W_ERR_WORKSPACE: return "workspace missing or too small";
        case B200W_ERR_BAD_WINDOW: return "SSIM window size must be odd and at most 11";
        default: return "unknown status";
    }
}
