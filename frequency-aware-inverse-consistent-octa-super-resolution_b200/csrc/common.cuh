// Shared device/host helpers for the b200wave kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdio>
#include "b200wave.h"

namespace b200w {

constexpr int kMaxTaps = B200W_MAX_TAPS;
constexpr int kThreads = 256;

// Filter taps travel by value in the kernel parameter block (constant bank): with the tap loops
// fully unrolled every FFMA takes its coefficient as a c[0x0][..] operand, no load instruction.
constexpr int kMaxTemplTaps = 16;   // tap counts the templated kernels are instantiated for
struct Taps {
    float w_lo[kMaxTaps];  // along W
    float w_hi[kMaxTaps];
    float h_lo[kMaxTaps];  // along H
    float h_hi[kMaxTaps];
    // the first kMaxTemplTaps H taps once more as (t, t) pairs: operands of the packed FFMA2 (fma.rn.f32x2), which
    // takes them straight from uniform registers
    float2 h_lo2[kMaxTemplTaps];
    float2 h_hi2[kMaxTemplTaps];
};

// Blackwell packed fp32 FMA: (a.x*b.x + c.x, a.y*b.y + c.y) in one issue slot (SASS FFMA2)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(d)
        : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)),
          "l"(*reinterpret_cast<unsigned long long*>(&c)));
    return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;"
        : "=l"(d)
        : "l"(*reinterpret_cast<unsigned long long*>(&a)), "l"(*reinterpret_cast<unsigned long long*>(&b)));
    return *reinterpret_cast<float2*>(&d);
}

// Extension index maps of mypad (pw/dwt/lowlevel.py:28-88) and of the periodization branch of
// afb1d (:134-150), folded into one function: returns the source index in [0,n) or -1 for "zero".
__host__ __device__ __forceinline__ int ext_index(int s, int n, int mode) {
    if ((unsigned)s < (unsigned)n) return s;
    switch (mode) {
        case B200W_MODE_SYMMETRIC: {  // half-sample symmetric, period 2n (utils.reflect(-0.5, n-0.5))
            int p = 2 * n;
            int m = s % p;
            if (m < 0) m += p;
            return m < n ? m : p - 1 - m;
        }
        case B200W_MODE_REFLECT: {  // whole-sample, period 2n-2 (F.pad reflect)
            if (n == 1) return 0;
            int p = 2 * n - 2;
            int m = s % p;
            if (m < 0) m += p;
            return m < n ? m : p - m;
        }
        case B200W_MODE_PERIODIC: {
            int m = s % n;
            if (m < 0) m += n;
            return m;
        }
        case B200W_MODE_PERIODIZATION: {  // odd n: last sample repeated once, then period n+1
            int p = n + (n & 1);
            int m = s % p;
            if (m < 0) m += p;
            return m < n ? m : n - 1;
        }
        default:
            return -1;  // zero
    }
}

// index of a coefficient for the synthesis bank: outside [0,m) is zero, except for periodization
// where the coefficient sequence is m-periodic (the wrap-add + roll of sfb1d, :252-261)
__device__ __forceinline__ int coef_index(int k, int m, bool periodic) {
    if ((unsigned)k < (unsigned)m) return k;
    if (!periodic) return -1;
    int r = k % m;
    if (r < 0) r += m;
    return r;
}

// Out-of-line variants for the stream kernels: the maps are only needed for the few rows / columns outside the
// image, and every inlined copy costs ~100 instructions (four integer divisions) of instruction-cache footprint.
static __device__ __noinline__ int ext_index_far(int s, int n, int mode) { return ext_index(s, n, mode); }
static __device__ __noinline__ int coef_index_far(int k, int m, int periodic) { return coef_index(k, m, periodic != 0); }

// ---- B200W_BOUNDS debug build (python -m b200wave._build --bounds; tests/test_gpu_parity.py::test_bounds_build) --------
// compute-sanitizer is closed on this pool, so the library carries its own memcheck: with -DB200W_BOUNDS every shared-memory
// access that goes through the wrappers below / in the kernels, every staged copy and every global store of the DWT
// kernels is checked -- shared addresses against the CTA's shared-memory size, global addresses against the list of
// buffers the launch was given (registered by the launcher) -- and a violation traps, which fails the launch.
#ifdef B200W_BOUNDS
struct BRange { const char* lo; const char* hi; };
constexpr int kMaxBRanges = 48;
static __device__ BRange g_bounds[kMaxBRanges];
static __device__ int g_nbounds;
static __device__ __noinline__ void bounds_fail(int what, unsigned long long a, unsigned bytes, unsigned limit, int line) {
    printf("b200wave B200W_BOUNDS: %s access of %u bytes at %llx out of bounds (limit %u) at line %d (block %d thread %d of %d)\n",
           what ? "global" : "shared", bytes, a, limit, line, (int)blockIdx.x, (int)threadIdx.x, (int)blockDim.x);
    __trap();
}
static __device__ __forceinline__ void bchk_shared(unsigned addr, unsigned bytes, int line, unsigned align = 0u) {
    // the CTA's window: [start of the shared window's user part, end of the dynamic allocation).  Every extern
    // __shared__ array starts at the same address (after the system-reserved 1 KB and any static variables).
    extern __shared__ __align__(16) unsigned char b200w_dyn_smem_base[];
    unsigned dyn;
    asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
    const unsigned tot = (unsigned)__cvta_generic_to_shared(b200w_dyn_smem_base) + dyn;
    const unsigned al = align ? align : (bytes >= 16 ? 16u : bytes);   // natural alignment unless stated
    if (addr > tot || bytes > tot - addr || (addr & (al - 1u))) bounds_fail(0, addr, bytes, tot, line);
}
static __device__ __forceinline__ void bchk(const void* p, unsigned bytes, int line, unsigned align = 0u) {
    // The address-space test is made on the FINAL address through opaque asm: the owner kernels form generic pointers to
    // shared-memory images as `image - first_row * pitch` (possibly below the shared window) and add the row back, and
    // the compiler is free to test `__isShared` on such a base instead of on the sum.
    const unsigned long long ga = reinterpret_cast<unsigned long long>(p);
    unsigned is_sh, sa;
    asm volatile("{\n.reg .pred q;\n.reg .u64 t;\nisspacep.shared q, %2;\nselp.u32 %0, 1, 0, q;\ncvta.to.shared.u64 t, %2;\n"
                 "cvt.u32.u64 %1, t;\n}" : "=r"(is_sh), "=r"(sa) : "l"(ga));
    if (is_sh) {
        bchk_shared(sa, bytes, line, align);
        return;
    }
    const char* c = reinterpret_cast<const char*>(p);
    const int n = g_nbounds;
    for (int i = 0; i < n; ++i)
        if (c >= g_bounds[i].lo && c + bytes <= g_bounds[i].hi) return;
    bounds_fail(1, (unsigned long long)c, bytes, 0u, line);
}
#define B200W_CHK(p, bytes) bchk((p), (unsigned)(bytes), __LINE__)
#define B200W_CHK_S(addr, bytes) bchk_shared((addr), (unsigned)(bytes), __LINE__)
#define B200W_CHK_A(p, bytes, align) bchk((p), (unsigned)(bytes), __LINE__, (unsigned)(align))
// host side: the buffers a launch may touch (called by the launcher of the same translation unit: the table is per TU)
struct BoundsList {
    BRange r[kMaxBRanges];
    int n = 0;
    void add(const void* p, size_t bytes) {
        if (p && bytes && n < kMaxBRanges) { r[n].lo = (const char*)p; r[n].hi = (const char*)p + bytes; ++n; }
    }
};
static inline void bounds_set(const BoundsList& b, cudaStream_t st) {
    cudaMemcpyToSymbolAsync(g_bounds, b.r, sizeof(BRange) * kMaxBRanges, 0, cudaMemcpyHostToDevice, st);
    cudaMemcpyToSymbolAsync(g_nbounds, &b.n, sizeof(int), 0, cudaMemcpyHostToDevice, st);
}
#else
#define B200W_CHK(p, bytes) ((void)0)
#define B200W_CHK_S(addr, bytes) ((void)0)
#define B200W_CHK_A(p, bytes, align) ((void)0)
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// cp.async (LDGSTS): global -> shared without register staging.  `dst` is a 32-bit shared-window address.
template <int V>
__device__ __forceinline__ void cp_async(unsigned dst, const float* src) {
    B200W_CHK_S(dst, 4 * V);
    B200W_CHK(src, 4 * V);
    if (V == 4) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
    else if (V == 2) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
// src-size 0: nothing is read, the destination is zero-filled (`src` only has to be a valid address)
template <int V>
__device__ __forceinline__ void cp_async_zero(unsigned dst, const float* src) {
    B200W_CHK_S(dst, 4 * V);
    const int z = 0;
    if (V == 4) asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(z) : "memory");
    else if (V == 2) asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(z) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(z) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Programmatic dependent launch: a kernel launched with launch_pdl() may start while its predecessor in the stream
// is still running; it must call pdl_wait() before it touches global memory (reads of the predecessor's results, and
// writes -- the allocator may have handed it memory the predecessor still reads).  pdl_trigger() in the predecessor
// lets the dependent grid be scheduled as soon as every CTA has issued it (or exited).  Both are no-ops for plain launches.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;"); }

template <typename Kernel, typename Params>
inline cudaError_t launch_pdl(Kernel kernel, unsigned grid, unsigned block, size_t smem, cudaStream_t st, const Params& prm) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, prm);
}

int set_last_cuda_error(cudaError_t e);
// diagnostics: counts the launch and remembers the kernel's name (b200w_kernel_launches / b200w_kernel_log)
void note_launch(const char* kernel);

}  // namespace b200w
