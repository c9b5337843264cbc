// Level geometry and chain bookkeeping shared by the DWT chain kernels (stream, owner and TMA variants).
//
// A multi-level transform is ONE launch.  In the stream kernels the work items of all levels form one ordered list
// (all items of the first level, then the next level, ...).  An item of level j+1 of image plane p may start once
// every item of level j of that plane has been written: per-(level, plane) completion counters, published with a
// gpu-scope release (fence + atomic) and consumed with ld.acquire.  Work items are handed out in list order by an
// atomic ticket taken when a CTA starts, so an item only ever waits for items that are already running or done: no
// deadlock, no launch gaps between the small coarse levels, and the LL intermediates are consumed out of L2.
#pragma once
#include "common.cuh"

namespace b200w {

constexpr int kMaxLevels = B200W_MAX_LEVELS;
constexpr int kStreamNT = 128;   // threads per CTA of the stream kernels

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// count the item with release semantics: this CTA's global stores (ordered before by a barrier) are visible to
// whoever acquires the new counter value
__device__ __forceinline__ void signal_done(unsigned* counter) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(counter), "r"(1u) : "memory");
}

// ---- analysis ------------------------------------------------------------------------------------
struct AfbLevel {
    const float* x;
    float* low;
    float* highs;          // dense (planes,3,Ho,Wo)
    long long x_ps, x_rs;  // input plane / row stride (elements)
    long long low_ps, low_rs;  // LL output strides: dense for the last level, padded scratch for intermediates
    int H, W;              // logical input size (including the zero extension below)
    int Hreal, Wreal;      // rows / columns >= these read as zero (SFB2D.backward through the 'unpad' crop)
    int Ho, Wo;
    int offH, offW;
    int out_vec2;          // 64-bit stores into highs allowed
    int low_vec2;          // 64-bit stores into low allowed
    // store epilogue (FS_Discriminator.filter_wavelet, model.py:166-179): a sub-band whose pointer is null is not
    // written, and the three detail bands are stored as hi_scale * v + hi_shift (1, 0 = plain DWT)
    int st_low, st_hi;
    float hi_scale, hi_shift;
    // stream kernels: a thread owns one pair of output columns over R output rows.  Column pairs whose input
    // window lies inside the image ("interior", cp0A <= cp < cp0A + ncpA) are staged through the per-warp ring;
    // the few pairs at the left / right border go through the per-thread path with a column map.
    long long cta_base;    // index of this level's first CTA item
    int R, ncp, cpp;       // rows per segment, column pairs per row, CTA items per plane (= cppA + edge CTAs)
    int cp0A, ncpA, itemsA, cppA;   // interior class: first pair, pairs per row, thread items, CTA items per plane
    int RB, itemsB;        // border class: rows per (short) segment, thread items per plane
};

struct AfbParams {
    AfbLevel lv[kMaxLevels];
    long long total;       // work items over all levels
    unsigned* done;        // [J][planes] completed-item counters (null when J == 1)
    unsigned* ticket;      // stream kernels, J > 1: next work item
    int J, planes, mode;
    Taps t;
};

// "Owner" kernels (small planes, J > 1): one CTA owns a horizontal part of one plane for ALL levels.  The first level
// streams its input rows from global memory, the low-pass image of every level but the last stays in the CTA's
// shared memory, so the dependent levels cost a block barrier instead of a trip through L2 and a grid-wide
// dependency.  Parts of a plane overlap by the few rows the deeper levels need (recomputed, not shared).
constexpr int kMaxParts = 8;
constexpr int kOwnerNT = 384;   // threads of an owner CTA for filters up to 8 taps: 12 warps with up to 168 registers each (measured best of 256..512, profiles/r01_notes.md)
struct OwnerLevel {
    int R;                 // output rows per thread segment
    int pitch;             // row pitch (floats, multiple of 4) of this level's low-pass image in shared memory
    int buf_off;           // its offset (floats) inside the low-pass area
    int map_off;           // offset (ints) of this level's extension maps inside the map area
    int c0[kMaxParts], c1[kMaxParts];   // output rows a part computes
    int h0[kMaxParts], h1[kMaxParts];   // output rows a part stores to global memory (a partition of [0, Ho))
};
struct AfbOwnerParams {
    AfbParams p;
    OwnerLevel ol[kMaxLevels];
    int parts;
    int ring_floats;       // size of the staging rings that precede the maps and the low-pass area
    int map_ints;          // size of the extension-map area (all levels)
};

static_assert(sizeof(AfbOwnerParams) <= 4096, "kernel parameter block");

// ---- synthesis -----------------------------------------------------------------------------------
struct SfbLevel {
    const float* low;
    const float* highs;    // dense (planes,3,h,w); may be null (= zeros)
    float* y;
    long long low_ps, low_rs;
    long long y_ps, y_rs;  // output strides: dense for the last level, padded scratch for intermediates
    int h, w, out_h, out_w;
    int offH, offW;
    // stream kernels: a thread owns four adjacent output columns over Rp output row pairs.  Threads whose
    // coefficient window and outputs lie inside the arrays ("interior", tA0 <= t < tA0 + ntA) stage through the
    // per-warp ring; the few border output columns are evaluated one thread per output position.
    long long cta_base;
    int Rp, cpp;           // row pairs per segment, CTA items per plane (= cppA + border CTAs)
    int tA0, ntA, itemsA, cppA;   // interior class: first thread, threads per row, thread items / CTA items per plane
    int nA0, nA1, itemsB;  // border class: output columns [0,nA0) and [nA1,out_w); thread items per plane
    int n0_off;            // first output column of thread t: n0 = 4t + n0_off (0 or -1)
    int kb_off;            // first staged coefficient column of thread t: kb = 2t + kb_off
    int m_lo;              // first output row pair (A-space) of the level: offH >> 1
    int y_vec;             // widest aligned store (1, 2 or 4 floats)
    int vec2;              // coefficient rows are 8-byte aligned: stage with 64-bit copies
};

struct SfbParams {
    SfbLevel lv[kMaxLevels];  // chain order: coarsest level first
    long long total;
    unsigned* done;
    unsigned* ticket;
    int J, planes, periodic;
    Taps t;
};

struct SfbOwnerParams {
    SfbParams p;
    OwnerLevel ol[kMaxLevels];   // per chain position: c0/c1 = output rows a part computes (h0/h1 the same)
    int parts;
    int ring_floats;       // size of the staging rings that precede the output images
    int y_floats;          // size of the output images of all positions but the last
};

// launchers of the stream kernels (dwt_stream_afb.cu / dwt_stream_sfb.cu); the level geometry is complete
// except for the stream work decomposition, which they fill in.  `sms` = SM count of the current device.
bool afb_stream_supported(const AfbParams& p, int L);
int launch_afb_stream(AfbParams& p, int L, int sms, cudaStream_t st);
bool sfb_stream_supported(const SfbParams& p, int L);
int launch_sfb_stream(SfbParams& p, int L, int sms, cudaStream_t st);

// owner kernel (dwt_stream_afb.cu): all levels of an analysis chain in one launch without grid-wide dependencies.
// afb_owner_plan fills `op` and returns true when the shapes qualify (16-byte aligned rows, low-pass images fit in
// shared memory, enough planes x parts to occupy the device -- unless `force`).
bool afb_owner_plan(const AfbParams& p, int L, int sms, bool force, AfbOwnerParams& op);
int launch_afb_owner(const AfbOwnerParams& op, int L, cudaStream_t st);

// synthesis owner kernel (dwt_stream_sfb.cu): all positions of a synthesis chain in one launch, the intermediate
// outputs in shared memory
bool sfb_owner_plan(const SfbParams& p, int L, int sms, bool force, SfbOwnerParams& op);
int launch_sfb_owner(const SfbOwnerParams& op, int L, cudaStream_t st);

// clears the ticket + completion counters of a chain on the stream (a kernel rather than a memset node: inside a
// CUDA graph a kernel -> memset -> kernel sequence costs several microseconds of engine switching)
int zero_sync_words(unsigned* words, size_t n, cudaStream_t st);

// B200W_BOUNDS build: the global buffers a chain launch may touch (see common.cuh); no-ops otherwise
#ifdef B200W_BOUNDS
static inline void afb_register_bounds(const AfbParams& p, cudaStream_t st) {
    BoundsList b;
    for (int j = 0; j < p.J; ++j) {
        const AfbLevel& lv = p.lv[j];
        b.add(lv.x, sizeof(float) * (size_t)((long long)(p.planes - 1) * lv.x_ps + (long long)(lv.Hreal - 1) * lv.x_rs + lv.Wreal));
        if (lv.low) b.add(lv.low, sizeof(float) * (size_t)((long long)(p.planes - 1) * lv.low_ps + (long long)(lv.Ho - 1) * lv.low_rs + lv.Wo));
        if (lv.highs) b.add(lv.highs, sizeof(float) * (size_t)p.planes * 3 * lv.Ho * lv.Wo);
    }
    if (p.ticket) b.add(p.ticket, sizeof(unsigned) * ((size_t)p.J * p.planes + 1));
    bounds_set(b, st);
}
static inline void sfb_register_bounds(const SfbParams& p, cudaStream_t st) {
    BoundsList b;
    for (int c = 0; c < p.J; ++c) {
        const SfbLevel& lv = p.lv[c];
        b.add(lv.low, sizeof(float) * (size_t)((long long)(p.planes - 1) * lv.low_ps + (long long)(lv.h - 1) * lv.low_rs + lv.w));
        if (lv.highs) b.add(lv.highs, sizeof(float) * (size_t)p.planes * 3 * lv.h * lv.w);
        b.add(lv.y, sizeof(float) * (size_t)((long long)(p.planes - 1) * lv.y_ps + (long long)(lv.out_h - 1) * lv.y_rs + lv.out_w));
    }
    if (p.ticket) b.add(p.ticket, sizeof(unsigned) * ((size_t)p.J * p.planes + 1));
    bounds_set(b, st);
}
#else
static inline void afb_register_bounds(const AfbParams&, cudaStream_t) {}
static inline void sfb_register_bounds(const SfbParams&, cudaStream_t) {}
#endif

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline bool aligned_to(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

// Kernel-family selection from the environment, read once per process (api.cu).  The switches run independently
// written kernel families against each other on the same inputs; the defaults are what every other run takes.
struct DwtPolicy {
    bool force_direct;   // B200W_FORCE_DIRECT=1: one-thread-per-output kernels only
    int owner;           // B200W_OWNER: 0 = no owner kernels (ticketed chains), 1 = where they pay off, 2 = whenever they fit
    bool tma;            // B200W_TMA=0: cp.async owner kernels instead of the TMA-staged ones
    bool tma_noboxes;    // B200W_TMA_NOBOXES: TMA analysis ring fetches every extension row from its source row
    int tma_G, tma_D;    // B200W_TMA_G / B200W_TMA_D: row streams / ring stages of the TMA kernels (0 = the plan's choice)
};
const DwtPolicy& dwt_policy();

// the owner kernels run one CTA per SM: a short last wave wastes too much of the device
static inline bool short_last_wave(long long ctas, int sms) {
    const long long waves = (ctas + sms - 1) / sms;
    return ctas * 4 < waves * sms * 3 && waves > 1;
}

constexpr size_t kMaxDynSmem = 227 * 1024;   // dynamic shared memory of one CTA on sm_100a

// lets `Kernel` use up to kMaxDynSmem of dynamic shared memory; the attribute is per device (a process may drive
// several GPUs), so it is set once per device
template <auto Kernel>
static cudaError_t allow_max_dyn_smem() {
    static bool attr_set[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && attr_set[dev]) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem);
    if (e == cudaSuccess && dev >= 0 && dev < 64) attr_set[dev] = true;
    return e;
}

// X(L) for each tap count the templated kernels are instantiated for; X returns, other L fall through
#define B200W_FOR_EACH_L(X) \
    switch (L) {             \
        case 2: X(2);        \
        case 4: X(4);        \
        case 6: X(6);        \
        case 8: X(8);        \
        case 10: X(10);      \
        case 12: X(12);      \
        case 14: X(14);      \
        case 16: X(16);      \
        default: break;      \
    }

}  // namespace b200w
