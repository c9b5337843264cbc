// Multi-level analysis filter bank, TMA-staged owner kernel (the fast path for chains of small planes, e.g. the
// headline workload 64 x 304 x 304, db3, J = 3).
//
// Replaces the J-level loop of DWTForward.forward (pw/dwt/transform2d.py:66-74) around AFB2D.forward
// (pw/dwt/lowlevel.py:336-347: afb1d along W, afb1d along H, reshape, 2x .contiguous()), and -- with the synthesis
// taps as correlators -- the analysis passes of SFB2D.backward (pw/dwt/lowlevel.py:682-694).
//
// One CTA owns a horizontal part of one plane for all levels (rows a part needs from beyond its share are recomputed,
// not exchanged).  The first level is cut into G row streams (G <= MAXG, chosen by the plan); stream g owns a ring of D
// stages of SR = 2 PS input rows.  Warp roles while the first level streams in from global memory:
//   service warp g (warps NTC/32 ..): lane 0 waits for a free ring stage (`empty` mbarrier), arms the stage's `full`
//            mbarrier with the byte count and issues ONE cp.async.bulk.tensor.3d per stage (box = SR full-width rows of
//            the plane; rows and columns outside the tensor are zero-filled by the copy engine -- the 'zero' mode and
//            every image border for free).  Stages whose rows the padding mode maps elsewhere in a non-monotonic way
//            (wrapping modes) are fetched row by row from their source rows instead.  Once a stage has landed, all 32
//            lanes write the extension columns left and right of the image rows (copies inside shared memory through a
//            host-built table) and arrive on the stage's `ready` mbarrier.  'zero' mode needs no patches: the consumers
//            wait on the copy engine's barrier directly.  The first two stages of every stream are issued in the
//            prologue, before the tables are copied.
//   consumer warps 0 .. NTC/32-1: a lane owns one pair of adjacent output columns of one row stream and marches down
//            its rows: window loads one row pair ahead (register double buffer), row pass in registers (4L FMAs per
//            input row pair), column pass scattered into a ring of L/2 pending output rows held as float2 (packed
//            FFMA2), completed rows stored with 64-bit stores -- the three detail bands to global memory, the low-pass
//            row into the CTA's shared-memory image (with its extension halo) -- then an arrive on `empty`.
// Every lane reads its window with 128-bit shared loads at a host-precomputed per-pair offset from the stage base: no
// border class, no per-lane address arithmetic for the copies, no index maps in the loop.  All row / offset / patch
// tables are built by the host and travel in the parameter block; the prologue copies the part's share into shared
// memory with coalesced generic loads.
// The later levels read their input rows from the low-pass image of the level before (rows through a table of row
// addresses, so the row extension costs nothing; extension columns written once per level by all threads).
#include <algorithm>
#include <type_traits>
#include "dwt_tma.cuh"

namespace b200w {

// left extension of the analysis bank (= mypad's pad / 2, or the periodization roll)
constexpr int afbt_off(int L, bool per) { return per ? L - 1 - L / 2 : L - 2; }

// L taps, OFF = left extension: the first float of a lane's window is image column 4*cp - (OFF + S), S pads the
// window start down to a multiple of 4 floats
template <int L, int OFF>
struct AfbT {
    static constexpr int S = (4 - OFF % 4) % 4;
    static constexpr int H2 = L / 2;
    static constexpr int NV = (S + L + 2 + 3) / 4;   // float4 per window (two adjacent output columns)
    static constexpr int NE = 4 * NV;
    static constexpr bool kRotate = L >= 10;         // accumulator ring shifted instead of statically renamed
    // input row pairs per ring stage (a multiple of L/2): long stages, because every stage costs its service warp a
    // fixed ~1 us of issue + patch work on a sub-partition that is busy with consumer warps
    static constexpr int PS = kRotate ? 4 : (H2 == 1 ? 4 : (H2 == 4 ? 8 : 6));   // 2 * PS >= 2 * (L - 2): mirrored rows lie in the same stage
    static constexpr int SR = 2 * PS;                // rows per stage
    // consumer threads.  db2 / db3: the cost model of the plan picks 3 row streams at the headline shapes (two busy warps
    // per SM sub-partition), so 256 consumer threads suffice -- and a CTA of 352 threads may use up to 184 registers
    // per thread, which the software-pipelined window loads of the level-0 loop need (measured: 18.6 -> 17.3 us at cfg2)
    static constexpr int NTC = L == 2 ? 416 : (L <= 6 ? 256 : (L <= 8 ? 352 : 256));
    static constexpr int MAXG = L == 2 ? 5 : (L <= 6 ? 3 : (L <= 8 ? 5 : 4));   // row streams of the first level = service warps
    static constexpr int NT = NTC + 32 * MAXG;
    // short filters keep their taps in registers: inside the (divergent) consumer branch the compiler cannot use
    // uniform-register / constant-bank operands and would otherwise re-load every tap for every row pair
    static constexpr bool kRegTaps = L <= 8;
    static constexpr bool kPrefetch = L <= 6;        // software-pipelined window loads in the level-0 loop
};

// the taps of one kernel as a register-resident copy (same member names as TapsT)
template <int L>
struct RegTaps {
    float w_lo[L], w_hi[L];
    float2 h_lo2[L], h_hi2[L];
    // `zero` = 0.f read from shared memory: adding it makes the values opaque to ptxas, which would otherwise
    // rematerialise the constant loads inside the loop instead of keeping the registers
    __device__ __forceinline__ RegTaps(const TapsT& t, float zero) {
#pragma unroll
        for (int i = 0; i < L; ++i) {
            w_lo[i] = t.w_lo[i] + zero; w_hi[i] = t.w_hi[i] + zero;
            h_lo2[i].x = h_lo2[i].y = t.h_lo2[i].x + zero;
            h_hi2[i].x = h_hi2[i].y = t.h_hi2[i].x + zero;
        }
    }
};

__device__ __forceinline__ float4 lds128t(unsigned addr) {
    B200W_CHK_S(addr, 16);
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds32t(unsigned addr) {
    B200W_CHK_S(addr, 4);
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts32t(unsigned addr, float v) {
    B200W_CHK_S(addr, 4);
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void sts64t(unsigned addr, float2 v) {
    B200W_CHK_S(addr, 8);
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(v.x), "f"(v.y) : "memory");
}

// source index of extended position s: inside [0, real) itself, else the padding mode's map; -1 = zero.
// One reflection / one wrap (every extension shorter than the signal) is resolved inline; the general map with its
// integer divisions is an out-of-line call.
__device__ __forceinline__ int afbt_map(int s, int n, int real, int mode) {
    if ((unsigned)s < (unsigned)real) return s;
    if ((unsigned)s < (unsigned)n) return -1;          // inside the logical size but beyond the data: zero extension
    if (mode == B200W_MODE_ZERO) return -1;
    int m;
    if (mode == B200W_MODE_SYMMETRIC) {
        m = s < 0 ? -1 - s : 2 * n - 1 - s;
    } else if (mode == B200W_MODE_REFLECT) {
        m = s < 0 ? -s : 2 * n - 2 - s;
    } else if (mode == B200W_MODE_PERIODIC) {
        m = s < 0 ? s + n : s - n;
    } else {                                           // periodization: odd n repeats its last sample, then wraps
        const int pp = n + (n & 1);
        m = s < 0 ? s + pp : s - pp;
        if ((unsigned)m < (unsigned)pp) m = min(m, n - 1);
    }
    if ((unsigned)m >= (unsigned)n) m = ext_index_far(s, n, mode);
    return (m < 0 || m >= real) ? -1 : m;
}

// the windows of one pair of input rows (shared addresses a0 / a1) into registers
template <int L, int OFF>
__device__ __forceinline__ void afbt_load(float (&v)[2][AfbT<L, OFF>::NE], unsigned a0, unsigned a1) {
    constexpr int NV = AfbT<L, OFF>::NV;
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            const float4 q = lds128t((e ? a1 : a0) + 16u * k);
            v[e][4 * k] = q.x; v[e][4 * k + 1] = q.y; v[e][4 * k + 2] = q.z; v[e][4 * k + 3] = q.w;
        }
}

// one pair of input rows: row pass for both, then scatter into the accumulator ring (ph = pair index mod L/2; with
// kRotate slot 0 is the oldest and the caller shifts after the store)
template <int L, int OFF, class T>
__device__ __forceinline__ void afbt_pair(const T& t, const float (&v)[2][AfbT<L, OFF>::NE], float2 (&acc)[L / 2][4], int ph) {
    using C = AfbT<L, OFF>;
    constexpr int H2 = C::H2, S = C::S;
    float2 rl[2], rh[2];   // [row of the pair] = (column 0, column 1)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        float lo0 = 0.f, lo1 = 0.f, hi0 = 0.f, hi1 = 0.f;
#pragma unroll
        for (int j = 0; j < L; ++j) {
            lo0 = fmaf(t.w_lo[j], v[e][S + j], lo0);
            hi0 = fmaf(t.w_hi[j], v[e][S + j], hi0);
            lo1 = fmaf(t.w_lo[j], v[e][S + j + 2], lo1);
            hi1 = fmaf(t.w_hi[j], v[e][S + j + 2], hi1);
        }
        rl[e] = make_float2(lo0, lo1);
        rh[e] = make_float2(hi0, hi1);
    }
    // this pair carries taps (2u, 2u+1) of output row q - u
#pragma unroll
    for (int u = 0; u < H2; ++u) {
        const int sl = C::kRotate ? H2 - 1 - u : (ph - u + H2) % H2;
        const float2 a = t.h_lo2[2 * u], b = t.h_hi2[2 * u];
        const float2 c = t.h_lo2[2 * u + 1], d = t.h_hi2[2 * u + 1];
        float2* s = acc[sl];
        if (u == 0) {   // first contribution: start the accumulators
            s[0] = fmul2(a, rl[0]);   // LL: W-lo, H-lo
            s[1] = fmul2(b, rl[0]);   // LH: W-lo, H-hi
            s[2] = fmul2(a, rh[0]);   // HL: W-hi, H-lo
            s[3] = fmul2(b, rh[0]);   // HH
        } else {
            s[0] = ffma2(a, rl[0], s[0]);
            s[1] = ffma2(b, rl[0], s[1]);
            s[2] = ffma2(a, rh[0], s[2]);
            s[3] = ffma2(b, rh[0], s[3]);
        }
        s[0] = ffma2(c, rl[1], s[0]);
        s[1] = ffma2(d, rl[1], s[1]);
        s[2] = ffma2(c, rh[1], s[2]);
        s[3] = ffma2(d, rh[1], s[3]);
    }
}

struct ConstTaps {   // long filters: the taps stay in the constant bank
    const TapsT& t;
    const float (&w_lo)[kMaxTemplTaps], (&w_hi)[kMaxTemplTaps];
    const float2 (&h_lo2)[kMaxTemplTaps], (&h_hi2)[kMaxTemplTaps];
    __device__ __forceinline__ ConstTaps(const TapsT& tt, float) : t(tt), w_lo(tt.w_lo), w_hi(tt.w_hi), h_lo2(tt.h_lo2), h_hi2(tt.h_hi2) {}
};

// where a lane's completed output rows go
struct AfbtOut {
    unsigned ll_s;         // shared address of the low-pass pair in the next level's input image (row of `orow`)
    unsigned ll_pitch_b;   // its row pitch in bytes
    float* low;            // last level: global address of the low-pass pair (row of `orow`)
    float* hi;             // global address of the LH pair (row of `orow`); HL / HH follow at +band, +2*band
    size_t band;
    int Wo;
    int orow;              // output row the next completed accumulator slot belongs to
    int i0, nout;          // rows of the segment
    int hlo, hn;           // rows [hlo, hlo + hn) are stored to global memory
    bool vec2, low_vec2, c1ok;
};

template <int L, int OFF, bool LAST>
__device__ __forceinline__ void afbt_store(const float2* s, AfbtOut& o) {
    if ((unsigned)(o.orow - o.i0) < (unsigned)o.nout) {
        const bool g = (unsigned)(o.orow - o.hlo) < (unsigned)o.hn;
        if (!LAST) {
            sts64t(o.ll_s, s[0]);
        } else if (g) {
            B200W_CHK(o.low, o.c1ok ? 8 : 4);
            if (o.low_vec2) {
                *reinterpret_cast<float2*>(o.low) = s[0];
            } else {
                o.low[0] = s[0].x;
                if (o.c1ok) o.low[1] = s[0].y;
            }
        }
        if (g) {
            B200W_CHK(o.hi, o.c1ok ? 8 : 4); B200W_CHK(o.hi + o.band, o.c1ok ? 8 : 4); B200W_CHK(o.hi + 2 * o.band, o.c1ok ? 8 : 4);
            if (o.vec2) {
                *reinterpret_cast<float2*>(o.hi) = s[1];
                *reinterpret_cast<float2*>(o.hi + o.band) = s[2];
                *reinterpret_cast<float2*>(o.hi + 2 * o.band) = s[3];
            } else {
                o.hi[0] = s[1].x; o.hi[o.band] = s[2].x; o.hi[2 * o.band] = s[3].x;
                if (o.c1ok) { o.hi[1] = s[1].y; o.hi[o.band + 1] = s[2].y; o.hi[2 * o.band + 1] = s[3].y; }
            }
        }
    }
    o.ll_s += o.ll_pitch_b;
    if (LAST) o.low += o.Wo;
    o.hi += o.Wo;
    ++o.orow;
}

template <int L, int OFF>
__device__ __forceinline__ void afbt_rotate(float2 (&acc)[L / 2][4]) {
    if (AfbT<L, OFF>::kRotate) {
#pragma unroll
        for (int k = 0; k + 1 < L / 2; ++k)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[k][i] = acc[k + 1][i];
    }
}

template <int L, int OFF, int NTAB>
__global__ void __launch_bounds__(AfbT<L, OFF>::NT, 1) afb_tma_kernel(const __grid_constant__ AfbTmaParamsN<NTAB> p) {
    using C = AfbT<L, OFF>;
    constexpr int H2 = C::H2, NE = C::NE, PS = C::PS, SR = C::SR, NT = C::NT, NTC = C::NTC, S = C::S;
    constexpr bool kRotate = C::kRotate;
    extern __shared__ __align__(128) unsigned char smem[];
    const unsigned sbase = smem_u32(smem);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int plane = blockIdx.x / p.parts;
    const int part = blockIdx.x - plane * p.parts;
    const int mode = p.mode;
    constexpr int off = OFF;
    constexpr int hl = OFF + S;                  // columns left of the image in every staged / stored row
    pdl_trigger();   // the next kernel in the stream may be scheduled as SMs free up (it waits before touching memory)
    // every 64-byte line of the parameter block is touched by a different thread first: the constant-cache misses of a
    // freshly scheduled CTA then overlap instead of queueing up behind each other in the set-up code below
    if (tid < (int)(sizeof(AfbTmaHead) / 64)) {
        const int v = reinterpret_cast<const int*>(&p)[tid * 16];
        asm volatile("" ::"r"(v));
    }

    int* const tabs = reinterpret_cast<int*>(smem + p.tab_off);
    const AfbTmaLevel& l0 = p.lv[0];
    const int D = p.D, nstrips = p.nstrips, cps = p.cps, BW = p.BW;
    const unsigned srbw4 = (unsigned)(SR * BW * 4);          // bytes of one tile
    const unsigned stage_b = srbw4 * (unsigned)nstrips;      // bytes of one stage
    const int G = l0.nseg;
    const unsigned bar_full = sbase + p.bar_off, bar_ready = bar_full + 8u * G * D, bar_empty = bar_ready + 8u * G * D;

    // ---- set-up, part 1: barriers; then the first two stages of every row stream go out BEFORE the tables are copied
    //      (a regular box needs nothing but the parameter block), so the ~1 us of DRAM latency of the first tiles runs
    //      under the rest of the set-up instead of in front of the consumers ----
    constexpr int kProducerWarp = NTC / 32;   // the consumers are warps 0 .. NTC/32 - 1, then one service warp per stream
    const int c0_0 = l0.c0[part], c1_0 = l0.c1[part];
    const int nseg0 = (c1_0 - c0_0 + l0.R - 1) / l0.R;      // row streams of this part (<= G)
    if (tid < G * D) {
        mbar_init(bar_full + 8u * tid, 1);
        mbar_init(bar_ready + 8u * tid, 32);
        mbar_init(bar_empty + 8u * tid, (unsigned)l0.ncp);
        mbar_fence_init();
    }
    if (tid == 0) {
        tma_prefetch_map(&p.map_full);
        tma_prefetch_map(&p.map_row);
    }
    __syncthreads();
    const int early = p.boxes ? 2 : 0;   // stages issued here (0: the service warps issue them all)
    if (early && warp >= kProducerWarp && lane == 0 && warp - kProducerWarp < nseg0) {
        const int g = warp - kProducerWarp;
        const int i0 = c0_0 + g * l0.R;
        const int nst = (min(l0.R, c1_0 - i0) + H2 - 1 + PS - 1) / PS;
        pdl_wait();      // the tiles read the input tensor (maybe the previous kernel's output)
        for (int k = 0; k < min(early, nst); ++k) {
            const unsigned full = bar_full + 8u * (g * D + k);
            const unsigned dst = sbase + p.ring_off + (unsigned)(g * D + k) * stage_b;
            mbar_expect_tx(full, stage_b);
            B200W_CHK_S(dst, 16);
            B200W_CHK_S(dst + stage_b - 16, 16);
            for (int t = 0; t < nstrips; ++t)
                tma_load_3d(dst + (unsigned)t * srbw4, &p.map_full, full, 4 * t * cps - hl, 2 * i0 - off + k * SR, plane);
        }
    }

    // ---- set-up, part 2: this part's row / patch tables (built by the host, in the parameter block), the zero row ----
    {
        // The tables sit in the parameter block.  Indexing them per lane compiles to LDC with a lane-dependent offset,
        // which the constant cache serialises address by address (32 passes per instruction: 1.3 us of set-up).  The
        // address of a __grid_constant__ parameter is an ordinary generic address, so it is made opaque and read with
        // coalesced loads through L1 / L2 instead.
        const int* src = p.tab + part * p.tab_ints;
        asm volatile("" : "+l"(src));
        for (int i = tid; i < p.tab_ints; i += NT) tabs[i] = src[i];
    }
    const int nfix0 = mode != B200W_MODE_ZERO ? p.fix0_n : 0;
    for (int i = tid; i < p.zrow_floats; i += NT) reinterpret_cast<float*>(smem + p.zrow_off)[i] = 0.f;
    pdl_wait();      // everything above used only the parameter block; from here on global memory is touched
    __syncthreads();

    const bool use_ready = mode != B200W_MODE_ZERO && nfix0 > 0;
    const int* const rt0 = tabs + l0.rtab_off;
    const int nrt0 = 2 * (c1_0 - c0_0) + L;

    // ================================ level 0: streamed through the ring ================================
    if (warp >= kProducerWarp) {
        // ---- service warp of row stream g (all its lanes wait on the same barriers, so the hardware can put the warp
        // to sleep and wake it when the barrier completes).  Lane 0 issues the tiles of a stage into a free ring slot;
        // all lanes write the extension columns of a landed stage and release it to the consumers.  The patches run
        // one stage ahead of the consumers, the copies D stages ahead. ----
        const int g = warp - kProducerWarp;
        if (g < nseg0) {
            const int i0 = c0_0 + g * l0.R;
            const int npairs = min(l0.R, c1_0 - i0) + H2 - 1;
            const int nst = (npairs + PS - 1) / PS;
            const int e0 = 2 * (i0 - c0_0);
            const int r_start = 2 * i0 - off;                            // first (virtual) input row of the stream
            const unsigned ring = sbase + p.ring_off + (unsigned)(g * D) * stage_b;
            const int* const cf = tabs + p.fix0_off;
            const int npatch = SR * nfix0;
            // p.boxes: every stage is ONE box of consecutive (virtual) rows; rows above / below the image arrive
            // zero-filled, and where the padding mode maps them onto image rows (symmetric, reflect) the consumers'
            // row table points at those rows instead.  Otherwise (wrapping modes) such stages are fetched row by row
            // from their source rows.
            const bool boxes = p.boxes != 0;
            auto issue = [&](int k) {
                const int st = k % D;
                const unsigned full = bar_full + 8u * (g * D + st);
                const unsigned dst = ring + (unsigned)st * stage_b;
                if (boxes) {   // rows outside the tensor are zero-filled by the copy engine
                    mbar_expect_tx(full, stage_b);
                    B200W_CHK_S(dst, 16);
                    B200W_CHK_S(dst + stage_b - 16, 16);
                    for (int t = 0; t < nstrips; ++t)
                        tma_load_3d(dst + (unsigned)t * srbw4, &p.map_full, full, 4 * t * cps - hl, r_start + k * SR, plane);
                    return;
                }
                const int eb = e0 + k * SR;
                const int need = min(SR, 2 * npairs - k * SR);          // rows of this stage somebody reads
                int rfirst = rt0[eb];
                bool regular = rfirst >= 0;
                for (int i = 1; i < need; ++i) regular = regular && rt0[eb + i] == rfirst + i;
                if (regular) {
                    mbar_expect_tx(full, stage_b);
                    for (int t = 0; t < nstrips; ++t)
                        tma_load_3d(dst + (unsigned)t * srbw4, &p.map_full, full, 4 * t * cps - hl, rfirst, plane);
                } else {
                    mbar_expect_tx(full, (unsigned)(need * nstrips * BW * 4));
                    for (int i = 0; i < need; ++i) {
                        const int e = eb + i;
                        const int r = e < nrt0 ? rt0[e] : -1;            // -1: a row outside the tensor (zeros)
                        for (int t = 0; t < nstrips; ++t)
                            tma_load_3d(dst + (unsigned)t * srbw4 + (unsigned)(i * BW * 4), &p.map_row, full,
                                        4 * t * cps - hl, r, plane);
                    }
                }
            };
            auto patch = [&](int k) {
                const int st = k % D;
                mbar_wait(bar_full + 8u * (g * D + st), (unsigned)((k / D) & 1));
                const unsigned base = ring + (unsigned)st * stage_b;
#pragma unroll 2
                for (int it = lane; it < npatch; it += 32) {
                    B200W_CHK(cf + 2 * it, 8);
                    const int2 ds = *reinterpret_cast<const int2*>(cf + 2 * it);
                    if (ds.y >= 0) sts32t(base + (unsigned)ds.x, lds32t(base + (unsigned)ds.y));
                }
                mbar_arrive(bar_ready + 8u * (g * D + st));
            };
            // the first two stages go out first, so that the consumers can start while the rest of the ring is filled
            if (lane == 0)
                for (int k = early; k < min(2, nst); ++k) issue(k);
            __syncwarp();
            if (use_ready) patch(0);
            if (lane == 0)
                for (int k = 2; k < min(D, nst); ++k) issue(k);
            __syncwarp();
#pragma unroll 1
            for (int k = 0; k < nst; ++k) {
                if (use_ready && k + 1 < nst) patch(k + 1);
                if (k + D < nst) {
                    mbar_wait(bar_empty + 8u * (g * D + k % D), (unsigned)((k / D) & 1));
                    if (lane == 0) issue(k + D);
                    __syncwarp();
                }
            }
        }
    } else {
        // ---- consumers: lane = (row stream g, column pair cp) ----
        const int ct = tid;
        const int g = ct / l0.ncp;
        const int cp = ct - g * l0.ncp;
        if (g < nseg0) {
            const int i0 = c0_0 + g * l0.R;
            const int nout = min(l0.R, c1_0 - i0);
            const int npairs = nout + H2 - 1;
            const int nst = (npairs + PS - 1) / PS;
            const int s = cp / cps, cl = cp - s * cps;
            // rows come through a per-pair table of shared-memory row addresses (built by the host): a row above /
            // below the image that the padding mode maps onto an image row is simply read from that row's ring slot
            const unsigned lane_ring = sbase + (unsigned)s * srbw4 + (unsigned)cl * 16u;
            const int2* const rp = reinterpret_cast<const int2*>(tabs + p.rp0_off) + g * p.rp0_stride;
            const unsigned bar_wait = (use_ready ? bar_ready : bar_full) + 8u * (g * D);
            const unsigned bar_rel = bar_empty + 8u * (g * D);
            const AfbTmaLevel& l1 = p.lv[1];
            AfbtOut o;
            o.orow = i0 - (H2 - 1);
            o.i0 = i0; o.nout = nout;
            o.hlo = max(i0, l0.h0[part]);
            o.hn = max(0, min(i0 + nout, l0.h1[part]) - o.hlo);
            o.ll_pitch_b = (unsigned)l1.in_pitch * 4u;
            o.ll_s = sbase + l1.in_off + (unsigned)((o.orow - c0_0) * l1.in_pitch + hl + 2 * cp) * 4u;
            o.low = nullptr;
            o.Wo = l0.Wo;
            o.band = (size_t)l0.Ho * l0.Wo;
            o.hi = l0.highs + (size_t)plane * 3 * o.band + (long long)o.orow * l0.Wo + 2 * cp;
            o.vec2 = l0.vec2 != 0; o.low_vec2 = false;
            o.c1ok = 2 * cp + 1 < l0.Wo;
            typename std::conditional<C::kRegTaps, RegTaps<L>, ConstTaps>::type taps(p.t, lds32t(sbase + p.zrow_off));
            float2 acc[H2][4];
            int st = 0;
            unsigned ph = 0;
#pragma unroll 1
            for (int k = 0; k < nst; ++k) {
                mbar_wait(bar_wait + 8u * st, ph);
                if (C::kPrefetch) {   // the windows of row pair u + PFD are requested before row pair u is filtered
                    constexpr int PFD = 1;
                    float v[PFD + 1][2][NE];
#pragma unroll
                    for (int u = 0; u < PFD; ++u) {
                        B200W_CHK(rp + k * PS + u, 8);
                        const int2 ro = rp[k * PS + u];
                        afbt_load<L, OFF>(v[u], lane_ring + (unsigned)ro.x, lane_ring + (unsigned)ro.y);
                    }
#pragma unroll
                    for (int u = 0; u < PS; ++u) {
                        if (u + PFD < PS) {
                            B200W_CHK(rp + k * PS + u + PFD, 8);
                            const int2 rn = rp[k * PS + u + PFD];
                            afbt_load<L, OFF>(v[(u + PFD) % (PFD + 1)], lane_ring + (unsigned)rn.x, lane_ring + (unsigned)rn.y);
                        }
                        afbt_pair<L, OFF>(taps, v[u % (PFD + 1)], acc, u % H2);
                        afbt_store<L, OFF, false>(acc[kRotate ? 0 : (u + 1) % H2], o);
                        afbt_rotate<L, OFF>(acc);
                    }
                } else
#pragma unroll
                for (int u = 0; u < PS; ++u) {
                    B200W_CHK(rp + k * PS + u, 8);
                    const int2 ro = rp[k * PS + u];
                    float v[2][NE];
                    afbt_load<L, OFF>(v, lane_ring + (unsigned)ro.x, lane_ring + (unsigned)ro.y);
                    afbt_pair<L, OFF>(taps, v, acc, u % H2);
                    afbt_store<L, OFF, false>(acc[kRotate ? 0 : (u + 1) % H2], o);
                    afbt_rotate<L, OFF>(acc);
                }
                mbar_arrive(bar_rel + 8u * st);
                if (++st == D) { st = 0; ph ^= 1u; }
            }
        }
    }

    // ================================ levels 1 .. J-1: input image in shared memory ================================
#pragma unroll 1
    for (int j = 1; j < p.J; ++j) {
        const AfbTmaLevel& lv = p.lv[j];
        const bool last = j + 1 == p.J;
        __syncthreads();   // the previous level's low-pass rows are complete
        {   // extension columns of the input image, all rows of the part
            const int* const cf = tabs + lv.cfix_off;
            const int n = lv.in_pitch - lv.Wreal;
            const int rows = p.lv[j - 1].c1[part] - p.lv[j - 1].c0[part];
            const unsigned img = sbase + lv.in_off;
            for (int e = lane; e < n; e += 32) {
                const int d = cf[2 * e], s = cf[2 * e + 1];
                for (int r = warp; r < rows; r += NT / 32) {
                    const unsigned rowa = img + (unsigned)(r * lv.in_pitch) * 4u;
                    sts32t(rowa + 4u * d, s >= 0 ? lds32t(rowa + 4u * s) : 0.f);
                }
            }
        }
        __syncthreads();
        if (warp >= kProducerWarp) continue;
        const int ct = tid;
        const int c0 = lv.c0[part], c1 = lv.c1[part];
        const int g = ct / lv.ncp;
        const int cp = ct - g * lv.ncp;
        const int i0 = c0 + g * lv.R;
        if (i0 >= c1) continue;
        const int nout = min(lv.R, c1 - i0);
        const int npairs = nout + H2 - 1;
        const int* const rt = tabs + lv.rtab_off + 2 * (i0 - c0);
        const unsigned lane_b = sbase + (unsigned)cp * 16u;   // + table entry = the window of this lane in that row
        AfbtOut o;
        o.orow = i0 - (H2 - 1);
        o.i0 = i0; o.nout = nout;
        o.hlo = max(i0, lv.h0[part]);
        o.hn = max(0, min(i0 + nout, lv.h1[part]) - o.hlo);
        o.ll_pitch_b = 0; o.ll_s = 0;
        if (!last) {
            const AfbTmaLevel& nx = p.lv[j + 1];
            o.ll_pitch_b = (unsigned)nx.in_pitch * 4u;
            o.ll_s = sbase + nx.in_off + (unsigned)((o.orow - c0) * nx.in_pitch + hl + 2 * cp) * 4u;
        }
        o.Wo = lv.Wo;
        o.band = (size_t)lv.Ho * lv.Wo;
        o.low = last ? lv.low + (size_t)plane * o.band + (long long)o.orow * lv.Wo + 2 * cp : nullptr;
        o.hi = lv.highs + (size_t)plane * 3 * o.band + (long long)o.orow * lv.Wo + 2 * cp;
        o.vec2 = lv.vec2 != 0; o.low_vec2 = lv.low_vec2 != 0;
        o.c1ok = 2 * cp + 1 < lv.Wo;
        typename std::conditional<C::kRegTaps, RegTaps<L>, ConstTaps>::type taps(p.t, lds32t(sbase + p.zrow_off));
        float2 acc[H2][4];
        constexpr int UQ = kRotate ? 1 : H2;
#pragma unroll 1
        for (int qb = 0; qb < npairs; qb += UQ) {
#pragma unroll
            for (int u = 0; u < UQ; ++u) {
                if (qb + u < npairs) {
                    B200W_CHK(rt + 2 * (qb + u), 8);
                    const int2 ro = *reinterpret_cast<const int2*>(rt + 2 * (qb + u));
                    float v[2][NE];
                    afbt_load<L, OFF>(v, lane_b + (unsigned)ro.x, lane_b + (unsigned)ro.y);
                    afbt_pair<L, OFF>(taps, v, acc, u);
                    if (last) afbt_store<L, OFF, true>(acc[kRotate ? 0 : (u + 1) % H2], o);
                    else afbt_store<L, OFF, false>(acc[kRotate ? 0 : (u + 1) % H2], o);
                    afbt_rotate<L, OFF>(acc);
                }
            }
        }
    }
}

// ---- host: plan + launch ------------------------------------------------------------------------------------------
template <int L, int OFF>
static bool afb_tma_plan_t(const AfbParams& p, int sms, bool force, int G_req, int D_req, bool noboxes, AfbTmaParams& tp) {
    using C = AfbT<L, OFF>;
    constexpr int NE = C::NE, SR = C::SR, NTC = C::NTC;
    const int J = p.J;
    if (J < 2) return false;
    const bool per = p.mode == B200W_MODE_PERIODIZATION;
    constexpr int off = OFF, hl = OFF + C::S;
    const AfbLevel& x0 = p.lv[0];
    // level 0 comes in through tensor maps: 16-byte aligned base and strides; every level writes dense outputs
    if ((x0.x_rs & 3) || (x0.x_ps & 3) || !aligned_to(x0.x, 16) || x0.x_rs < x0.Wreal) return false;
    for (int j = 0; j < J; ++j) {
        const AfbLevel& lv = p.lv[j];
        if (lv.offW != off || lv.offH != off) return false;
        if (!lv.highs || !lv.st_hi || lv.hi_scale != 1.f || lv.hi_shift != 0.f) return false;   // plain DWT only
        if (lv.Wo < 2 || lv.Ho < 1) return false;
    }
    if (!p.lv[J - 1].low) return false;
    const bool wraps = per || p.mode == B200W_MODE_PERIODIC;
    int parts = std::min(kMaxParts, std::max(1, sms / p.planes));
    if (wraps) parts = 1;   // a part would need rows from the far end of the image
    parts = std::min(parts, p.lv[J - 1].Ho);
    if (!force && short_last_wave((long long)p.planes * parts, sms)) return false;
    AfbTmaParams& t = tp;
    t.J = J; t.planes = p.planes; t.parts = parts; t.mode = p.mode;
    for (int i = 0; i < kMaxTemplTaps; ++i) {
        t.t.w_lo[i] = p.t.w_lo[i]; t.t.w_hi[i] = p.t.w_hi[i];
        t.t.h_lo2[i] = p.t.h_lo2[i]; t.t.h_hi2[i] = p.t.h_hi2[i];
    }
    // rows: every level's output rows are split evenly over the parts (what a part stores); a part computes those
    // plus whatever the next level's computed rows read through the row extension
    for (int j = 0; j < J; ++j) {
        AfbTmaLevel& lv = t.lv[j];
        const AfbLevel& s = p.lv[j];
        lv.low = j == J - 1 ? s.low : nullptr;
        lv.highs = s.highs;
        lv.H = s.H; lv.W = s.W; lv.Hreal = s.Hreal; lv.Wreal = s.Wreal; lv.Ho = s.Ho; lv.Wo = s.Wo;
        lv.ncp = (s.Wo + 1) / 2;
        lv.vec2 = ((s.Wo % 2) == 0 && aligned_to(s.highs, 8)) ? 1 : 0;
        lv.low_vec2 = (j == J - 1 && (s.Wo % 2) == 0 && aligned_to(s.low, 8)) ? 1 : 0;
        if (lv.ncp > NTC) return false;
        for (int q = 0; q < kMaxParts; ++q) lv.c0[q] = lv.c1[q] = lv.h0[q] = lv.h1[q] = 0;
        for (int q = 0; q < parts; ++q) {
            lv.h0[q] = (int)((long long)s.Ho * q / parts);
            lv.h1[q] = (int)((long long)s.Ho * (q + 1) / parts);
        }
    }
    for (int q = 0; q < parts; ++q) {
        t.lv[J - 1].c0[q] = t.lv[J - 1].h0[q];
        t.lv[J - 1].c1[q] = t.lv[J - 1].h1[q];
        for (int j = J - 2; j >= 0; --j) {
            const AfbLevel& nx = p.lv[j + 1];   // reads this level's low-pass image
            int lo = t.lv[j].h0[q], hi = t.lv[j].h1[q];
            const int r_lo = 2 * t.lv[j + 1].c0[q] - off, r_hi = 2 * (t.lv[j + 1].c1[q] - 1) - off + L - 1;
            for (int r = r_lo; r <= r_hi; ++r) {
                int sr = r;
                if (r < 0 || r >= nx.Hreal) {
                    if (r >= 0 && r < nx.H) continue;   // zero extension
                    sr = ext_index(r, nx.H, p.mode);
                    if (sr < 0 || sr >= nx.Hreal) continue;   // zero row
                }
                lo = std::min(lo, sr);
                hi = std::max(hi, sr + 1);
            }
            t.lv[j].c0[q] = lo;
            t.lv[j].c1[q] = hi;
        }
    }
    int maxrows[kMaxLevels];
    for (int j = 0; j < J; ++j) {
        maxrows[j] = 0;
        for (int q = 0; q < parts; ++q) maxrows[j] = std::max(maxrows[j], t.lv[j].c1[q] - t.lv[j].c0[q]);
    }
    // segments: level 0 = the row streams (each needs ring stages and barriers), later levels as many as lanes allow
    {
        AfbTmaLevel& lv = t.lv[0];
        // streams: the busiest SM sub-partition bounds the level (the march is FP32-pipe bound): it runs
        // ceil(warps / 4) warps for R + L/2 - 1 row pairs each -- fewer, longer streams often beat filling every lane
        const int gmax = std::min(std::min(C::MAXG, std::max(1, NTC / lv.ncp)), std::min(32, maxrows[0]));
        int G = 1;
        long long best = -1;
        for (int g = 1; g <= gmax; ++g) {
            const int warps = ceil_div(g * lv.ncp, 32);
            const long long cost = (long long)ceil_div(warps, 4) * (ceil_div(maxrows[0], g) + C::H2 - 1);
            if (best < 0 || cost < best) { best = cost; G = g; }
        }
        if (G_req > 0) G = std::min(gmax, G_req);
        lv.R = ceil_div(maxrows[0], G);
        lv.nseg = ceil_div(maxrows[0], lv.R);
    }
    for (int j = 1; j < J; ++j) {
        AfbTmaLevel& lv = t.lv[j];
        const int G = std::min(std::max(1, NTC / lv.ncp), maxrows[j]);
        lv.R = ceil_div(maxrows[j], G);
        lv.nseg = ceil_div(maxrows[j], lv.R);
    }
    // level-0 tiles: column pairs split evenly over the fewest tiles of at most 256 floats
    {
        const int ncp = t.lv[0].ncp;
        int ns = 1;
        while (ns <= kTmaMaxStrips && 4 * ceil_div(ncp, ns) + NE - 4 > 256) ++ns;
        if (ns > kTmaMaxStrips) return false;
        t.nstrips = ns;
        t.cps = ceil_div(ncp, ns);
        t.BW = (4 * t.cps + NE - 4 + 31) / 32 * 32;
        if (t.BW > 256) return false;
    }
    // shared-memory layout: [barriers | tables | zero row | LL_0 | ring (LL_1.. alias it: the ring is dead by then)]
    size_t o = 0;
    t.bar_off = 0;
    o += (size_t)3 * 8 * t.lv[0].nseg * 8;   // up to 8 stages
    int ti = 0;
    for (int j = 0; j < J; ++j) {
        t.lv[j].rtab_off = ti;
        ti += (2 * maxrows[j] + L + 1) & ~1;   // int2 reads: even offsets
    }
    int maxpitch = 4;
    for (int j = 1; j < J; ++j) {
        AfbTmaLevel& lv = t.lv[j];
        // the row holds hl extension floats, the data, and everything the last lane's window / the stores touch
        const int need = std::max(4 * (lv.ncp - 1) + NE, hl + 2 * t.lv[j - 1].ncp);
        lv.in_pitch = (need + 3) & ~3;
        lv.in_rows = maxrows[j - 1];
        lv.cfix_off = ti;
        ti += 2 * (lv.in_pitch - lv.Wreal);
        maxpitch = std::max(maxpitch, lv.in_pitch);
    }
    {
        t.fix0_off = ti;
        int n = 0;
        for (int s = 0; s < t.nstrips; ++s) {
            const int b = 4 * s * t.cps - hl;
            const int pairs = std::min(t.cps, t.lv[0].ncp - s * t.cps);
            if (pairs < 1) return false;
            const int fmax = 4 * (pairs - 1) + NE - 1;
            const int nl = s == 0 ? hl : 0;
            const int fr = std::max(nl, t.lv[0].Wreal - b);
            n += nl + std::max(0, fmax + 1 - fr);
        }
        t.fix0_n = n;
        ti += 2 * n * SR;
    }
    // per-pair row tables of the first level: G streams x (R + L/2 - 1 rounded up to whole stages) x int2
    t.rp0_stride = ceil_div(t.lv[0].R + C::H2 - 1, C::PS) * C::PS;
    t.rp0_off = ti;
    ti += 2 * t.rp0_stride * t.lv[0].nseg;
    t.tab_ints = ti;
    t.tab_off = (int)o;
    o += (size_t)ti * 4;
    o = (o + 15) & ~(size_t)15;
    t.zrow_off = (int)o;
    t.zrow_floats = maxpitch;
    o += (size_t)maxpitch * 4;
    o = (o + 127) & ~(size_t)127;
    t.lv[0].in_pitch = 0; t.lv[0].in_off = 0; t.lv[0].in_rows = 0; t.lv[0].cfix_off = 0;
    t.lv[1].in_off = (int)o;
    o += (size_t)t.lv[1].in_rows * t.lv[1].in_pitch * 4;
    o = (o + 127) & ~(size_t)127;
    t.ring_off = (int)o;
    size_t later = 0;   // LL_1 .. LL_{J-2} (inputs of levels 2 ..) live where the ring was
    for (int j = 2; j < J; ++j) {
        t.lv[j].in_off = t.ring_off + (int)later;
        later += ((size_t)t.lv[j].in_rows * t.lv[j].in_pitch * 4 + 127) & ~(size_t)127;
    }
    const size_t stage_b = (size_t)t.nstrips * SR * t.BW * 4;
    if (o + std::max(later, 2 * stage_b * t.lv[0].nseg) > kMaxDynSmem) return false;
    int D = (int)((kMaxDynSmem - o) / (stage_b * t.lv[0].nseg));
    D = std::min(D, 8);
    if (D_req > 0) D = std::max(2, std::min(D, D_req));
    if (D < 2) return false;
    t.D = D;
    t.smem_bytes = (int)(o + std::max(later, (size_t)D * stage_b * t.lv[0].nseg));
    // the tables, per part (the same layout the kernel indexes: row tables, column-patch tables, ring patch table)
    if ((long long)t.tab_ints * parts > kAfbTabMax) return false;
    {
        auto map = [&](int sidx, int n, int real) {
            if (sidx >= 0 && sidx < real) return sidx;
            if (sidx >= 0 && sidx < n) return -1;                 // zero extension inside the logical size
            if (p.mode == B200W_MODE_ZERO) return -1;
            const int m = ext_index(sidx, n, p.mode);
            return (m < 0 || m >= real) ? -1 : m;
        };
        const int srbw4 = SR * t.BW * 4;
        const int stage_bytes = t.nstrips * srbw4;
        // Can every stage be one box of consecutive virtual rows?  Yes for 'zero'; for symmetric / reflect when every
        // extension row finds its image row in a ring slot that is still valid when it is read: the same stage, or an
        // earlier stage of the stream that is never refilled (one of the last D stages).
        bool boxes = p.mode == B200W_MODE_ZERO || p.mode == B200W_MODE_SYMMETRIC || p.mode == B200W_MODE_REFLECT;
        if (noboxes && p.mode != B200W_MODE_ZERO) boxes = false;
        for (int pass = 0; pass < 2; ++pass) {   // pass 0: decide `boxes`; pass 1: fill the tables
        for (int q = 0; q < parts; ++q) {
            int* const tb = t.tab + q * t.tab_ints;
            const AfbTmaLevel& lz = t.lv[0];
            for (int g = 0; g * lz.R < lz.c1[q] - lz.c0[q]; ++g) {
                const int i0 = lz.c0[q] + g * lz.R;
                const int npairs = std::min(lz.R, lz.c1[q] - i0) + C::H2 - 1;
                const int nst = ceil_div(npairs, C::PS);
                const int r_start = 2 * i0 - off;
                for (int qq = 0; qq < t.rp0_stride; ++qq)
                    for (int e = 0; e < 2; ++e) {
                        const int v = r_start + 2 * qq + e;          // virtual input row of this pair
                        int rowv = v;                                 // the (virtual) row whose ring slot is read
                        if (boxes && qq < npairs && !(v >= 0 && v < lz.H)) {
                            const int m = map(v, lz.H, lz.Hreal);
                            if (m >= 0) {
                                const int ks = m >= r_start ? (m - r_start) / SR : -1, k = (v - r_start) / SR;
                                if (ks < 0 || ks >= nst || ks > k || (ks < k && ks + t.D < nst)) boxes = false;
                                rowv = m;
                            }
                        }
                        if (pass == 1) {
                            const int kk = (rowv - r_start) / SR, ii = (rowv - r_start) - kk * SR;
                            tb[t.rp0_off + 2 * (g * t.rp0_stride + qq) + e] =
                                t.ring_off + (g * t.D + kk % t.D) * stage_bytes + ii * t.BW * 4;
                        }
                    }
            }
            if (pass == 0) continue;
            for (int i = 0; i < t.rp0_off; ++i) tb[i] = 0;
            for (int j = 0; j < J; ++j) {
                const AfbTmaLevel& lv = t.lv[j];
                const int c0 = lv.c0[q];
                const int nr = 2 * (lv.c1[q] - c0) + L;
                for (int e = 0; e < nr; ++e) {
                    const int m = map(2 * c0 - off + e, lv.H, lv.Hreal);
                    int val = m;
                    if (j > 0) val = m < 0 ? t.zrow_off : lv.in_off + (m - t.lv[j - 1].c0[q]) * lv.in_pitch * 4;
                    tb[lv.rtab_off + e] = val;
                }
                if (j > 0) {   // patch table of the input image: every float of a row that is not image data
                    const int n = lv.in_pitch - lv.Wreal;
                    for (int k = 0; k < n; ++k) {
                        const int f = k < hl ? k : lv.Wreal + k;      // float index inside the row (column f - hl)
                        const int m = map(f - hl, lv.W, lv.Wreal);
                        tb[lv.cfix_off + 2 * k] = f;
                        tb[lv.cfix_off + 2 * k + 1] = m < 0 ? -1 : m + hl;
                    }
                }
            }
            // ring patch table: extension columns inside the tiles of a stage, one entry per (row of the stage,
            // column): (destination, source) byte offsets from the stage base; source -1 = leave the engine's zero
            const AfbTmaLevel& l0t = t.lv[0];
            int base = 0;
            for (int s = 0; s < t.nstrips && p.mode != B200W_MODE_ZERO; ++s) {
                const int b = 4 * s * t.cps - hl;                          // image column of the tile's first float
                const int pairs = std::min(t.cps, l0t.ncp - s * t.cps);
                const int fmax = 4 * (pairs - 1) + NE - 1;                 // last float a lane of this tile reads
                const int nl = s == 0 ? hl : 0;                            // left extension (first tile only)
                const int fr = std::max(nl, l0t.Wreal - b);                // first float right of the data
                const int n = nl + std::max(0, fmax + 1 - fr);
                for (int k = 0; k < n; ++k) {
                    const int f = k < nl ? k : fr + (k - nl);
                    const int m = map(b + f, l0t.W, l0t.Wreal);
                    int src = -1;
                    if (m >= 0) {   // the tile that holds column m: this one if it does, else the one its pair lives in
                        int s2 = s;
                        if (m < b || m >= b + t.BW) s2 = std::min(t.nstrips - 1, std::max(0, (m + hl) / (4 * t.cps)));
                        src = s2 * srbw4 + (m - (4 * s2 * t.cps - hl)) * 4;
                    }
                    const int dst = s * srbw4 + f * 4;
                    for (int i = 0; i < SR; ++i) {
                        tb[t.fix0_off + 2 * (i * t.fix0_n + base + k)] = dst + i * t.BW * 4;
                        tb[t.fix0_off + 2 * (i * t.fix0_n + base + k) + 1] = src < 0 ? -1 : src + i * t.BW * 4;
                    }
                }
                base += n;
            }
        }
        if (pass == 0 && !boxes) {   // the tables are rebuilt with every pair reading its own virtual rows
            // (nothing to undo: pass 0 wrote nothing)
        }
        }
        t.boxes = boxes ? 1 : 0;
    }
    // tensor maps of the level-0 input
    const uint64_t dims[3] = {(uint64_t)x0.Wreal, (uint64_t)x0.Hreal, (uint64_t)p.planes};
    const uint64_t strides[2] = {(uint64_t)x0.x_rs * 4, (uint64_t)x0.x_ps * 4};
    const uint32_t box_full[3] = {(uint32_t)t.BW, (uint32_t)SR, 1}, box_row[3] = {(uint32_t)t.BW, 1, 1};
    if (p.planes > 1 && (strides[1] & 15)) return false;
    if (!tma_make_map_f32(&t.map_full, x0.x, 3, dims, strides, box_full)) return false;
    if (!tma_make_map_f32(&t.map_row, x0.x, 3, dims, strides, box_row)) return false;
    return true;
}

template <int L, int OFF, int NTAB>
static int launch_afb_tma_n(const AfbTmaParamsN<NTAB>& tp, cudaStream_t st) {
    using C = AfbT<L, OFF>;
    if (const cudaError_t e = allow_max_dyn_smem<afb_tma_kernel<L, OFF, NTAB>>()) return set_last_cuda_error(e);
#ifdef B200W_BOUNDS
    {
        BoundsList b;
        for (int j = 0; j < tp.J; ++j) {
            const AfbTmaLevel& lv = tp.lv[j];
            b.add(lv.highs, sizeof(float) * (size_t)tp.planes * 3 * lv.Ho * lv.Wo);
            if (lv.low) b.add(lv.low, sizeof(float) * (size_t)tp.planes * lv.Ho * lv.Wo);
        }
        bounds_set(b, st);
    }
#endif
    const cudaError_t le = launch_pdl(afb_tma_kernel<L, OFF, NTAB>, (unsigned)(tp.planes * tp.parts), C::NT,
                                      (size_t)tp.smem_bytes, st, tp);
    note_launch("afb_tma_kernel");
    const cudaError_t e = le != cudaSuccess ? le : cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

// the smaller parameter block when the tables fit in it (see AfbTmaParamsN)
template <int L, int OFF>
static int launch_afb_tma_t(const AfbTmaParams& tp, cudaStream_t st) {
    const int n = tp.tab_ints * tp.parts;
    if (n > kAfbTabSmall) return launch_afb_tma_n<L, OFF, kAfbTabMax>(tp, st);
    AfbTmaParamsN<kAfbTabSmall> sp;
    static_cast<AfbTmaHead&>(sp) = tp;
    std::copy(tp.tab, tp.tab + n, sp.tab);
    std::fill(sp.tab + n, sp.tab + kAfbTabSmall, 0);
    return launch_afb_tma_n<L, OFF, kAfbTabSmall>(sp, st);
}

bool afb_tma_plan(const AfbParams& p, int L, int sms, bool force, int G, int D, bool noboxes, AfbTmaParams& tp) {
    if (!tma_encode_fn()) return false;
    const bool per = p.mode == B200W_MODE_PERIODIZATION;
#define X(LL) return per ? afb_tma_plan_t<LL, afbt_off(LL, true)>(p, sms, force, G, D, noboxes, tp) \
                         : afb_tma_plan_t<LL, afbt_off(LL, false)>(p, sms, force, G, D, noboxes, tp)
    B200W_FOR_EACH_L(X)
#undef X
    return false;
}

int launch_afb_tma(const AfbTmaParams& tp, int L, cudaStream_t st) {
    const bool per = tp.mode == B200W_MODE_PERIODIZATION;
#define X(LL) return per ? launch_afb_tma_t<LL, afbt_off(LL, true)>(tp, st) \
                         : launch_afb_tma_t<LL, afbt_off(LL, false)>(tp, st)
    B200W_FOR_EACH_L(X)
#undef X
    return B200W_ERR_BAD_TAPS;
}

}  // namespace b200w
