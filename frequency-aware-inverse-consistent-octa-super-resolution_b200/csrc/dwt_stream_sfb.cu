// Synthesis filter bank, streaming register-blocked kernel (fused upsample + filter + accumulate).
//
// Replaces the six F.conv_transpose2d + three adds of SFB2D.forward (pw/dwt/lowlevel.py:671-680, 226-271), the
// J-level loop of DWTInverse.forward incl. the 'unpad' crop (pw/dwt/transform2d.py:134-148), and -- with the
// analysis taps and a crop -- AFB2D.backward (pw/dwt/lowlevel.py:349-365).
//
// "A-space": a = n + off (off = L-2, periodization L/2-1), so output a uses taps of parity a&1 only:
//     y[a] = sum_u c[(a>>1) - u] * g[(a&1) + 2u],  u = 0 .. L/2-1            (the polyphase form of sfb1d)
// A thread owns FOUR adjacent output columns (two coefficient pairs) and marches down Rp output row pairs:
//   * W synthesis in registers: the L/2+1 coefficients of each of the four sub-bands in its window give 4 outputs
//     for the h_lo branch (LL, HL) and 4 for the h_hi branch (LH, HH),
//   * H synthesis "accumulate forward": the coefficient row is scattered into the L/2 output row pairs it
//     contributes to (8 accumulators each); the oldest pair is complete and is written with 128-bit stores.
// The loop is unrolled by L/2 rows so that the accumulator ring has static register names.
//
// Input staging mirrors the analysis kernel: interior threads (window and outputs inside the arrays) share a
// per-WARP cp.async ring -- every lane copies its own coefficient pair of each sub-band row (64-bit copies when
// the rows are 8-byte aligned, else 2 x 32-bit), the last lane of a run adds the trailing pairs, D rows deep --
// and read their window with 64-bit shared loads; only __syncwarp is needed.  Coefficient rows outside the
// sub-band are zero-filled (periodization: wrapped).  The few border output columns run in separate CTAs, one
// thread per output position.  A null `highs` means zeros (transform2d.py:137-139); out_h / out_w smaller than
// the natural size crop.
#include <algorithm>
#include <cmath>
#include "dwt_levels.cuh"

namespace b200w {

constexpr int sfb_off(int L, bool per) { return per ? L / 2 - 1 : L - 2; }
constexpr int sfb_a0_off(int L, bool per) { return sfb_off(L, per) & ~1; }          // A-space start of thread 0 (even)
constexpr int sfb_q0_off(int L, bool per) { return sfb_a0_off(L, per) / 2; }
constexpr int sfb_n0_off(int L, bool per) { return sfb_a0_off(L, per) - sfb_off(L, per); }   // 0 or -1
constexpr int sfb_ks_off(int L, bool per) { return sfb_q0_off(L, per) - L / 2 + 1; }        // first needed coefficient
constexpr int sfb_shift2(int L, bool per) { return ((sfb_ks_off(L, per) % 2) + 2) % 2; }    // pad down to even

constexpr int kSfbMaxRuns = 5;
constexpr int kSfbMinThreads = 8;   // interior threads per row needed for the ring path (=> at most kSfbMaxRuns runs)

template <int L, int S2>
struct SfbStreamCfg {
    static constexpr int H2 = L / 2;
    static constexpr int NCF = 2 * ((S2 + H2 + 2) / 2);   // coefficients per window (even)
    static constexpr int NS = NCF / 2;                    // float2 slots per window
    static constexpr int RPB = 32 + kSfbMaxRuns * (NS - 1);   // float2 slots per band row of the ring
    static constexpr int STAGE = 4 * RPB;                 // float2 per stage (one coefficient row, four bands)
    static constexpr int D = L <= 8 ? 8 : 6;              // ring depth (coefficient rows)
    static constexpr size_t smem = sizeof(float2) * (size_t)(kStreamNT / 32) * D * STAGE;
    static constexpr int MINB = L <= 8 ? 5 : (L <= 12 ? 4 : 3);
};
template <int L>
struct SfbSmem {   // one launch may mix 64-bit and 32-bit staged levels: size the ring for the larger window
    static constexpr size_t a = SfbStreamCfg<L, sfb_shift2(L, false)>::smem;
    static constexpr size_t b = SfbStreamCfg<L, sfb_shift2(L, true)>::smem;
    static constexpr size_t c = SfbStreamCfg<L, 0>::smem;
    static constexpr size_t value = a > b ? (a > c ? a : c) : (b > c ? b : c);
};

// source row of coefficient row kr: itself inside the sub-band, else zero (-1) or the periodic wrap
__device__ __forceinline__ int sfb_src_row(int kr, int h, int periodic) {
    if ((unsigned)kr < (unsigned)h) return kr;
    return periodic ? coef_index_far(kr, h, periodic) : -1;
}

// block until every CTA item of the previous level of this plane has been published
__device__ __forceinline__ void sfb_chain_wait(const unsigned* ctr, unsigned need) {
    if (ctr != nullptr) {
        if (threadIdx.x == 0)
            while (ld_acquire_u32(ctr) < need) __nanosleep(20);
        __syncthreads();
    }
}

// rows of a chain position that an owner CTA works on (owner kernel only): it computes output rows [n0, n1) -- into
// its shared-memory image of the level output, or into global memory at the last position
struct SfbOwnRows {
    int n0, n1;
    int itemsA;            // thread items of the interior class over those rows
    unsigned low_s;        // SMEM_LOW: shared address of the low-pass image (row low_row0, column 0)
    int low_row0;
};

__device__ __forceinline__ float2 lds64(unsigned addr) {
    B200W_CHK_S(addr, 8);
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds32(unsigned addr) {
    B200W_CHK_S(addr, 4);
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}

// ---- interior threads: per-warp cp.async ring ----------------------------------------------------------
// `it` = the thread's item (segment-major: segment * ntA + interior thread).  OWNER: the rows come from `own`
// instead of the whole level; SMEM_LOW (owner kernel, every position but the first): the low-pass input is the
// previous position's output in shared memory -- only the three detail bands go through the ring.
template <int L, int V, int S2, bool OWNER = false, bool SMEM_LOW = false>
__device__ __forceinline__ void sfb_ring_cta(const SfbParams& p, const SfbLevel& lv, int plane, int it, float2* ring_all,
                                             const unsigned* wait_ctr, unsigned wait_need, const SfbOwnRows& own) {
    using C = SfbStreamCfg<L, S2>;
    constexpr int H2 = C::H2, NCF = C::NCF, NS = C::NS, D = C::D;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int itemsA = OWNER ? own.itemsA : lv.itemsA;
    const bool active = it < itemsA;
    const int ntA = lv.ntA;
    const int itc = active ? it : itemsA - 1;        // inactive lanes shadow the last item (no copies, no stores)
    const int seg = itc / ntA;
    const int tl = itc - seg * ntA;
    const int t = lv.tA0 + tl;
    const int m0 = (OWNER ? (own.n0 + lv.offH) >> 1 : lv.m_lo) + seg * lv.Rp;   // first output row pair (A-space)
    const int m_end = ((lv.offH + (OWNER ? own.n1 : lv.out_h) - 1) >> 1) + 1;
    const int nm = min(lv.Rp, m_end - m0);
    const int nrows = active ? nm + H2 - 1 : 0;                      // coefficient rows feeding them
    const int kr0 = m0 - (H2 - 1);
    const int h = lv.h, w = lv.w, periodic = p.periodic;
    const int kb = 2 * t + lv.kb_off;                                // first staged coefficient column (>= 0)
    const int seg_first = __shfl_sync(0xffffffffu, seg, 0);
    const int slot = lane + (NS - 1) * (seg - seg_first);
    const bool run_last = NS > 1 && active && (lane == 31 || tl == ntA - 1);
    const size_t band = (size_t)h * w;
    const long long low_rs = lv.low_rs;
    const float* lowcol = lv.low + (long long)plane * lv.low_ps + kb;
    const bool has_hi = lv.highs != nullptr;
    const float* hicol = has_hi ? lv.highs + (size_t)plane * 3 * band + kb : lowcol;
    float2* ring = ring_all + (size_t)(tid >> 5) * D * C::STAGE;
    const unsigned ring_s = (unsigned)__cvta_generic_to_shared(ring) + (unsigned)slot * 8u;
    const bool vec2 = lv.vec2 != 0;   // V == 0: copy width chosen at run time (same window geometry either way)

    // stage coefficient row q of this lane's segment into ring stage `st`.  Rows inside the sub-band take the
    // plain cp.async (the zero-filling form costs three padding instructions each); zero rows and a missing
    // `highs` are cleared with shared stores.
    auto issue = [&](int q, int st) {
        // nothing is staged beyond this lane's segment: the lanes that would read those slots (same run, same
        // segment) are past their last row too, and an idle lane must not touch slots that belong to others
        if (q < nrows) {
            const int sr = sfb_src_row(kr0 + q, h, periodic);
#pragma unroll
            for (int b = SMEM_LOW ? 1 : 0; b < 4; ++b) {
                const unsigned dst = ring_s + (unsigned)((st * 4 + b) * C::RPB) * 8u;
                if (sr >= 0 && (b == 0 || has_hi)) {
                    const float* src = b == 0 ? lowcol + (long long)sr * low_rs : hicol + (size_t)(b - 1) * band + (size_t)sr * w;
                    if (V == 2 || (V == 0 && vec2)) {
                        cp_async<2>(dst, src);
                        if (run_last) {
#pragma unroll
                            for (int k = 1; k < NS; ++k) cp_async<2>(dst + 8u * k, src + 2 * k);
                        }
                    } else {
                        cp_async<1>(dst, src);
                        cp_async<1>(dst + 4u, src + 1);
                        if (run_last) {
#pragma unroll
                            for (int k = 2; k < NCF; ++k) cp_async<1>(dst + 4u * k, src + k);
                        }
                    }
                } else {
                    float2* d = ring + (st * 4 + b) * C::RPB + slot;
                    B200W_CHK(d, 8);
                    if (run_last) B200W_CHK(d + NS - 1, 8);
                    d[0] = make_float2(0.f, 0.f);
                    if (run_last) {
#pragma unroll
                        for (int k = 1; k < NS; ++k) d[k] = make_float2(0.f, 0.f);
                    }
                }
            }
        }
    };

    const int row_lo = OWNER ? own.n0 : 0, row_hi = OWNER ? own.n1 : lv.out_h;
    const int n0 = 4 * t + lv.n0_off;                                // first output column (all four are valid)
    const long long y_rs = lv.y_rs;
    int nrow = 2 * m0 - lv.offH;                                     // output row of the even row of pair m0
    float* yq = lv.y + (long long)plane * lv.y_ps + (long long)nrow * y_rs + n0;   // dereferenced only where valid
    const int yv = lv.y_vec;

    // warp-uniform trip count (lanes of a warp may sit in segments of different length)
    int npw = nrows;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) npw = max(npw, __shfl_xor_sync(0xffffffffu, npw, o));

    if (!OWNER) sfb_chain_wait(wait_ctr, wait_need);
#pragma unroll 1
    for (int s = 0; s < D - 1; ++s) {
        issue(s, s);
        cp_async_commit();
    }
    // SMEM_LOW: shared address of this lane's low-pass window in row 0
    const unsigned loww_s = SMEM_LOW ? own.low_s + (unsigned)(kb - own.low_row0 * (int)low_rs) * 4u : 0u;
    float2 acc[H2][4];    // ring of pending output row pairs: even row (cols 0-1, 2-3), odd row (cols 0-1, 2-3)
    int st_r = 0, st_w = D - 1;
    // long filters keep the accumulator ring in age order and shift it after each store instead of unrolling by
    // L/2 (the unrolled body would not fit the instruction cache)
    constexpr bool kRotate = L >= 10;
    constexpr int UQ = kRotate ? 1 : H2;
    for (int qb = 0; qb < npw; qb += UQ) {
#pragma unroll
        for (int ph = 0; ph < UQ; ++ph) {
            const int q = qb + ph;
            if (q < npw) {   // warp-uniform
                cp_async_wait<D - 2>();   // this lane's copies of row q have landed ...
                __syncwarp();             // ... and everybody's; all lanes are done reading row q-1
                issue(q + D - 1, st_w);   // refill the stage row q-1 was read from
                cp_async_commit();
                st_w = st_w + 1 == D ? 0 : st_w + 1;
                float c[4][NCF];
                const float2* src = ring + (st_r * 4) * C::RPB + slot;
#pragma unroll
                for (int b = SMEM_LOW ? 1 : 0; b < 4; ++b)
#pragma unroll
                    for (int k = 0; k < NS; ++k) {
                        B200W_CHK(src + b * C::RPB + k, 8);
                        const float2 v = src[b * C::RPB + k];
                        c[b][2 * k] = v.x;
                        c[b][2 * k + 1] = v.y;
                    }
                if (SMEM_LOW) {
                    const int sr = q < nrows ? sfb_src_row(kr0 + q, h, periodic) : -1;
                    const unsigned a = loww_s + (unsigned)(max(sr, 0) * (int)low_rs) * 4u;
#pragma unroll
                    for (int k = 0; k < NS; ++k) {
                        float2 v = make_float2(0.f, 0.f);
                        if (sr >= 0) {
                            if (V != 1) {   // V == 0: the window start is even whichever way the rows were staged
                                v = lds64(a + 8u * k);
                            } else {
                                v.x = lds32(a + 8u * k);
                                v.y = lds32(a + 8u * k + 4u);
                            }
                        }
                        c[0][2 * k] = v.x;
                        c[0][2 * k + 1] = v.y;
                    }
                }
                // W synthesis of this coefficient row: lo = h_lo branch (LL, HL), hi = h_hi branch (LH, HH)
                float lo[4], hi[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int qo = e >> 1, par = e & 1;
                    float a = 0.f, b = 0.f;
#pragma unroll
                    for (int u = 0; u < H2; ++u) {
                        const int kl = S2 + qo + H2 - 1 - u;
                        a = fmaf(c[0][kl], p.t.w_lo[par + 2 * u], a);
                        a = fmaf(c[2][kl], p.t.w_hi[par + 2 * u], a);
                        b = fmaf(c[1][kl], p.t.w_lo[par + 2 * u], b);
                        b = fmaf(c[3][kl], p.t.w_hi[par + 2 * u], b);
                    }
                    lo[e] = a;
                    hi[e] = b;
                }
                // H synthesis: coefficient row q carries taps (2u, 2u+1) of output row pair q - (H2-1) + u.  The
                // accumulators hold two adjacent columns per float2, so the updates run on the packed FFMA2 with the
                // (t, t) tap pairs from uniform registers.
                const float2 lo01 = make_float2(lo[0], lo[1]), lo23 = make_float2(lo[2], lo[3]);
                const float2 hi01 = make_float2(hi[0], hi[1]), hi23 = make_float2(hi[2], hi[3]);
#pragma unroll
                for (int u = H2 - 1; u >= 0; --u) {
                    const int sl = kRotate ? u : (ph + u + 1) % H2;
                    const float2 a0 = p.t.h_lo2[2 * u], b0 = p.t.h_hi2[2 * u];
                    const float2 a1 = p.t.h_lo2[2 * u + 1], b1 = p.t.h_hi2[2 * u + 1];
                    float2* s = acc[sl];   // [0..1] even output row (columns 0-1, 2-3), [2..3] odd output row
                    if (u == H2 - 1) {   // first contribution to that pair
                        s[0] = fmul2(lo01, a0); s[1] = fmul2(lo23, a0);
                        s[2] = fmul2(lo01, a1); s[3] = fmul2(lo23, a1);
                    } else {
                        s[0] = ffma2(lo01, a0, s[0]); s[1] = ffma2(lo23, a0, s[1]);
                        s[2] = ffma2(lo01, a1, s[2]); s[3] = ffma2(lo23, a1, s[3]);
                    }
                    s[0] = ffma2(hi01, b0, s[0]); s[1] = ffma2(hi23, b0, s[1]);
                    s[2] = ffma2(hi01, b1, s[2]); s[3] = ffma2(hi23, b1, s[3]);
                }
                // pair q - (H2-1) is complete
                if (q >= H2 - 1 && q < nrows) {
                    const float2* s = acc[kRotate ? 0 : (ph + 1) % H2];
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        const int row = nrow + r;
                        if (row >= row_lo && row < row_hi) {
                            float* d = yq + r * y_rs;
                            B200W_CHK_A(d, 16, yv == 4 ? 16 : (yv == 2 ? 8 : 4));
                            if (yv == 4) {
                                *reinterpret_cast<float4*>(d) = make_float4(s[2 * r].x, s[2 * r].y, s[2 * r + 1].x, s[2 * r + 1].y);
                            } else if (yv == 2) {
                                *reinterpret_cast<float2*>(d) = s[2 * r];
                                *reinterpret_cast<float2*>(d + 2) = s[2 * r + 1];
                            } else {
                                d[0] = s[2 * r].x; d[1] = s[2 * r].y; d[2] = s[2 * r + 1].x; d[3] = s[2 * r + 1].y;
                            }
                        }
                    }
                    nrow += 2;
                    yq += 2 * y_rs;
                }
                if (kRotate) {
#pragma unroll
                    for (int k = 0; k + 1 < H2; ++k)
#pragma unroll
                        for (int i = 0; i < 4; ++i) acc[k][i] = acc[k + 1][i];
                }
                st_r = st_r + 1 == D ? 0 : st_r + 1;
            }
        }
    }
    cp_async_wait<0>();
}

// ---- border output columns: one thread per output position ---------------------------------------------
// All (L/2)^2 x 4 coefficients of an output are loaded before any arithmetic (clamped address + select), so the
// thread pays one memory round trip; rows are done in chunks to bound the registers.
template <int L, bool OWNER = false>
__device__ __forceinline__ void sfb_border_item(const SfbParams& p, const SfbLevel& lv, int plane, int it, bool active,
                                                const unsigned* wait_ctr, unsigned wait_need, const SfbOwnRows& own) {
    constexpr int H2 = L / 2;
    if (!active) it = 0;                             // idle threads shadow item 0 (they only take part in the wait)
    const int ncB = lv.nA0 + lv.out_w - lv.nA1;      // border columns per output row
    const int ib = it / ncB;
    const int nH = (OWNER ? own.n0 : 0) + ib;
    const int e0 = it - ib * ncB;
    const int nW = e0 < lv.nA0 ? e0 : e0 - lv.nA0 + lv.nA1;
    const int h = lv.h, w = lv.w, periodic = p.periodic;
    const size_t band = (size_t)h * w;
    const float* lowp = lv.low + (long long)plane * lv.low_ps;
    const bool has_hi = lv.highs != nullptr;
    const float* hip = has_hi ? lv.highs + (size_t)plane * 3 * band : lowp;
    const int AH = nH + lv.offH, AW = nW + lv.offW;
    const int parH = AH & 1, parW = AW & 1;
    int kc[H2];
#pragma unroll
    for (int u = 0; u < H2; ++u) {
        const int k = (AW >> 1) - u;
        kc[u] = (unsigned)k < (unsigned)w ? k : (periodic ? coef_index_far(k, w, periodic) : -1);
    }
    int krow[H2];
#pragma unroll
    for (int u = 0; u < H2; ++u) krow[u] = sfb_src_row((AH >> 1) - u, h, periodic);
    if (!OWNER) sfb_chain_wait(wait_ctr, wait_need); // index arithmetic above overlaps the wait
    if (!active) return;
    float y = 0.f;
    constexpr int CH = H2 < 3 ? H2 : 3;
#pragma unroll
    for (int u0 = 0; u0 < H2; u0 += CH) {
        float v[CH][4][H2];
        bool rok[CH];
#pragma unroll
        for (int uu = 0; uu < CH; ++uu) {
            const int uH = u0 + uu;
            const int kr = uH < H2 ? krow[uH < H2 ? uH : 0] : -1;
            rok[uu] = kr >= 0;
            const int row = max(kr, OWNER ? own.low_row0 : 0);   // a zero row is read from a row that exists
            const float* lp = lowp + (long long)row * lv.low_rs;
            const float* hp = hip + (size_t)row * w;
#pragma unroll
            for (int u = 0; u < H2; ++u) {
                const int col = max(kc[u], 0);
                B200W_CHK(lp + col, 4);
                if (has_hi) { B200W_CHK(hp + col, 4); B200W_CHK(hp + band + col, 4); B200W_CHK(hp + 2 * band + col, 4); }
                v[uu][0][u] = lp[col];
                v[uu][1][u] = has_hi ? hp[col] : 0.f;
                v[uu][2][u] = has_hi ? hp[band + col] : 0.f;
                v[uu][3][u] = has_hi ? hp[2 * band + col] : 0.f;
            }
        }
#pragma unroll
        for (int uu = 0; uu < CH; ++uu) {
            const int uH = u0 + uu;
            if (uH < H2) {
                float lo = 0.f, hi = 0.f;   // W-synthesised values to be combined with h_lo / h_hi
#pragma unroll
                for (int u = 0; u < H2; ++u) {
                    const bool ok = rok[uu] && kc[u] >= 0;
                    const float gl = p.t.w_lo[parW + 2 * u], gh = p.t.w_hi[parW + 2 * u];
                    lo = fmaf(ok ? v[uu][0][u] : 0.f, gl, lo);    // LL
                    hi = fmaf(ok ? v[uu][1][u] : 0.f, gl, hi);    // LH
                    lo = fmaf(ok ? v[uu][2][u] : 0.f, gh, lo);    // HL
                    hi = fmaf(ok ? v[uu][3][u] : 0.f, gh, hi);    // HH
                }
                y = fmaf(lo, p.t.h_lo[parH + 2 * uH], y);
                y = fmaf(hi, p.t.h_hi[parH + 2 * uH], y);
            }
        }
    }
    B200W_CHK(lv.y + (long long)plane * lv.y_ps + (long long)nH * lv.y_rs + nW, 4);
    lv.y[(long long)plane * lv.y_ps + (long long)nH * lv.y_rs + nW] = y;
}

template <int L, int S2V>
__global__ void __launch_bounds__(kStreamNT, SfbStreamCfg<L, S2V>::MINB) sfb_stream_kernel(const __grid_constant__ SfbParams p) {
    extern __shared__ float2 sfb_ring_all[];
    __shared__ unsigned s_item;
    const int tid = threadIdx.x;
    unsigned item = blockIdx.x;
    if (p.J > 1) {   // work items are handed out in list order: an item only waits for earlier, running ones
        if (tid == 0) s_item = atomicAdd(p.ticket, 1u);
        __syncthreads();
        item = s_item;
    }
    int level = 0;
    for (int j = 1; j < p.J; ++j)
        if ((long long)item >= p.lv[j].cta_base) level = j;
    const SfbLevel& lv = p.lv[level];
    const unsigned local = item - (unsigned)lv.cta_base;
    const int plane = (int)(local / (unsigned)lv.cpp);
    const int cta = (int)(local - (unsigned)plane * (unsigned)lv.cpp);
    // the previous (coarser) level of this plane must be complete before its output is read as `low`
    const unsigned* wait_ctr = level > 0 ? p.done + (size_t)(level - 1) * p.planes + plane : nullptr;
    const unsigned wait_need = level > 0 ? (unsigned)p.lv[level - 1].cpp : 0u;
    const SfbOwnRows none{};
    if (cta < lv.cppA) {
        const int it = cta * kStreamNT + tid;
        // without a shift the 64-bit and the 32-bit staged windows coincide: one code path picks the copy width at
        // run time (half the code in the instruction cache); periodization shifts the 64-bit window by one
        if (S2V == 0) sfb_ring_cta<L, 0, 0>(p, lv, plane, it, sfb_ring_all, wait_ctr, wait_need, none);
        else if (lv.vec2) sfb_ring_cta<L, 2, S2V>(p, lv, plane, it, sfb_ring_all, wait_ctr, wait_need, none);
        else sfb_ring_cta<L, 1, 0>(p, lv, plane, it, sfb_ring_all, wait_ctr, wait_need, none);
    } else {
        const int it = (cta - lv.cppA) * kStreamNT + tid;
        sfb_border_item<L>(p, lv, plane, it, it < lv.itemsB, wait_ctr, wait_need, none);
    }
    if (level + 1 < p.J) {
        __syncthreads();
        if (tid == 0) signal_done(p.done + (size_t)level * p.planes + plane);
    }
}

// ---- owner kernel: every position of a synthesis chain for one (plane, part) in one CTA ------------------------
// The coarsest position reads its low-pass input from global memory through the ring like the stream kernel; every
// output but the last stays in shared memory, where the next position reads it as its low-pass input (SMEM_LOW),
// the detail bands still streaming in through the ring.  One block barrier per position, no tickets or counters.
template <int L>
struct SfbOwnerCfg {
    static constexpr int NT = L <= 8 ? kOwnerNT : 256;   // one CTA per SM; long filters need > 128 registers per thread
};

template <int L, int S2V>
__global__ void __launch_bounds__(SfbOwnerCfg<L>::NT, 1) sfb_owner_kernel(const __grid_constant__ SfbOwnerParams op) {
    extern __shared__ float2 sfb_ring_all[];
    constexpr int NT = SfbOwnerCfg<L>::NT;
    const SfbParams& p = op.p;
    const int tid = threadIdx.x;
    const int plane = blockIdx.x / op.parts;
    const int part = blockIdx.x - plane * op.parts;
    float* const y_area = reinterpret_cast<float*>(sfb_ring_all) + op.ring_floats;
    pdl_trigger();   // see afb_owner_kernel
    pdl_wait();
#pragma unroll 1
    for (int c = 0; c < p.J; ++c) {
        SfbLevel lv = p.lv[c];
        const OwnerLevel& ol = op.ol[c];
        SfbOwnRows own;
        own.n0 = ol.c0[part];
        own.n1 = ol.c1[part];
        own.low_s = 0;
        own.low_row0 = 0;
        const bool smem_low = c > 0;
        if (smem_low) {   // low-pass input = the previous position's output rows in shared memory
            const OwnerLevel& pv = op.ol[c - 1];
            float* buf = y_area + pv.buf_off;
            own.low_s = (unsigned)__cvta_generic_to_shared(buf);
            own.low_row0 = pv.c0[part];
            lv.low = buf - (long long)pv.c0[part] * pv.pitch;   // generic pointer for the border items
            lv.low_ps = 0;
            lv.low_rs = pv.pitch;
        }
        if (c + 1 < p.J) {   // the output stays on chip
            lv.y = y_area + ol.buf_off - (long long)own.n0 * ol.pitch;
            lv.y_ps = 0;
            lv.y_rs = ol.pitch;
        }
        lv.Rp = ol.R;
        const int npairs = ((lv.offH + own.n1 - 1) >> 1) + 1 - ((own.n0 + lv.offH) >> 1);
        own.itemsA = ((npairs + lv.Rp - 1) / lv.Rp) * lv.ntA;
        for (int base = 0; base < own.itemsA; base += NT) {
            __syncwarp();   // the warp's ring is reused from pass to pass
            const int it = base + tid;
            if (smem_low) {
                if (S2V == 0) sfb_ring_cta<L, 0, 0, true, true>(p, lv, plane, it, sfb_ring_all, nullptr, 0u, own);
                else if (lv.vec2) sfb_ring_cta<L, 2, S2V, true, true>(p, lv, plane, it, sfb_ring_all, nullptr, 0u, own);
                else sfb_ring_cta<L, 1, 0, true, true>(p, lv, plane, it, sfb_ring_all, nullptr, 0u, own);
            } else {
                if (S2V == 0) sfb_ring_cta<L, 0, 0, true, false>(p, lv, plane, it, sfb_ring_all, nullptr, 0u, own);
                else if (lv.vec2) sfb_ring_cta<L, 2, S2V, true, false>(p, lv, plane, it, sfb_ring_all, nullptr, 0u, own);
                else sfb_ring_cta<L, 1, 0, true, false>(p, lv, plane, it, sfb_ring_all, nullptr, 0u, own);
            }
        }
        // border columns go to the last threads first: warps with no or short segments start them early
        const int itemsB = (own.n1 - own.n0) * (lv.nA0 + lv.out_w - lv.nA1);
        for (int it = NT - 1 - tid; it < itemsB; it += NT)
            sfb_border_item<L, true>(p, lv, plane, it, true, nullptr, 0u, own);
        __syncthreads();   // this position's output is complete before the next one reads it
    }
}

bool sfb_stream_supported(const SfbParams& p, int L) {
    if (L < 2 || L > 16 || (L & 1)) return false;
    const bool per = p.periodic != 0;
    for (int j = 0; j < p.J; ++j)
        if (p.lv[j].offW != sfb_off(L, per) || p.lv[j].offH != sfb_off(L, per)) return false;
    return true;
}

// interior / border split of the output columns of a level and the staging geometry (stream and owner kernels)
template <int L, bool PER>
static void sfb_stream_columns(SfbLevel& lv) {
    constexpr int S2V = sfb_shift2(L, PER);
    using CV = SfbStreamCfg<L, S2V>;
    using C1 = SfbStreamCfg<L, 0>;
    lv.vec2 = (!(lv.low_rs & 1) && !(lv.low_ps & 1) && aligned_to(lv.low, 8) &&
               (!lv.highs || (!(lv.w & 1) && aligned_to(lv.highs, 8)))) ? 1 : 0;
    const int ncf = lv.vec2 ? CV::NCF : C1::NCF;
    lv.n0_off = sfb_n0_off(L, PER);
    lv.kb_off = lv.vec2 ? sfb_ks_off(L, PER) - S2V : sfb_ks_off(L, PER);
    lv.m_lo = lv.offH >> 1;
    // interior threads: window [kb, kb+ncf) inside [0, w) and outputs n0 .. n0+3 inside [0, out_w)
    int t0 = lv.kb_off < 0 ? (-lv.kb_off + 1) / 2 : 0;
    if (lv.n0_off < 0 && t0 < 1) t0 = 1;
    int t1 = lv.w - ncf - lv.kb_off >= 0 ? (lv.w - ncf - lv.kb_off) / 2 + 1 : 0;
    const int t1o = lv.out_w - 4 - lv.n0_off >= 0 ? (lv.out_w - 4 - lv.n0_off) / 4 + 1 : 0;
    t1 = std::min(t1, t1o);
    lv.tA0 = t0;
    lv.ntA = t1 - t0;
    if (lv.ntA < kSfbMinThreads) lv.ntA = 0;   // too narrow for the ring: every column takes the border path
    lv.nA0 = lv.ntA > 0 ? 4 * lv.tA0 + lv.n0_off : lv.out_w;
    lv.nA1 = lv.ntA > 0 ? 4 * (lv.tA0 + lv.ntA) + lv.n0_off : lv.out_w;
    lv.y_vec = 1;
    if (lv.n0_off == 0 && !(lv.y_rs & 1) && !(lv.y_ps & 1) && aligned_to(lv.y, 8)) lv.y_vec = 2;
    if (lv.y_vec == 2 && !(lv.y_rs & 3) && !(lv.y_ps & 3) && aligned_to(lv.y, 16)) lv.y_vec = 4;
}

template <int L, bool PER>
static bool sfb_owner_plan_t(const SfbParams& p, int sms, bool force, SfbOwnerParams& op) {
    constexpr int NT = SfbOwnerCfg<L>::NT;
    constexpr int H2 = L / 2;
    const int J = p.J;
    if (J < 2) return false;
    int parts = std::min(kMaxParts, std::max(1, sms / p.planes));
    if (PER) parts = 1;   // the coefficient rows wrap around: a part would need rows from the far end
    parts = std::min(parts, p.lv[J - 1].out_h);
    // one CTA per SM: a short last wave wastes up to half of the time (few CTAs are fine: small batches are
    // latency-bound either way, and measured faster here than as ticketed chains, profiles/r01_smallbatch.log)
    if (!force && short_last_wave((long long)p.planes * parts, sms)) return false;
    op.p = p;
    op.parts = parts;
    // ring of the staging variants this launch can use (64-bit copies with the mode's shift, or 32-bit copies)
    constexpr size_t ring128 = std::max(SfbStreamCfg<L, sfb_shift2(L, PER)>::smem, SfbStreamCfg<L, 0>::smem);
    op.ring_floats = (int)(ring128 / kStreamNT * NT / 4);
    // rows: the last position's output rows are split evenly over the parts; every earlier position computes the
    // rows the next one reads as low-pass coefficients
    for (int q = 0; q < parts; ++q) {
        op.ol[J - 1].c0[q] = (int)((long long)p.lv[J - 1].out_h * q / parts);
        op.ol[J - 1].c1[q] = (int)((long long)p.lv[J - 1].out_h * (q + 1) / parts);
        for (int c = J - 2; c >= 0; --c) {
            const SfbLevel& nx = p.lv[c + 1];
            int lo = ((op.ol[c + 1].c0[q] + nx.offH) >> 1) - (H2 - 1);
            int hi = ((op.ol[c + 1].c1[q] - 1 + nx.offH) >> 1) + 1;
            if (PER) {
                lo = 0;
                hi = nx.h;
            }
            lo = std::max(lo, 0);
            hi = std::min(hi, nx.h);
            if (hi <= lo) {   // nothing of this output is read (degenerate crop): keep one row so that sizes stay positive
                lo = std::min(lo, nx.h - 1);
                lo = std::max(lo, 0);
                hi = lo + 1;
            }
            op.ol[c].c0[q] = lo;
            op.ol[c].c1[q] = hi;
        }
    }
    size_t floats = 0;
    for (int c = 0; c < J; ++c) {
        SfbLevel& lv = op.p.lv[c];
        OwnerLevel& ol = op.ol[c];
        int rows = 0;
        for (int q = 0; q < parts; ++q) {
            rows = std::max(rows, ol.c1[q] - ol.c0[q]);
            ol.h0[q] = ol.c0[q];
            ol.h1[q] = ol.c1[q];
        }
        ol.map_off = 0;
        if (c + 1 < J) {   // output image in shared memory: 16-byte aligned rows
            ol.pitch = (lv.out_w + 3) / 4 * 4;
            ol.buf_off = (int)floats;
            floats += (size_t)rows * ol.pitch;
            lv.y_rs = ol.pitch;
            lv.y_ps = 0;
        } else {
            ol.pitch = 0;
            ol.buf_off = 0;
        }
        if (c > 0) {       // low-pass input = that image: even pitch, aligned base
            lv.low_rs = op.ol[c - 1].pitch;
            lv.low_ps = 0;
        }
        // geometry with the shared-memory strides; the alignment tests on lv.low / lv.y must see aligned pointers
        const float* low_keep = lv.low;
        float* y_keep = lv.y;
        if (c > 0) lv.low = nullptr;
        if (c + 1 < J) lv.y = nullptr;
        sfb_stream_columns<L, PER>(lv);
        lv.low = low_keep;
        lv.y = y_keep;
        const int npairs = ((lv.offH + rows - 1) >> 1) + 2;   // upper bound over the parts' row offsets
        const int ntA = std::max(1, lv.ntA);
        int Rp = std::max(std::max(2, H2 - 1), ceil_div(npairs, std::max(1, NT / ntA)));
        // one pass of somewhat longer segments beats a second, mostly empty pass; far longer ones do not
        if (Rp > 2 * std::max(16, 4 * (H2 - 1))) Rp = std::max(16, 4 * (H2 - 1));
        ol.R = std::max(1, Rp);
    }
    op.y_floats = (int)floats;
    return ((size_t)op.ring_floats + floats) * 4 <= kMaxDynSmem;
}

template <int L, bool PER>
static int launch_sfb_owner_t(const SfbOwnerParams& op, cudaStream_t st) {
    constexpr int NT = SfbOwnerCfg<L>::NT;
    constexpr int S2V = sfb_shift2(L, PER);
    if (const cudaError_t e = allow_max_dyn_smem<sfb_owner_kernel<L, S2V>>()) return set_last_cuda_error(e);
    const size_t smem = ((size_t)op.ring_floats + op.y_floats) * 4;
    sfb_register_bounds(op.p, st);
    const cudaError_t le = launch_pdl(sfb_owner_kernel<L, S2V>, (unsigned)(op.p.planes * op.parts), NT, smem, st, op);
    note_launch("sfb_owner_kernel");
    const cudaError_t e = le != cudaSuccess ? le : cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

bool sfb_owner_plan(const SfbParams& p, int L, int sms, bool force, SfbOwnerParams& op) {
    if (!sfb_stream_supported(p, L)) return false;
#define X(LL) return p.periodic ? sfb_owner_plan_t<LL, true>(p, sms, force, op) : sfb_owner_plan_t<LL, false>(p, sms, force, op)
    B200W_FOR_EACH_L(X)
#undef X
    return false;
}

int launch_sfb_owner(const SfbOwnerParams& op, int L, cudaStream_t st) {
#define X(LL) return op.p.periodic ? launch_sfb_owner_t<LL, true>(op, st) : launch_sfb_owner_t<LL, false>(op, st)
    B200W_FOR_EACH_L(X)
#undef X
    return B200W_ERR_BAD_TAPS;
}

template <int L, bool PER>
static int launch_sfb_stream_t(SfbParams& p, int sms, cudaStream_t st) {
    constexpr int H2 = L / 2;
    constexpr int S2V = sfb_shift2(L, PER);
    using CV = SfbStreamCfg<L, S2V>;
    using C1 = SfbStreamCfg<L, 0>;
    // segments of ~16 output row pairs (see the analysis launcher for the rationale); the dependent levels of a
    // chain -- every level but the last, finest one -- shrink until they fill the resident CTA slots
    const int rpref = std::max(16, 4 * (H2 - 1));
    const long long slots = (long long)sms * CV::MINB;
    long long base = 0;
    for (int j = 0; j < p.J; ++j) {
        SfbLevel& lv = p.lv[j];
        sfb_stream_columns<L, PER>(lv);
        const int npairs = ((lv.offH + lv.out_h - 1) >> 1) + 1 - lv.m_lo;
        int Rp = rpref;
        if (j + 1 < p.J) {
            const int rmin = std::max(2, H2 - 1);
            while (Rp > rmin && (long long)p.planes * ceil_div(ceil_div(npairs, Rp) * std::max(lv.ntA, 1), kStreamNT) < slots)
                Rp = std::max(rmin, Rp - 2);
        }
        if (Rp > npairs) Rp = npairs;
        lv.Rp = Rp;
        lv.itemsA = ceil_div(npairs, Rp) * lv.ntA;
        lv.cppA = ceil_div(lv.itemsA, kStreamNT);
        lv.itemsB = lv.out_h * (lv.nA0 + lv.out_w - lv.nA1);
        lv.cpp = lv.cppA + ceil_div(lv.itemsB, kStreamNT);
        lv.cta_base = base;
        base += (long long)lv.cpp * p.planes;
    }
    p.total = base;
    if (base > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    if (p.J > 1) {
        const int rc = zero_sync_words(p.ticket, (size_t)p.J * p.planes + 1, st);
        if (rc) return rc;
    }
    sfb_register_bounds(p, st);
    sfb_stream_kernel<L, S2V><<<(unsigned)base, kStreamNT, SfbSmem<L>::value, st>>>(p);
    note_launch("sfb_stream_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

template <int L>
static int launch_sfb_stream_l(SfbParams& p, int sms, cudaStream_t st) {
    if (p.periodic) return launch_sfb_stream_t<L, true>(p, sms, st);
    return launch_sfb_stream_t<L, false>(p, sms, st);
}

int launch_sfb_stream(SfbParams& p, int L, int sms, cudaStream_t st) {
#define X(LL) return launch_sfb_stream_l<LL>(p, sms, st)
    B200W_FOR_EACH_L(X)
#undef X
    return B200W_ERR_BAD_TAPS;
}

}  // namespace b200w
