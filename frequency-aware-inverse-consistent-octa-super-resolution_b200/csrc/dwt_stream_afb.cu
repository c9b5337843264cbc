// Analysis filter bank, streaming register-blocked kernel (every row alignment; the fast path of the templated taps).
//
// Replaces afb1d(dim=3) + afb1d(dim=2) + reshape + 2x .contiguous() of AFB2D.forward
// (pw/dwt/lowlevel.py:336-347, 91-172) -- and the J-level loop around it (pw/dwt/transform2d.py:66-74).
//
// A thread owns ONE PAIR of adjacent output columns and marches down R output rows of one image plane:
//   * row pass in registers: per input row the 4*NV floats its two outputs need give lo/hi for both columns,
//     4L FMAs with the taps as constant-bank operands,
//   * column pass "accumulate forward": each pair of input rows is scattered into the L/2 output rows it
//     contributes to (8 accumulators each); the oldest one is complete, is stored with 64-bit coalesced stores
//     (LL into `low`, LH/HL/HH straight into `highs[:, :, 0..2]`) and its registers are recycled.
// ~2L FMAs + a handful of memory instructions per input pixel, no block-wide barriers.  The loop is unrolled by
// L/2 row pairs so that the accumulator ring has static register names.
//
// Input staging.  Column pairs whose window lies inside the image ("interior": all but 2..8 per row) are served by
// a per-WARP ring in shared memory: every lane cp.async-copies its own 16 bytes of each input row (a warp = 512
// contiguous bytes per row; the last lane of a run adds the NV-1 trailing float4), D row pairs deep, so ~D KB per
// warp are in flight without holding registers; a lane then reads its window (own float4 + the neighbours')
// with NV 128-bit shared loads.  Only __syncwarp is needed.  Rows outside the image are remapped per row
// (symmetric / reflect / periodic / periodization) or cleared with shared stores.
// The window starts at a multiple of 4 columns of the row, so the 16 bytes a lane copies are 16-byte aligned in
// global memory exactly when the rows are (V = 4: one copy); for other rows (odd widths, strided views) the same
// 16 bytes are copied as four 4-byte cp.async (V = 1).  Ring, window reads and arithmetic do not depend on V.
// The few border columns of each row run in separate CTAs, one thread per output position, through the row /
// column maps of the padding mode.
// Segments overlap by L-2 input rows (re-read through L2).
#include <algorithm>
#include <cmath>
#include "dwt_levels.cuh"

namespace b200w {

constexpr int afb_off(int L, bool per) { return per ? L - 1 - L / 2 : L - 2; }
// the first loaded column is 4*cp - (off + S): S pads the window start down to a multiple of 4
constexpr int afb_shift(int L, bool per) { return (4 - afb_off(L, per) % 4) % 4; }

// ring geometry: per warp, D stages of one input row pair; a row holds the 32 lanes' own float4 plus NV-1 extra
// float4 for each run of lanes that sits on one image row (a warp may straddle up to kMaxRuns segment rows)
constexpr int kMaxRuns = 5;
constexpr int kMinColPairs = 8;   // interior pairs per row needed for the ring path (=> at most kMaxRuns runs)
template <int L, int S>
struct AfbStreamCfg {
    static constexpr int H2 = L / 2;
    static constexpr int NV = (S + L + 2 + 3) / 4;   // float4 per window
    static constexpr int NE = 4 * NV;
    static constexpr int RP = 32 + kMaxRuns * (NV - 1);   // float4 per ring row
    static constexpr int D = L <= 8 ? 6 : 4;         // ring depth (row pairs)
    static constexpr int STAGE = 2 * RP;             // float4 per stage
    // resident CTAs per SM the ring path is compiled for (caps the registers; the rare border path may spill)
    static constexpr int MINB = L <= 8 ? 5 : (L <= 12 ? 4 : 3);
    static constexpr size_t smem = sizeof(float4) * (size_t)(kStreamNT / 32) * D * STAGE;
    // Q adjacent column pairs per lane (owner kernel, short filters: Q = 2 amortises the per-row-pair overhead --
    // staging, addresses, loop control -- over twice the arithmetic): a lane stages Q float4 per input row
    // (a warp of Q = 2 lanes may straddle up to 9 rows of >= 4 lanes each)
    __host__ __device__ static constexpr int rp(int Q) { return 32 * Q + (Q == 1 ? kMaxRuns : 9) * (NV - 1); }
    __host__ __device__ static constexpr int depth(int Q) { return Q == 1 ? D : 4; }
    __host__ __device__ static constexpr int ring_float4_per_warp(int Q) { return depth(Q) * 2 * rp(Q); }
};

// source row of input row r: r itself inside the image, else the padding mode's map; -1 = zero row
__device__ __forceinline__ int afb_src_row(int r, int H, int Hreal, int mode) {
    if ((unsigned)r < (unsigned)Hreal) return r;
    const int sr = ext_index_far(r, H, mode);
    return sr >= Hreal ? -1 : sr;
}

// one pair of input rows: row pass for both, then scatter into the accumulator ring (ph = pair index mod L/2).
// The ring keeps each sub-band's two columns as one float2, so the column pass runs on the packed FFMA2: the two
// columns share the tap, which comes as a (t, t) pair from uniform registers.
// With kRotate the ring is kept in age order instead (slot 0 = oldest) and shifted by the caller after the store:
// L/2-1 register moves per row pair, but the loop needs no unrolling by L/2 -- for long filters the unrolled
// body would not fit the instruction cache.
template <int L, int S, int NE>
__device__ __forceinline__ void afb_pair_fma(const Taps& t, const float (&v)[2][NE], float2 (&acc)[L / 2][4], int ph) {
    constexpr int H2 = L / 2;
    constexpr bool kRotate = L >= 10;
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
        const int sl = kRotate ? H2 - 1 - u : (ph - u + H2) % H2;
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

// block until every CTA item of the previous level of this plane has been published (called by all threads,
// after their index arithmetic so that the set-up overlaps the wait)
__device__ __forceinline__ void chain_wait(const unsigned* ctr, unsigned need) {
    if (ctr != nullptr) {
        if (threadIdx.x == 0)
            while (ld_acquire_u32(ctr) < need) __nanosleep(20);
        __syncthreads();
    }
}

// rows of a level that an owner CTA works on (owner kernel only): it computes output rows [c0, c1) -- all of them
// feed its low-pass image in shared memory -- and stores the detail bands of rows [h0, h1) to global memory
struct OwnRows {
    int c0, c1, h0, h1;
    int itemsA;            // thread items of the interior class over [c0, c1)
    unsigned src_s;        // SMEM_SRC: shared address of the source image (row src_row0, column 0)
    int src_row0;
    // extension maps of the level in shared memory (the out-of-line index functions cost ~100 instructions per
    // call, and an owner CTA runs its border items itself instead of spreading them over the device):
    const int* rmap;       // rmap[r - (2*c0 - offH)] = source row of input row r, -1 = zero row
    const int* cmap;       // cmap[c + offW] = source column of input column c, -1 = zero
};

__device__ __forceinline__ float4 lds128(unsigned addr) {
    B200W_CHK_S(addr, 16);
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

// one 16-byte ring slot from global memory: a single 16-byte cp.async (V = 4, `src` 16-byte aligned) or four 4-byte
// ones (V = 1, `src` 4-byte aligned)
template <int V>
__device__ __forceinline__ void ring_copy16(unsigned dst, const float* src) {
    static_assert(V == 4 || V == 1, "ring copy width");
    if constexpr (V == 4) {
        cp_async<4>(dst, src);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) cp_async<1>(dst + 4u * i, src + i);
    }
}

// ---- interior column pairs: per-warp cp.async ring ---------------------------------------------------
// `it` = the thread's item (segment-major: segment * ncpA + interior column pair).  V = global copy width (above).
// OWNER: the rows come from `own` instead of the whole level; SMEM_SRC (owner kernel, dependent levels): the input
// image already lies in shared memory, so a lane reads its window straight from there and the ring is not used.
template <int L, int S, int V, bool OWNER = false, bool SMEM_SRC = false, int Q = 1>
__device__ __forceinline__ void afb_ring_cta(const AfbParams& p, const AfbLevel& lv, int plane, int it, float4* ring_all,
                                             const unsigned* wait_ctr, unsigned wait_need, const OwnRows& own) {
    using C = AfbStreamCfg<L, S>;
    constexpr int H2 = C::H2, NV = C::NV, NE = C::NE, D = C::depth(Q);
    constexpr int RP = C::rp(Q), STAGE = 2 * RP;
    constexpr int NVQ = NV + (Q - 1), NEQ = 4 * NVQ;   // float4 / floats of a lane's window (Q pairs)
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int itemsA = OWNER ? own.itemsA : lv.itemsA;
    const bool active = it < itemsA;
    const int ncpA = lv.ncpA;
    const int nq = Q == 1 ? ncpA : (ncpA + Q - 1) / Q;   // lanes per row
    const int itc = active ? it : itemsA - 1;        // inactive lanes shadow the last item (no copies, no stores)
    const int seg = itc / nq;
    const int cpl = itc - seg * nq;
    const int cp = lv.cp0A + Q * cpl;
    const bool second = Q == 2 && Q * cpl + 1 < ncpA;   // the lane's second column pair exists (odd pair counts)
    const int i0 = (OWNER ? own.c0 : 0) + seg * lv.R;   // first output row of the segment
    const int nout = min(lv.R, (OWNER ? own.c1 : lv.Ho) - i0);
    const int npairs = active ? nout + H2 - 1 : 0;   // input row pairs feeding them
    const int r0 = 2 * i0 - lv.offH;                 // first input row
    const int H = lv.H, Hreal = lv.Hreal, mode = p.mode;
    const int cb = 4 * cp - (lv.offW + S);           // first column of the window: >= 0, multiple of 4
    // position in the ring row: own float4 at slot lane + (NV-1)*run; the last lane of a run adds the NV-1 extras
    const int seg_first = __shfl_sync(0xffffffffu, seg, 0);
    const int slot = Q * lane + (NV - 1) * (seg - seg_first);
    const bool run_last = NV > 1 && active && (lane == 31 || cpl == nq - 1);
    // float4 the lane copies per row: its own Q (a missing second pair's float4 still belongs to the first pair's
    // window when NV > 1) and, at the end of a run, the rest of the last window
    const int ncopy = (Q == 2 && (second || NV > 1) ? 2 : 1);
    const int nextra = run_last ? (NV - 1) - (Q == 2 && !second ? 1 : 0) : 0;
    const long long rs = lv.x_rs;
    const unsigned rs_b = (unsigned)rs * 4u;                      // row stride in bytes (< 4 GB, checked by the host)
    const float* xcol = lv.x + (long long)plane * lv.x_ps + cb;   // column cb of row 0
    float4* ring = ring_all + (size_t)(tid >> 5) * D * STAGE;
    const unsigned ring_s = (unsigned)__cvta_generic_to_shared(ring) + (unsigned)slot * 16u;

    // stage one input row pair (pair index q of this lane's segment) into ring stage `st`.  Rows inside the image
    // take the plain cp.async (the zero-filling form costs three padding instructions each); zero rows are cleared
    // with shared stores.
    auto issue = [&](int q, int st) {
        // nothing is staged beyond this lane's segment: the lanes that would read those slots (same run, same
        // segment) are past their last pair too, and an idle lane must not touch slots that belong to others
        if (!SMEM_SRC && q < npairs) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int sr = OWNER ? own.rmap[2 * (i0 - own.c0) + 2 * q + e] : afb_src_row(r0 + 2 * q + e, H, Hreal, mode);
                const unsigned dst = ring_s + (unsigned)((st * 2 + e) * RP) * 16u;
                if (sr >= 0) {
                    const float* src = reinterpret_cast<const float*>(reinterpret_cast<const char*>(xcol) +
                                                                      (unsigned long long)(unsigned)sr * rs_b);
                    ring_copy16<V>(dst, src);
                    if (Q == 2 && ncopy == 2) ring_copy16<V>(dst + 16u, src + 4);
                    if (run_last) {
#pragma unroll
                        for (int k = 0; k < NV - 1; ++k)
                            if (k < nextra) ring_copy16<V>(dst + 16u * (ncopy + k), src + 4 * (ncopy + k));
                    }
                } else {
                    float4* d = ring + (st * 2 + e) * RP + slot;
                    B200W_CHK(d, 16 * (ncopy + nextra));
                    d[0] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (Q == 2 && ncopy == 2) d[1] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (run_last) {
#pragma unroll
                        for (int k = 0; k < NV - 1; ++k)
                            if (k < nextra) d[ncopy + k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
            }
        }
    };

    const int Wo = lv.Wo;
    const size_t band = (size_t)lv.Ho * Wo;
    // store switches of the level in one register (kept there: re-reading them from the parameter block inside the
    // loop costs an indexed constant load each)
    unsigned flags = (lv.low_vec2 ? 1u : 0u) | (lv.out_vec2 ? 2u : 0u) | (lv.st_low ? 4u : 0u) | (lv.st_hi ? 8u : 0u) |
                     ((lv.hi_scale != 1.f || lv.hi_shift != 0.f) ? 16u : 0u);
    asm volatile("" : "+r"(flags));
    const bool v2lo = flags & 1u, v2hi = flags & 2u, st_low = flags & 4u, st_hi = flags & 8u;
    const float2 hsc = make_float2(lv.hi_scale, lv.hi_scale), hsh = make_float2(lv.hi_shift, lv.hi_shift);
    const long long low_rs = lv.low_rs;
    float* q0 = lv.low + (long long)plane * lv.low_ps + (long long)i0 * low_rs + 2 * cp;   // only dereferenced if st_low
    float* q1 = lv.highs + (size_t)plane * 3 * band + (size_t)i0 * Wo + 2 * cp;            // ... if st_hi

    // warp-uniform trip count (lanes of a warp may sit in segments of different length)
    int npw = npairs;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) npw = max(npw, __shfl_xor_sync(0xffffffffu, npw, o));

    if (!OWNER) chain_wait(wait_ctr, wait_need);
    if (!SMEM_SRC) {
#pragma unroll 1
        for (int s = 0; s < D - 1; ++s) {
            issue(s, s);
            cp_async_commit();
        }
    }
    // SMEM_SRC: shared address of this lane's window in source row 0
    const unsigned win_s = SMEM_SRC ? own.src_s + (unsigned)(cb - own.src_row0 * (int)rs) * 4u : 0u;
    int orow = i0;         // OWNER: output row the next store belongs to
    float2 acc[Q][H2][4];   // per pair: ring of pending output rows: LL, LH, HL, HH, each (column 0, column 1)
    int st_r = 0, st_w = D - 1;
    constexpr bool kRotate = L >= 10;
    constexpr int UQ = kRotate ? 1 : H2;
    for (int qb = 0; qb < npw; qb += UQ) {
#pragma unroll
        for (int ph = 0; ph < UQ; ++ph) {
            const int q = qb + ph;
            if (q < npw) {   // warp-uniform
                if (!SMEM_SRC) {
                    cp_async_wait<D - 2>();   // this lane's copies of pair q have landed ...
                    __syncwarp();             // ... and everybody's; all lanes are done reading pair q-1
                    issue(q + D - 1, st_w);   // refill the stage pair q-1 was read from
                    cp_async_commit();
                    st_w = st_w + 1 == D ? 0 : st_w + 1;
                }
                {
                    float v[2][NEQ];
                    // a lane without a second pair reads one float4 less (it was not staged / may lie past the row)
                    const int nv = NVQ - (Q == 2 && !second ? 1 : 0);
                    if (SMEM_SRC) {
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int sr = q < npairs ? own.rmap[2 * (i0 - own.c0) + 2 * q + e] : -1;
                            const unsigned a = win_s + (unsigned)(max(sr, 0) * (int)rs) * 4u;
#pragma unroll
                            for (int k = 0; k < NVQ; ++k) {
                                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                                if (sr >= 0 && k < nv) t = lds128(a + 16u * k);
                                v[e][4 * k] = t.x; v[e][4 * k + 1] = t.y; v[e][4 * k + 2] = t.z; v[e][4 * k + 3] = t.w;
                            }
                        }
                    } else {
                        const float4* src = ring + (st_r * 2) * RP + slot;
#pragma unroll
                        for (int e = 0; e < 2; ++e)
#pragma unroll
                            for (int k = 0; k < NVQ; ++k) {
                                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                                if (Q == 1 || k < nv) { B200W_CHK(src + e * RP + k, 16); t = src[e * RP + k]; }
                                v[e][4 * k] = t.x; v[e][4 * k + 1] = t.y; v[e][4 * k + 2] = t.z; v[e][4 * k + 3] = t.w;
                            }
                    }
#pragma unroll
                    for (int u = 0; u < Q; ++u) {
                        float vu[2][NE];   // the pair's window: a register renaming, not a copy
#pragma unroll
                        for (int e = 0; e < 2; ++e)
#pragma unroll
                            for (int k = 0; k < NE; ++k) vu[e][k] = v[e][4 * u + k];
                        afb_pair_fma<L, S, NE>(p.t, vu, acc[u], ph);
                    }
                    // output row q - (H2-1) has now seen all its L input rows
                    if (q >= H2 - 1 && q < npairs) {
                        const bool hi_row = st_hi && (!OWNER || (orow >= own.h0 && orow < own.h1));
#pragma unroll
                        for (int u = 0; u < Q; ++u) {
                            if (u == 0 || second) {
                                const float2* s = acc[u][kRotate ? 0 : (ph + 1) % H2];
                                float* d0 = q0 + 2 * u;
                                float* d1 = q1 + 2 * u;
                                if (st_low) {
                                    B200W_CHK_A(d0, 8, v2lo ? 8 : 4);
                                    if (v2lo) {
                                        *reinterpret_cast<float2*>(d0) = s[0];
                                    } else {
                                        d0[0] = s[0].x; d0[1] = s[0].y;
                                    }
                                }
                                if (hi_row) {
                                    B200W_CHK(d1, 8); B200W_CHK(d1 + band, 8); B200W_CHK(d1 + 2 * band, 8);
                                    const float2 lh = ffma2(s[1], hsc, hsh), hl = ffma2(s[2], hsc, hsh), hh = ffma2(s[3], hsc, hsh);
                                    if (v2hi) {
                                        *reinterpret_cast<float2*>(d1) = lh;
                                        *reinterpret_cast<float2*>(d1 + band) = hl;
                                        *reinterpret_cast<float2*>(d1 + 2 * band) = hh;
                                    } else {
                                        d1[0] = lh.x; d1[band] = hl.x; d1[2 * band] = hh.x;
                                        d1[1] = lh.y; d1[band + 1] = hl.y; d1[2 * band + 1] = hh.y;
                                    }
                                }
                            }
                        }
                        q0 += low_rs;
                        q1 += Wo;
                        if (OWNER) ++orow;
                    }
                    if (kRotate) {
#pragma unroll
                        for (int u = 0; u < Q; ++u)
#pragma unroll
                            for (int k = 0; k + 1 < H2; ++k)
#pragma unroll
                                for (int i = 0; i < 4; ++i) acc[u][k][i] = acc[u][k + 1][i];
                    }
                }
                st_r = st_r + 1 == D ? 0 : st_r + 1;
            }
        }
    }
    if (!SMEM_SRC) cp_async_wait<0>();
}

// ---- border columns: one thread per output position -----------------------------------------------------
// The 2..8 column pairs per row whose window leaves the image are evaluated directly: thread = (output row,
// border column); its L x L input samples are independent loads through the row / column maps (one memory
// latency instead of a dependent march), at the price of recomputing the row pass L/2 times -- for < 3 % of
// the outputs.
template <int L, int S, bool OWNER = false>
__device__ __forceinline__ void afb_border_item(const AfbParams& p, const AfbLevel& lv, int plane, int it, bool active,
                                                const unsigned* wait_ctr, unsigned wait_need, const OwnRows& own) {
    if (!active) it = 0;                             // idle threads shadow item 0 (they only take part in the wait)
    const int ncB = lv.Wo - 2 * lv.ncpA;             // border columns per output row
    const int ib = it / ncB;
    const int i = (OWNER ? own.c0 : 0) + ib;
    const int e0 = it - ib * ncB;
    const int k = e0 < 2 * lv.cp0A ? e0 : e0 + 2 * lv.ncpA;   // left border columns, then right border columns
    const int mode = p.mode;
    int cidx[L];
#pragma unroll
    for (int j = 0; j < L; ++j) {
        int c = 2 * k + j - lv.offW;
        if (OWNER) {
            c = own.cmap[2 * k + j];
        } else if ((unsigned)c >= (unsigned)lv.Wreal) {
            c = ext_index_far(c, lv.W, mode);
            if (c >= lv.Wreal) c = -1;
        }
        cidx[j] = c;
    }
    int srow[L];
#pragma unroll
    for (int jh = 0; jh < L; ++jh)
        srow[jh] = OWNER ? own.rmap[2 * ib + jh] : afb_src_row(2 * i + jh - lv.offH, lv.H, lv.Hreal, mode);
    if (!OWNER) chain_wait(wait_ctr, wait_need);     // index arithmetic above overlaps the wait
    if (!active) return;
    const float* xp = lv.x + (long long)plane * lv.x_ps;
    // all L x L samples are loaded before any arithmetic (clamped address + select instead of branches), so
    // the thread pays one memory round trip; rows are done in chunks of <= 6 to bound the registers
    float ll = 0.f, lh = 0.f, hl = 0.f, hh = 0.f;
    constexpr int CH = L < 6 ? L : 6;
#pragma unroll
    for (int j0 = 0; j0 < L; j0 += CH) {
        float v[CH][L];
        bool rok[CH];
#pragma unroll
        for (int jj = 0; jj < CH; ++jj) {
            const int jh = j0 + jj;
            const int sr = jh < L ? srow[jh < L ? jh : 0] : -1;
            rok[jj] = sr >= 0;
            // a zero row is read from a row that exists (and discarded): row 0 of an owner CTA's shared-memory image
            // would lie before the buffer
            const float* rowp = xp + (long long)max(sr, OWNER ? own.src_row0 : 0) * lv.x_rs;
#pragma unroll
            for (int j = 0; j < L; ++j) { B200W_CHK(rowp + max(cidx[j], 0), 4); v[jj][j] = rowp[max(cidx[j], 0)]; }
        }
#pragma unroll
        for (int jj = 0; jj < CH; ++jj) {
            const int jh = j0 + jj;
            if (jh < L) {
                float lo = 0.f, hi = 0.f;
#pragma unroll
                for (int j = 0; j < L; ++j) {
                    const float x = (rok[jj] && cidx[j] >= 0) ? v[jj][j] : 0.f;
                    lo = fmaf(p.t.w_lo[j], x, lo);
                    hi = fmaf(p.t.w_hi[j], x, hi);
                }
                ll = fmaf(p.t.h_lo[jh], lo, ll);
                lh = fmaf(p.t.h_hi[jh], lo, lh);
                hl = fmaf(p.t.h_lo[jh], hi, hl);
                hh = fmaf(p.t.h_hi[jh], hi, hh);
            }
        }
    }
    const size_t band = (size_t)lv.Ho * lv.Wo;
    const size_t o = (size_t)i * lv.Wo + k;
    if (lv.st_low) {
        B200W_CHK(lv.low + (long long)plane * lv.low_ps + (long long)i * lv.low_rs + k, 4);
        lv.low[(long long)plane * lv.low_ps + (long long)i * lv.low_rs + k] = ll;
    }
    if (lv.st_hi && (!OWNER || (i >= own.h0 && i < own.h1))) {
        float* hip = lv.highs + (size_t)plane * 3 * band + o;
        B200W_CHK(hip, 4); B200W_CHK(hip + band, 4); B200W_CHK(hip + 2 * band, 4);
        hip[0] = fmaf(lh, lv.hi_scale, lv.hi_shift);
        hip[band] = fmaf(hl, lv.hi_scale, lv.hi_shift);
        hip[2 * band] = fmaf(hh, lv.hi_scale, lv.hi_shift);
    }
}

template <int L, int S, int V>
__global__ void __launch_bounds__(kStreamNT, AfbStreamCfg<L, S>::MINB) afb_stream_kernel(const __grid_constant__ AfbParams p) {
    extern __shared__ float4 ring_all[];
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
    const AfbLevel& lv = p.lv[level];
    const unsigned local = item - (unsigned)lv.cta_base;
    const int plane = (int)(local / (unsigned)lv.cpp);
    const int cta = (int)(local - (unsigned)plane * (unsigned)lv.cpp);
    // the previous level of this plane must be complete before its low-pass image is read
    const unsigned* wait_ctr = level > 0 ? p.done + (size_t)(level - 1) * p.planes + plane : nullptr;
    const unsigned wait_need = level > 0 ? (unsigned)p.lv[level - 1].cpp : 0u;
    const OwnRows none{};
    if (cta < lv.cppA) {
        afb_ring_cta<L, S, V>(p, lv, plane, cta * kStreamNT + tid, ring_all, wait_ctr, wait_need, none);
    } else {
        const int it = (cta - lv.cppA) * kStreamNT + tid;
        afb_border_item<L, S>(p, lv, plane, it, it < lv.itemsB, wait_ctr, wait_need, none);
    }
    if (level + 1 < p.J) {
        __syncthreads();
        if (tid == 0) signal_done(p.done + (size_t)level * p.planes + plane);
    }
}

// ---- owner kernel: every level of one (plane, part) in one CTA ------------------------------------------------
// The first level streams from global memory through the same per-warp rings as above; its low-pass rows land in
// shared memory, where the next level reads its windows directly (SMEM_SRC), and so on.  No tickets, no counters:
// the only synchronisation is one block barrier per level.
template <int L>
struct AfbOwnerCfg {
    // one CTA per SM; long filters need more than 128 registers per thread
    static constexpr int NT = L <= 8 ? kOwnerNT : 256;
    // column pairs per lane: two for the short filters (their accumulators fit the register budget twice)
    static constexpr int Q = 1;
};

template <int L, int S>
__global__ void __launch_bounds__(AfbOwnerCfg<L>::NT, 1) afb_owner_kernel(const __grid_constant__ AfbOwnerParams op) {
    extern __shared__ float4 ring_all[];
    constexpr int NT = AfbOwnerCfg<L>::NT, Q = AfbOwnerCfg<L>::Q;
    const AfbParams& p = op.p;
    const int tid = threadIdx.x;
    const int plane = blockIdx.x / op.parts;
    const int part = blockIdx.x - plane * op.parts;
    pdl_trigger();   // the next kernel in the stream may be scheduled as SMs free up (it waits before touching memory)
    int* const maps = reinterpret_cast<int*>(reinterpret_cast<float*>(ring_all) + op.ring_floats);
    float* const ll_area = reinterpret_cast<float*>(maps) + op.map_ints;
    // extension maps of every level, built once: input rows 2*c0 - offH + [0, 2*nrows + L) and input columns
    // -offW + [0, 2*Wo + L) of level j at maps + map_off[j]
#pragma unroll 1
    for (int j = 0; j < p.J; ++j) {
        const AfbLevel& lv = p.lv[j];
        const OwnerLevel& ol = op.ol[j];
        const int c0 = ol.c0[part];
        const int nr = 2 * (ol.c1[part] - c0) + L, nc = 2 * lv.Wo + L;
        int* const m_out = maps + ol.map_off;
        for (int e = tid; e < nr + nc; e += NT) {
            const bool row = e < nr;
            const int s = row ? 2 * c0 - lv.offH + e : e - nr - lv.offW;
            const int real = row ? lv.Hreal : lv.Wreal;
            int m = s;
            if ((unsigned)s >= (unsigned)real) {
                m = ext_index_far(s, row ? lv.H : lv.W, p.mode);
                if (m >= real) m = -1;
            }
            m_out[e] = m;
        }
    }
    pdl_wait();      // everything above used only the parameter block; from here on global memory is touched
    __syncthreads();
#pragma unroll 1
    for (int j = 0; j < p.J; ++j) {
        AfbLevel lv = p.lv[j];
        const OwnerLevel& ol = op.ol[j];
        OwnRows own;
        own.c0 = ol.c0[part]; own.c1 = ol.c1[part]; own.h0 = ol.h0[part]; own.h1 = ol.h1[part];
        own.src_s = 0; own.src_row0 = 0;
        const bool smem_src = j > 0;
        if (smem_src) {   // input = the previous level's low-pass rows [c0', c1') in shared memory
            const OwnerLevel& pv = op.ol[j - 1];
            float* buf = ll_area + pv.buf_off;
            own.src_s = (unsigned)__cvta_generic_to_shared(buf);
            own.src_row0 = pv.c0[part];
            lv.x = buf - (long long)pv.c0[part] * pv.pitch;   // generic pointer for the border items
            lv.x_ps = 0;
            lv.x_rs = pv.pitch;
        }
        if (j + 1 < p.J) {   // low-pass output stays on chip
            lv.low = ll_area + ol.buf_off - (long long)own.c0 * ol.pitch;
            lv.low_ps = 0;
            lv.low_rs = ol.pitch;
            lv.low_vec2 = 1;
            lv.st_low = 1;
        }
        lv.R = ol.R;
        const int nrows = own.c1 - own.c0;
        own.itemsA = ((nrows + lv.R - 1) / lv.R) * ((lv.ncpA + Q - 1) / Q);
        own.rmap = maps + ol.map_off;
        own.cmap = own.rmap + 2 * nrows + L;
        const int itemsB = nrows * (lv.Wo - 2 * lv.ncpA);
        const int padA = (own.itemsA + 31) & ~31;
        // When the interior segments leave warps free (the plan sizes them so), those warps evaluate the border
        // positions meanwhile; otherwise every thread does its interior items first and border items after, the
        // border positions going to the last threads first (warps with no or short segments start them early).
        const bool beside = itemsB > 0 && (NT - padA) * 4 >= itemsB;
        const int ntA = beside ? padA : NT;
        if (tid < ntA) {
            for (int base = 0; base < own.itemsA; base += ntA) {
                __syncwarp();   // the warp's ring is reused from pass to pass
                if (smem_src)
                    afb_ring_cta<L, S, 4, true, true, Q>(p, lv, plane, base + tid, ring_all, nullptr, 0u, own);
                else
                    afb_ring_cta<L, S, 4, true, false, Q>(p, lv, plane, base + tid, ring_all, nullptr, 0u, own);
            }
        }
        if (!beside || tid >= padA) {
            const int nb = beside ? NT - padA : NT;
            for (int it = beside ? tid - padA : NT - 1 - tid; it < itemsB; it += nb)
                afb_border_item<L, S, true>(p, lv, plane, it, true, nullptr, 0u, own);
        }
        __syncthreads();   // this level's low-pass rows are complete before the next level reads them
    }
}

bool afb_stream_supported(const AfbParams& p, int L) {
    if (L < 2 || L > 16 || (L & 1)) return false;
    const bool per = p.mode == B200W_MODE_PERIODIZATION;
    for (int j = 0; j < p.J; ++j) {
        const AfbLevel& lv = p.lv[j];
        if (lv.x_rs < 0 || lv.x_rs >= (1LL << 30)) return false;   // the ring addresses rows with a 32-bit byte stride
        if (lv.offW != afb_off(L, per) || lv.offH != afb_off(L, per)) return false;
    }
    return true;
}

// every level's input rows start 16-byte aligned: the ring may copy with 16-byte cp.async (V = 4).  Only level 0 can
// fail this; the intermediate low-pass images lie in the 256-byte aligned workspace with a pitch of 4 floats.
static bool afb_rows_16b(const AfbParams& p) {
    for (int j = 0; j < p.J; ++j) {
        const AfbLevel& lv = p.lv[j];
        if ((lv.x_rs & 3) || (lv.x_ps & 3) || !aligned_to(lv.x, 16)) return false;
    }
    return true;
}

// interior / border split of the output columns of a level (the same for the stream and the owner kernel)
template <int L, int S>
static void afb_stream_columns(AfbLevel& lv) {
    using C = AfbStreamCfg<L, S>;
    lv.ncp = ceil_div(lv.Wo, 2);
    // interior column pairs: window [4cp - (offW+S), +NE) inside [0, Wreal) and both output columns valid
    lv.cp0A = (lv.offW + S) / 4;
    int cpR = (lv.Wreal + lv.offW + S - C::NE) / 4 + 1;   // first pair whose window leaves the image
    if (lv.Wreal + lv.offW + S - C::NE < 0) cpR = 0;
    if (cpR > lv.Wo / 2) cpR = lv.Wo / 2;
    lv.ncpA = cpR - lv.cp0A;
    if (lv.ncpA < kMinColPairs) lv.ncpA = 0;              // too narrow for the ring: all columns take the border path
}

template <int L, int S>
static int launch_afb_stream_t(AfbParams& p, int sms, cudaStream_t st) {
    using C = AfbStreamCfg<L, S>;
    constexpr int H2 = L / 2;
    // Segments of ~16 output rows (longer for long filters, to amortise the L-2 warm-up rows): many short work
    // items balance better than one wave of long ones (measured, profiles/r01_sweep_rows.log).  A level that
    // cannot fill the resident CTA slots anyway is latency-bound (per-CTA set-up + one dependent row pair after
    // the other): it gets shorter segments, down to 2 rows for the small dependent levels of a chain.
    // rows per work item of the first level.  Every item re-reads L/2 - 1 row pairs of warm-up, which favours long items
    // for long filters; short filters have (almost) no warm-up and balance better with short items.  Measured at
    // 64 x 1024^2 (rows-per-item sweep, profiles/r02_notes.md): haar 6 / 16 rows = 81.5 / 85.8 us, db2 92.8 (8 rows:
    // 94.1) / 104.7 us; db3 gains 2 % at J = 1 with 10 rows but loses 1-3 % in chains (J >= 2), so it keeps 16 like
    // db4 and longer, where 16+ rows are best.
    const int rpref = H2 == 1 ? 6 : (H2 == 2 ? 8 : std::max(16, 4 * (H2 - 1)));
    const long long slots = (long long)sms * C::MINB;
    long long base = 0;
    for (int j = 0; j < p.J; ++j) {
        AfbLevel& lv = p.lv[j];
        afb_stream_columns<L, S>(lv);
        // the first level keeps the preferred length (measured best even when it leaves CTA slots empty; an
        // SM-balancing search over R was tried and was not better, profiles/r01_notes.md); the dependent levels of a
        // chain shrink until they fill the resident slots
        int R = rpref;
        if (j > 0) {
            const int rmin = std::max(2, H2 - 1);
            while (R > rmin && (long long)p.planes * ceil_div(ceil_div(lv.Ho, R) * std::max(lv.ncpA, 1), kStreamNT) < slots)
                R = std::max(rmin, R - 2);
        }
        if (R > lv.Ho) R = lv.Ho;
        lv.R = R;
        const int nseg = ceil_div(lv.Ho, R);
        lv.itemsA = nseg * lv.ncpA;
        lv.RB = 1;
        lv.itemsB = lv.Ho * (lv.Wo - 2 * lv.ncpA);   // border columns: one thread per output position
        lv.cppA = ceil_div(lv.itemsA, kStreamNT);
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
    afb_register_bounds(p, st);
    if (afb_rows_16b(p))
        afb_stream_kernel<L, S, 4><<<(unsigned)base, kStreamNT, C::smem, st>>>(p);
    else
        afb_stream_kernel<L, S, 1><<<(unsigned)base, kStreamNT, C::smem, st>>>(p);
    note_launch("afb_stream_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

template <int L>
static int launch_afb_stream_l(AfbParams& p, int sms, cudaStream_t st) {
    if (p.mode == B200W_MODE_PERIODIZATION) return launch_afb_stream_t<L, afb_shift(L, true)>(p, sms, st);
    return launch_afb_stream_t<L, afb_shift(L, false)>(p, sms, st);
}

// dynamic shared memory of the owner kernel: [rings | extension maps | low-pass images]
template <int L, int S>
static bool afb_owner_plan_t(const AfbParams& p, int sms, bool force, AfbOwnerParams& op) {
    using C = AfbStreamCfg<L, S>;
    constexpr int NT = AfbOwnerCfg<L>::NT, Q = AfbOwnerCfg<L>::Q;
    constexpr int H2 = L / 2;
    const int J = p.J;
    if (J < 2) return false;
    const bool wraps = p.mode == B200W_MODE_PERIODIZATION || p.mode == B200W_MODE_PERIODIC;
    int parts = std::min(kMaxParts, std::max(1, sms / p.planes));
    if (wraps) parts = 1;   // a part would need rows from the far end of the image
    parts = std::min(parts, p.lv[J - 1].Ho);
    // one CTA per SM: a short last wave wastes up to half of the time (few CTAs are fine: small batches are
    // latency-bound either way, and measured faster here than as ticketed chains, profiles/r01_smallbatch.log)
    if (!force && short_last_wave((long long)p.planes * parts, sms)) return false;
    op.p = p;
    op.parts = parts;
    op.ring_floats = (int)((size_t)(NT / 32) * C::ring_float4_per_warp(Q) * 4);
    // rows: every level's output rows are split evenly over the parts (what a part stores); a part computes those
    // plus whatever the next level's computed rows read through the row extension
    for (int j = 0; j < J; ++j) {
        afb_stream_columns<L, S>(op.p.lv[j]);
        for (int q = 0; q < parts; ++q) {
            op.ol[j].h0[q] = (int)((long long)p.lv[j].Ho * q / parts);
            op.ol[j].h1[q] = (int)((long long)p.lv[j].Ho * (q + 1) / parts);
        }
    }
    for (int q = 0; q < parts; ++q) {
        op.ol[J - 1].c0[q] = op.ol[J - 1].h0[q];
        op.ol[J - 1].c1[q] = op.ol[J - 1].h1[q];
        for (int j = J - 2; j >= 0; --j) {
            const AfbLevel& nx = p.lv[j + 1];   // reads this level's low-pass image
            int lo = op.ol[j].h0[q], hi = op.ol[j].h1[q];
            const int r_lo = 2 * op.ol[j + 1].c0[q] - nx.offH, r_hi = 2 * (op.ol[j + 1].c1[q] - 1) - nx.offH + L - 1;
            for (int r = r_lo; r <= r_hi; ++r) {
                int sr = r;
                if (r < 0 || r >= nx.Hreal) {
                    sr = ext_index(r, nx.H, p.mode);
                    if (sr < 0 || sr >= nx.Hreal) continue;   // zero row
                }
                lo = std::min(lo, sr);
                hi = std::max(hi, sr + 1);
            }
            op.ol[j].c0[q] = lo;
            op.ol[j].c1[q] = hi;
        }
    }
    // the low-pass images of every level but the last must fit next to the rings
    size_t floats = 0;
    for (int j = 0; j < J - 1; ++j) {
        int rows = 0;
        for (int q = 0; q < parts; ++q) rows = std::max(rows, op.ol[j].c1[q] - op.ol[j].c0[q]);
        op.ol[j].pitch = (p.lv[j].Wo + 3) / 4 * 4;
        op.ol[j].buf_off = (int)floats;
        floats += (size_t)rows * op.ol[j].pitch;
    }
    int map_ints = 0;
    for (int j = 0; j < J; ++j) {
        int rows = 0;
        for (int q = 0; q < parts; ++q) rows = std::max(rows, op.ol[j].c1[q] - op.ol[j].c0[q]);
        op.ol[j].map_off = map_ints;
        map_ints += 2 * rows + L + 2 * p.lv[j].Wo + L;
    }
    op.map_ints = (map_ints + 3) / 4 * 4;
    if (((size_t)op.ring_floats + op.map_ints + floats) * 4 > kMaxDynSmem) return false;
    for (int j = 0; j < J; ++j) {
        // segments sized so that one pass of the CTA's threads covers the part
        int rows = 0;
        for (int q = 0; q < parts; ++q) rows = std::max(rows, op.ol[j].c1[q] - op.ol[j].c0[q]);
        const int ncpA = std::max(1, (op.p.lv[j].ncpA + Q - 1) / Q);   // lanes per row
        const int rmin = std::max(2, H2 - 1);
        // some warps are kept free for the border positions (about four rounds of them), which then run
        // beside the interior segments instead of after them
        const int itemsB = rows * (p.lv[j].Wo - 2 * op.p.lv[j].ncpA);
        int spare = itemsB > 0 ? std::min(NT / 2, std::max(32, (ceil_div(itemsB, 4) + 31) & ~31)) : 0;
        if ((NT - spare) / ncpA < 1) spare = 0;
        const int rmax = std::max(16, 4 * (H2 - 1));
        int R = std::max(rmin, ceil_div(rows, std::max(1, (NT - spare) / ncpA)));
        if (R > rmax) {   // no room for spare warps: one class after the other
            R = std::max(rmin, ceil_div(rows, std::max(1, NT / ncpA)));
            // one pass of somewhat longer segments beats a second, mostly empty pass; far longer ones do not
            if (R > 2 * rmax) R = rmax;
        }
        op.ol[j].R = std::max(1, std::min(R, rows));
    }
    return true;
}

template <int L, int S>
static int launch_afb_owner_t(const AfbOwnerParams& op, cudaStream_t st) {
    constexpr int NT = AfbOwnerCfg<L>::NT;
    size_t floats = (size_t)op.ring_floats + op.map_ints;
    for (int j = 0; j < op.p.J - 1; ++j) {
        int rows = 0;
        for (int q = 0; q < op.parts; ++q) rows = std::max(rows, op.ol[j].c1[q] - op.ol[j].c0[q]);
        floats = std::max(floats, (size_t)op.ring_floats + op.map_ints + op.ol[j].buf_off + (size_t)rows * op.ol[j].pitch);
    }
    if (const cudaError_t e = allow_max_dyn_smem<afb_owner_kernel<L, S>>()) return set_last_cuda_error(e);
    afb_register_bounds(op.p, st);
    const cudaError_t le = launch_pdl(afb_owner_kernel<L, S>, (unsigned)(op.p.planes * op.parts), NT, floats * 4, st, op);
    note_launch("afb_owner_kernel");
    const cudaError_t e = le != cudaSuccess ? le : cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

bool afb_owner_plan(const AfbParams& p, int L, int sms, bool force, AfbOwnerParams& op) {
    // the owner kernel's ring is instantiated with 16-byte copies only
    if (!afb_stream_supported(p, L) || !afb_rows_16b(p)) return false;
    const bool per = p.mode == B200W_MODE_PERIODIZATION;
#define X(LL) return per ? afb_owner_plan_t<LL, afb_shift(LL, true)>(p, sms, force, op) \
                         : afb_owner_plan_t<LL, afb_shift(LL, false)>(p, sms, force, op)
    B200W_FOR_EACH_L(X)
#undef X
    return false;
}

int launch_afb_owner(const AfbOwnerParams& op, int L, cudaStream_t st) {
    const bool per = op.p.mode == B200W_MODE_PERIODIZATION;
#define X(LL) return per ? launch_afb_owner_t<LL, afb_shift(LL, true)>(op, st) \
                         : launch_afb_owner_t<LL, afb_shift(LL, false)>(op, st)
    B200W_FOR_EACH_L(X)
#undef X
    return B200W_ERR_BAD_TAPS;
}

int launch_afb_stream(AfbParams& p, int L, int sms, cudaStream_t st) {
#define X(LL) return launch_afb_stream_l<LL>(p, sms, st)
    B200W_FOR_EACH_L(X)
#undef X
    return B200W_ERR_BAD_TAPS;
}

}  // namespace b200w
