// Multi-level synthesis filter bank, TMA-staged owner kernel (chains of small planes; all padding modes but
// periodization, whose coefficient sequence wraps around).
//
// Replaces the J-level loop of DWTInverse.forward (pw/dwt/transform2d.py:134-148, incl. the 'unpad' crop) around
// SFB2D.forward (pw/dwt/lowlevel.py:671-680: six conv_transpose2d + three adds), and -- with the analysis taps and a
// crop -- the chain of AFB2D.backward calls (pw/dwt/lowlevel.py:349-365).
//
// "A-space": a = n + off (off = L-2), so output a uses taps of parity a&1 only:
//     y[a] = sum_u c[(a>>1) - u] * g[(a&1) + 2u],  u = 0 .. L/2-1            (the polyphase form of sfb1d)
// Every coefficient a valid output needs lies inside its sub-band, so there is no border case at all: whatever a lane
// reads beyond a row end only feeds outputs that are never stored.
//
// One CTA owns a horizontal part of one plane for every chain position (coarsest first).  The outputs of all positions
// but the last stay in shared memory and are the next position's low-pass input.  The detail rows come in through the
// copy engine as plain bulk copies (cp.async.bulk, SASS UBLKCP): the rows a part needs from one band are contiguous in
// global memory, so ONE copy per band fetches the 16-byte aligned superset of them and the data sits 0..3 floats into
// its (16-byte aligned) destination with the rows dense at pitch w -- any width, any row alignment (tensor-map copies
// need 16-byte aligned box starts and fault on the odd sub-band widths of the deeper levels).  For the small coarse
// positions all rows are fetched at kernel start; the last, finest position streams its rows through per-stream
// mbarrier rings fed by one service warp per stream.  Even widths read their windows with 64-bit shared loads, odd ones
// with 32-bit loads.
// A consumer lane owns FOUR adjacent output columns of one row stream and marches down its coefficient rows: W synthesis
// of the four sub-bands in registers (taps in registers), H synthesis scattered into a ring of L/2 pending output row
// pairs (packed FFMA2), completed pairs written with 128-bit stores.
#include <algorithm>
#include <type_traits>
#include "dwt_tma.cuh"

namespace b200w {

template <int L>
struct SfbT {
    static constexpr int H2 = L / 2;
    static constexpr int NS = (H2 + 2) / 2;          // float2 slots per window (H2 + 1 coefficients, rounded up to even)
    static constexpr int NCF = 2 * NS;
    static constexpr bool kRotate = L >= 10;
    static constexpr int SR = H2 == 3 ? 6 : 4;       // coefficient rows per ring stage: even, a multiple of L/2 (L <= 8)
    static constexpr int NTC = L <= 6 ? 416 : (L <= 8 ? 352 : 256);   // consumer threads
    static constexpr int MAXG = L <= 8 ? 5 : 4;      // row streams of the last position = service warps
    static constexpr int NT = NTC + 32 * MAXG;
    static constexpr bool kRegTaps = L <= 8;
};

__device__ __forceinline__ float2 lds64s(unsigned addr) {
    B200W_CHK_S(addr, 8);
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds32s(unsigned addr) {
    B200W_CHK_S(addr, 4);
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128s(unsigned addr, float4 v) {
    B200W_CHK_S(addr, 16);
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// the taps of one kernel as a register-resident copy (`zero` = 0.f read from shared memory keeps ptxas from
// rematerialising the constant loads inside the loop)
template <int L>
struct SfbRegTaps {
    float w_lo[L], w_hi[L];
    float2 h_lo2[L], h_hi2[L];
    __device__ __forceinline__ SfbRegTaps(const TapsT& t, float zero) {
#pragma unroll
        for (int i = 0; i < L; ++i) {
            w_lo[i] = t.w_lo[i] + zero; w_hi[i] = t.w_hi[i] + zero;
            h_lo2[i].x = h_lo2[i].y = t.h_lo2[i].x + zero;
            h_hi2[i].x = h_hi2[i].y = t.h_hi2[i].x + zero;
        }
    }
};
struct SfbConstTaps {
    const float (&w_lo)[kMaxTemplTaps], (&w_hi)[kMaxTemplTaps];
    const float2 (&h_lo2)[kMaxTemplTaps], (&h_hi2)[kMaxTemplTaps];
    __device__ __forceinline__ SfbConstTaps(const TapsT& tt, float) : w_lo(tt.w_lo), w_hi(tt.w_hi), h_lo2(tt.h_lo2), h_hi2(tt.h_hi2) {}
};

// one window of NCF coefficients at shared address a: 64-bit loads (V = 2, 8-byte aligned) or 32-bit loads
template <int NCF, int V>
__device__ __forceinline__ void sfbt_window(float (&c)[NCF], unsigned a) {
#pragma unroll
    for (int k = 0; k < NCF / 2; ++k) {
        if (V == 2) {
            const float2 v = lds64s(a + 8u * k);
            c[2 * k] = v.x; c[2 * k + 1] = v.y;
        } else {
            c[2 * k] = lds32s(a + 8u * k);
            c[2 * k + 1] = lds32s(a + 8u * k + 4u);
        }
    }
}

// one coefficient row: the four sub-band windows at shared addresses aLL / aH0..2, W synthesis, then H synthesis into
// the accumulator ring (ph = row index mod L/2)
template <int L, int VL, int VH, class T>
__device__ __forceinline__ void sfbt_row(const T& t, unsigned aLL, unsigned aH0, unsigned aH1, unsigned aH2,
                                         float2 (&acc)[L / 2][4], int ph) {
    using C = SfbT<L>;
    constexpr int H2 = C::H2, NCF = C::NCF;
    float c[4][NCF];
    sfbt_window<NCF, VL>(c[0], aLL);
    sfbt_window<NCF, VH>(c[1], aH0);
    sfbt_window<NCF, VH>(c[2], aH1);
    sfbt_window<NCF, VH>(c[3], aH2);
    // W synthesis: lo = h_lo branch (LL, HL), hi = h_hi branch (LH, HH); output e = 2*qo + par of the lane's four columns
    float lo[4], hi[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int qo = e >> 1, par = e & 1;
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int u = 0; u < H2; ++u) {
            const int kl = qo + H2 - 1 - u;
            a = fmaf(c[0][kl], t.w_lo[par + 2 * u], a);
            a = fmaf(c[2][kl], t.w_hi[par + 2 * u], a);
            b = fmaf(c[1][kl], t.w_lo[par + 2 * u], b);
            b = fmaf(c[3][kl], t.w_hi[par + 2 * u], b);
        }
        lo[e] = a;
        hi[e] = b;
    }
    // H synthesis: this row carries taps (2u, 2u+1) of output row pair q - (H2-1) + u
    const float2 lo01 = make_float2(lo[0], lo[1]), lo23 = make_float2(lo[2], lo[3]);
    const float2 hi01 = make_float2(hi[0], hi[1]), hi23 = make_float2(hi[2], hi[3]);
#pragma unroll
    for (int u = H2 - 1; u >= 0; --u) {
        const int sl = C::kRotate ? u : (ph + u + 1) % H2;
        const float2 a0 = t.h_lo2[2 * u], b0 = t.h_hi2[2 * u];
        const float2 a1 = t.h_lo2[2 * u + 1], b1 = t.h_hi2[2 * u + 1];
        float2* s = acc[sl];   // [0..1] even output row (columns 0-1, 2-3), [2..3] odd output row
        if (u == H2 - 1) {     // first contribution to that pair
            s[0] = fmul2(lo01, a0); s[1] = fmul2(lo23, a0);
            s[2] = fmul2(lo01, a1); s[3] = fmul2(lo23, a1);
        } else {
            s[0] = ffma2(lo01, a0, s[0]); s[1] = ffma2(lo23, a0, s[1]);
            s[2] = ffma2(lo01, a1, s[2]); s[3] = ffma2(lo23, a1, s[3]);
        }
        s[0] = ffma2(hi01, b0, s[0]); s[1] = ffma2(hi23, b0, s[1]);
        s[2] = ffma2(hi01, b1, s[2]); s[3] = ffma2(hi23, b1, s[3]);
    }
}

// Bulk copy of `n` floats starting at element `e` of the dense tensor `base` into shared memory at `dst` (16-byte
// aligned): copies the 16-byte aligned superset; returns the bytes copied.  The data starts (e & 3) floats into dst.
__device__ __forceinline__ unsigned sfbt_copy(unsigned dst, const float* base, long long e, int n, unsigned bar) {
    const long long e0 = e & ~3LL;
    const unsigned bytes = (unsigned)(((e - e0) + n + 3) & ~3LL) * 4u;
    bulk_load(dst, base + e0, bytes, bar);
    return bytes;
}
__device__ __forceinline__ unsigned sfbt_copy_bytes(long long e, int n) {
    return (unsigned)((((e & 3LL)) + n + 3) & ~3LL) * 4u;
}

// where a lane's completed output row pairs go
struct SfbtOut {
    unsigned y_s, y_pitch_b;   // intermediate positions: shared address of the lane's four columns (row `nrow`), pitch
    float* y;                  // last position: global address of the lane's four columns in row `nrow`
    int y_rs;                  // global row stride (floats)
    int nrow;                  // output row of the even row of the next completed pair
    int row_lo, row_hi;        // rows [row_lo, row_hi) are stored
    int ncol;                  // valid columns of this lane (0..4)
    bool vec4;
};

template <bool LAST>
__device__ __forceinline__ void sfbt_store(const float2* s, SfbtOut& o) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int row = o.nrow + r;
        if (row >= o.row_lo && row < o.row_hi) {
            const float4 v = make_float4(s[2 * r].x, s[2 * r].y, s[2 * r + 1].x, s[2 * r + 1].y);
            if (!LAST) {
                sts128s(o.y_s + (unsigned)r * o.y_pitch_b, v);
            } else {
                float* d = o.y + (long long)r * o.y_rs;
                B200W_CHK(d, 4 * (o.ncol > 0 ? o.ncol : 1));
                if (o.vec4) {
                    *reinterpret_cast<float4*>(d) = v;
                } else {
                    if (o.ncol > 0) d[0] = v.x;
                    if (o.ncol > 1) d[1] = v.y;
                    if (o.ncol > 2) d[2] = v.z;
                    if (o.ncol > 3) d[3] = v.w;
                }
            }
        }
    }
    o.nrow += 2;
    o.y_s += 2u * o.y_pitch_b;
    if (LAST) o.y += 2LL * o.y_rs;
}

template <int L>
__device__ __forceinline__ void sfbt_rotate(float2 (&acc)[L / 2][4]) {
    if (SfbT<L>::kRotate) {
#pragma unroll
        for (int k = 0; k + 1 < L / 2; ++k)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[k][i] = acc[k + 1][i];
    }
}

template <int L>
__global__ void __launch_bounds__(SfbT<L>::NT, 1) sfb_tma_kernel(const __grid_constant__ SfbTmaParams p) {
    using C = SfbT<L>;
    constexpr int H2 = C::H2, NTC = C::NTC;
    constexpr bool kRotate = C::kRotate;
    constexpr int off = L - 2;
    extern __shared__ __align__(128) unsigned char smem[];
    const unsigned sbase = smem_u32(smem);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int plane = blockIdx.x / p.parts;
    const int part = blockIdx.x - plane * p.parts;
    const int J = p.J;
    pdl_trigger();
    // every 64-byte line of the parameter block is touched by a different thread first (overlapping constant-cache misses)
    if (tid < (int)(sizeof(SfbTmaParams) / 64)) {
        const int v = reinterpret_cast<const int*>(&p)[tid * 16];
        asm volatile("" ::"r"(v));
    }
    const SfbTmaPos& pl = p.pos[J - 1];
    const int D = p.D, SR = p.SR;
    const int G = pl.nseg;
    // barriers: [resident position c (J-1 of them)] [ring full: G x D] [ring empty: G x D] [a zero word]
    const unsigned bar_res = sbase + p.bar_off;
    const unsigned bar_full = bar_res + 8u * (J - 1), bar_empty = bar_full + 8u * G * D;
    if (tid < J - 1) mbar_init(bar_res + 8u * tid, 1);
    if (tid < G * D) {
        mbar_init(bar_full + 8u * tid, 1);
        mbar_init(bar_empty + 8u * tid, (unsigned)pl.nq);
    }
    if (tid < max(J - 1, G * D)) mbar_fence_init();
    if (tid == 0) *reinterpret_cast<float*>(smem + p.bar_off + 8 * (J - 1 + 2 * G * D)) = 0.f;   // the zero the taps are made opaque with
    pdl_wait();      // everything above used only the parameter block; from here on global memory is touched
    __syncthreads();

    // ---- resident positions: one bulk copy per band (and one for yl); position c is issued by warp c ----
    if (warp < J - 1) {
        {
            const int c = warp;
            const SfbTmaPos& ps = p.pos[c];
            const int k0 = ps.k0[part], rows = ps.k1[part] - k0;
            const size_t band = (size_t)ps.h * ps.w;
            const unsigned bar = bar_res + 8u * c;
            const long long e_low = ((long long)plane * ps.h + k0) * ps.w;   // c == 0: yl is dense (planes, h, w)
            if (lane == 0) {
                unsigned tx = 0;
                for (int b = 0; b < 3; ++b) tx += sfbt_copy_bytes((long long)(((size_t)plane * 3 + b) * band) + (long long)k0 * ps.w, rows * ps.w);
                if (c == 0) tx += sfbt_copy_bytes(e_low, rows * ps.w);
                mbar_expect_tx(bar, tx);
            }
            __syncwarp();
            if (lane < 3)
                sfbt_copy(sbase + ps.res_off + (unsigned)lane * ps.res_band, ps.highs,
                          (long long)(((size_t)plane * 3 + lane) * band) + (long long)k0 * ps.w, rows * ps.w, bar);
            if (lane == 3 && c == 0) sfbt_copy(sbase + p.low_off, p.yl, e_low, rows * ps.w, bar);
        }
    }

    constexpr int kServiceWarp = NTC / 32;   // the consumers are warps 0 .. NTC/32 - 1, then one service warp per ring stream
    const unsigned band_l = (unsigned)p.ring_band;                           // bytes reserved per band inside a ring stage
    const unsigned stage_b = 3u * band_l;                                    // bytes of one ring stage
    const size_t bandL = (size_t)pl.h * pl.w;
    // rows of the last position for this part
    const int ln0 = pl.n0[part], ln1 = pl.n1[part];
    const int lm_lo = (ln0 + off) >> 1, lm_hi = ((ln1 - 1 + off) >> 1) + 1;
    const int nsegL = (lm_hi - lm_lo + pl.Rp - 1) / pl.Rp;                   // ring streams of this part (<= G)

    if (warp >= kServiceWarp) {
        // ---- service warp of ring stream g (last position): lanes 0..2 issue the three band copies of a stage into a free
        // ring slot ----
        const int g = warp - kServiceWarp;
        if (g < nsegL) {
            const int m0 = lm_lo + g * pl.Rp;
            const int nm = min(pl.Rp, lm_hi - m0);
            const int kr0 = m0 - (H2 - 1);
            const int nrows = nm + H2 - 1;                                   // coefficient rows this stream reads
            const int nst = (nrows + SR - 1) / SR;
            const unsigned ring = sbase + p.ring_off + (unsigned)(g * D) * stage_b;
            auto issue = [&](int k) {
                const int st = k % D;
                const unsigned full = bar_full + 8u * (g * D + st);
                const unsigned dst = ring + (unsigned)st * stage_b;
                const int r0 = kr0 + k * SR;
                const int cnt = min(SR, kr0 + nrows - r0);                   // rows of this stage the stream reads
                if (lane == 0) {
                    unsigned tx = 0;
                    for (int b = 0; b < 3; ++b) tx += sfbt_copy_bytes((long long)(((size_t)plane * 3 + b) * bandL) + (long long)r0 * pl.w, cnt * pl.w);
                    mbar_expect_tx(full, tx);
                }
                __syncwarp();
                if (lane < 3)
                    sfbt_copy(dst + (unsigned)lane * band_l, pl.highs,
                              (long long)(((size_t)plane * 3 + lane) * bandL) + (long long)r0 * pl.w, cnt * pl.w, full);
            };
            for (int k = 0; k < min(D, nst); ++k) issue(k);
#pragma unroll 1
            for (int k = 0; k + D < nst; ++k) {
                mbar_wait(bar_empty + 8u * (g * D + k % D), (unsigned)((k / D) & 1));
                issue(k + D);
            }
        }
    }

    // ---- all chain positions, coarsest first ----
    // The consumer code below runs in warp-uniform control flow (role and trip counts are broadcast values, lanes
    // without work only skip their barrier operations and stores), so that the compiler may keep the taps and the
    // loop state in uniform registers: inside a divergent region every tap would be a register operand of its own.
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
#pragma unroll 1
    for (int c = 0; c < J; ++c) {
        const SfbTmaPos& ps = p.pos[c];
        const bool last = c + 1 == J;
        if (warp_u >= kServiceWarp) break;   // the service warps feed the last position's ring meanwhile: they must not be
                                             // waited for between positions
        // the previous position's output image is complete: barrier among the consumer warps only
        if (c > 0) asm volatile("bar.sync 1, %0;" ::"r"(NTC) : "memory");
        const int n0 = ps.n0[part], n1 = ps.n1[part];
        const int m_lo = (n0 + off) >> 1, m_hi = ((n1 - 1 + off) >> 1) + 1;
        const int ct = tid;
        int g = ct / ps.nq;
        int t = ct - g * ps.nq;
        int m0 = m_lo + g * ps.Rp;
        const bool has_work = m0 < m_hi && !(last && g >= nsegL);
        if (!has_work) { g = 0; t = 0; m0 = m_lo; }           // a lane without work shadows lane 0's addresses
        const int nm = min(ps.Rp, m_hi - m0);
        const int nrows = has_work ? nm + H2 - 1 : 0;
        int nrows_u = nrows;                                   // the warp's trip count: the longest lane's
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) nrows_u = max(nrows_u, __shfl_xor_sync(0xffffffffu, nrows_u, o2));
        nrows_u = __shfl_sync(0xffffffffu, nrows_u, 0);
        if (nrows_u == 0) continue;
        const int kr0 = m0 - (H2 - 1);
        const int k0 = ps.k0[part];
        const size_t band = (size_t)ps.h * ps.w;
        const unsigned w_b = (unsigned)ps.w * 4u;
        // low-pass input: the previous position's output image (rows from its n0), or the resident yl rows
        unsigned a_low, low_pitch_b;
        if (c == 0) {
            low_pitch_b = w_b;
            const long long e_low = ((long long)plane * ps.h + k0) * ps.w;
            a_low = sbase + p.low_off + (unsigned)((int)(e_low & 3) + (kr0 - k0) * ps.w + 2 * t) * 4u;
        } else {
            const SfbTmaPos& pv = p.pos[c - 1];
            low_pitch_b = (unsigned)pv.y_pitch * 4u;
            a_low = sbase + pv.y_off + (unsigned)(kr0 - pv.n0[part]) * low_pitch_b + 8u * t;
        }
        SfbtOut o;
        o.nrow = 2 * m0 - off;
        o.row_lo = n0; o.row_hi = has_work ? n1 : n0;          // no work: nothing is stored
        o.ncol = min(4, ps.out_w - 4 * t);
        o.vec4 = ps.vec4 != 0;
        o.y_pitch_b = (unsigned)ps.y_pitch * 4u;
        o.y_s = sbase + ps.y_off + (unsigned)((o.nrow - n0) * ps.y_pitch + 4 * t) * 4u;   // wraps for the rows before n0 (never stored)
        o.y_rs = ps.out_w;
        o.y = last ? ps.y + (size_t)plane * ps.out_h * ps.out_w + (long long)o.nrow * ps.out_w + 4 * t : nullptr;
        const SfbConstTaps taps(p.t, 0.f);
        float2 acc[H2][4];
        constexpr int UQ = kRotate ? 1 : H2;
        // shift of band b's data inside its copy destination: (first copied element) & 3
        const int eb = (int)((((size_t)plane * 3) * band) & 3), es = (int)(band & 3);
        if (!last) {
            // resident detail rows
            mbar_wait(bar_res + 8u * c, 0u);
            unsigned aH[3];
#pragma unroll
            for (int b = 0; b < 3; ++b)
                aH[b] = sbase + ps.res_off + (unsigned)b * ps.res_band +
                        (unsigned)(((eb + b * es + k0 * ps.w) & 3) + (kr0 - k0) * ps.w + 2 * t) * 4u;
            auto run = [&](auto vl, auto vh) {
#pragma unroll 1
                for (int qb = 0; qb < nrows_u; qb += UQ) {
#pragma unroll
                    for (int u = 0; u < UQ; ++u) {
                        if (qb + u < nrows_u) {
                            sfbt_row<L, decltype(vl)::value, decltype(vh)::value>(taps, a_low, aH[0], aH[1], aH[2], acc, u);
                            if (qb + u >= H2 - 1) sfbt_store<false>(acc[kRotate ? 0 : (u + 1) % H2], o);
                            sfbt_rotate<L>(acc);
                            a_low += low_pitch_b;
                            aH[0] += w_b; aH[1] += w_b; aH[2] += w_b;
                        }
                    }
                }
            };
            using I1 = std::integral_constant<int, 1>;
            using I2 = std::integral_constant<int, 2>;
            if (ps.v2) run(I2{}, I2{});
            else if (c == 0) run(I1{}, I1{});
            else run(I2{}, I1{});
        } else {
            // detail rows through the ring of stream g
            const unsigned ring = sbase + p.ring_off + (unsigned)(g * D) * stage_b + 8u * t;
            const unsigned bw = bar_full + 8u * (g * D), be = bar_empty + 8u * (g * D);
            auto run = [&](auto vh) {
                int jr = 0;                               // row inside the current stage
                int r0 = kr0;                             // first coefficient row of the current stage
                int st = 0;
                unsigned ph = 0;
                unsigned aH[3];
#pragma unroll
                for (int b = 0; b < 3; ++b) aH[b] = ring + (unsigned)b * band_l;
                bool fresh = true;                        // the current stage has not been waited for yet
#pragma unroll 1
                for (int qb = 0; qb < nrows_u; qb += UQ) {
#pragma unroll
                    for (int u = 0; u < UQ; ++u) {
                        if (qb + u < nrows_u) {
                            const bool live = qb + u < nrows;      // this lane's stream still has rows
                            if (fresh) {
                                if (live) mbar_wait(bw + 8u * st, ph);
                                fresh = false;
#pragma unroll
                                for (int b = 0; b < 3; ++b)
                                    aH[b] = ring + (unsigned)st * stage_b + (unsigned)b * band_l + (unsigned)((eb + b * es + r0 * ps.w) & 3) * 4u;
                            }
                            sfbt_row<L, 2, decltype(vh)::value>(taps, a_low, aH[0], aH[1], aH[2], acc, u);
                            if (qb + u >= H2 - 1) sfbt_store<true>(acc[kRotate ? 0 : (u + 1) % H2], o);
                            sfbt_rotate<L>(acc);
                            a_low += low_pitch_b;
                            aH[0] += w_b; aH[1] += w_b; aH[2] += w_b;
                            if (++jr == SR || qb + u + 1 == nrows) {   // done with this stage
                                if (live) mbar_arrive(be + 8u * st);
                                jr = 0;
                                r0 += SR;
                                fresh = true;
                                if (++st == D) { st = 0; ph ^= 1u; }
                            }
                        }
                    }
                }
            };
            if (ps.v2) run(std::integral_constant<int, 2>{});
            else run(std::integral_constant<int, 1>{});
        }
    }
}

// ---- host: plan + launch ------------------------------------------------------------------------------------------
static size_t up128(size_t n) { return (n + 127) & ~(size_t)127; }

template <int L>
static bool sfb_tma_plan_t(const SfbParams& p, int sms, bool force, int G_req, int D_req, SfbTmaParams& t) {
    using C = SfbT<L>;
    constexpr int H2 = C::H2, NTC = C::NTC, NCF = C::NCF;
    constexpr int off = L - 2;
    const int J = p.J;
    if (J < 2 || p.periodic) return false;
    for (int c = 0; c < J; ++c) {
        const SfbLevel& lv = p.lv[c];
        if (!lv.highs || lv.offW != off || lv.offH != off) return false;
        if (lv.w < 2 || lv.h < 1) return false;
        // the bulk copies fetch 16-byte aligned supersets of the rows: the tensors must start 16-byte aligned and
        // end on a 16-byte boundary, so that a superset never leaves them
        if (!aligned_to(lv.highs, 16) || ((long long)p.planes * 3 * lv.h * lv.w) % 4 != 0) return false;
    }
    const SfbLevel& l0 = p.lv[0];
    if (!aligned_to(l0.low, 16) || l0.low_rs != l0.w || l0.low_ps != (long long)l0.h * l0.w ||
        ((long long)p.planes * l0.h * l0.w) % 4 != 0)
        return false;
    if (!p.lv[J - 1].y) return false;
    int parts = std::min(kMaxParts, std::max(1, sms / p.planes));
    parts = std::min(parts, std::max(1, p.lv[J - 1].out_h / 2));
    if (!force && short_last_wave((long long)p.planes * parts, sms)) return false;
    t.J = J; t.planes = p.planes; t.parts = parts;
    for (int i = 0; i < kMaxTemplTaps; ++i) {
        t.t.w_lo[i] = p.t.w_lo[i]; t.t.w_hi[i] = p.t.w_hi[i];
        t.t.h_lo2[i] = p.t.h_lo2[i]; t.t.h_hi2[i] = p.t.h_hi2[i];
    }
    // rows: the last position's output rows are split evenly over the parts; every earlier position computes the rows
    // the next one reads as low-pass coefficients
    for (int c = 0; c < J; ++c) {
        SfbTmaPos& ps = t.pos[c];
        const SfbLevel& lv = p.lv[c];
        ps.y = c == J - 1 ? lv.y : nullptr;
        ps.highs = lv.highs;
        ps.h = lv.h; ps.w = lv.w; ps.out_h = lv.out_h; ps.out_w = lv.out_w;
        ps.nq = (lv.out_w + 3) / 4;
        if (ps.nq > NTC) return false;
        // the window of the last lane reaches coefficient 2*(nq-1) + NCF - 1: at most a few floats past the row end
        for (int q = 0; q < kMaxParts; ++q) ps.n0[q] = ps.n1[q] = ps.k0[q] = ps.k1[q] = 0;
    }
    for (int q = 0; q < parts; ++q) {
        t.pos[J - 1].n0[q] = (int)((long long)p.lv[J - 1].out_h * q / parts);
        t.pos[J - 1].n1[q] = (int)((long long)p.lv[J - 1].out_h * (q + 1) / parts);
        for (int c = J - 1; c >= 0; --c) {
            SfbTmaPos& ps = t.pos[c];
            if (ps.n1[q] <= ps.n0[q]) return false;
            int lo = ((ps.n0[q] + off) >> 1) - (H2 - 1);
            int hi = ((ps.n1[q] - 1 + off) >> 1) + 1;
            lo = std::max(lo, 0);
            hi = std::min(hi, ps.h);
            if (hi <= lo) return false;
            ps.k0[q] = lo; ps.k1[q] = hi;
            if (c > 0) {   // those coefficient rows are rows of the previous position's output
                if (hi > p.lv[c - 1].out_h) return false;
                t.pos[c - 1].n0[q] = lo;
                t.pos[c - 1].n1[q] = hi;
            }
        }
    }
    // segments
    for (int c = 0; c < J; ++c) {
        SfbTmaPos& ps = t.pos[c];
        int npairs = 0;
        for (int q = 0; q < parts; ++q)
            npairs = std::max(npairs, ((ps.n1[q] - 1 + off) >> 1) + 1 - ((ps.n0[q] + off) >> 1));
        int G = std::min(std::max(1, NTC / ps.nq), npairs);
        if (c == J - 1) {
            G = std::min(G, C::MAXG);
            if (G_req > 0) G = std::min(G, G_req);
        }
        ps.Rp = ceil_div(npairs, G);
        ps.nseg = ceil_div(npairs, ps.Rp);
    }
    // shared-memory layout: [barriers + a zero word | yl rows | per position: detail rows, output image | ring]
    auto chunk_bytes = [](int rows, int w) { return up128(((size_t)rows * w + 8) * 4); };   // + shift and rounding slack
    size_t o = 0;
    t.bar_off = 0;
    o += up128(8 * ((size_t)(J - 1) + 2 * (size_t)t.pos[J - 1].nseg * 8) + 16);
    {
        const SfbTmaPos& ps = t.pos[0];
        int rows = 0;
        for (int q = 0; q < parts; ++q) rows = std::max(rows, ps.k1[q] - ps.k0[q]);
        t.low_off = (int)o;
        o += chunk_bytes(rows, ps.w) + 64;    // the last lane's window may pass the last row's end by a few floats
    }
    for (int c = 0; c < J; ++c) {
        SfbTmaPos& ps = t.pos[c];
        int rows = 0, orows = 0;
        for (int q = 0; q < parts; ++q) {
            rows = std::max(rows, ps.k1[q] - ps.k0[q]);
            orows = std::max(orows, ps.n1[q] - ps.n0[q]);
        }
        ps.v2 = (ps.w % 2) == 0 ? 1 : 0;
        ps.vec4 = 0;
        if (c < J - 1) {
            ps.res_band = (int)chunk_bytes(rows, ps.w);
            ps.res_off = (int)o;
            o += (size_t)3 * ps.res_band + 64;
            // output image: what the next position reads as low-pass rows (window of its last lane) and what we store
            const int need = std::max(4 * ps.nq, 2 * (t.pos[c + 1].nq - 1) + NCF);
            ps.y_pitch = (need + 3) & ~3;
            ps.y_rows = orows;
            ps.y_off = (int)o;
            o += up128((size_t)orows * ps.y_pitch * 4 + 64);
        } else {
            ps.res_band = 0; ps.res_off = 0; ps.y_pitch = 0; ps.y_rows = 0; ps.y_off = 0;
            ps.vec4 = ((ps.out_w % 4) == 0 && aligned_to(ps.y, 16)) ? 1 : 0;
        }
    }
    t.ring_off = (int)o;
    const int G = t.pos[J - 1].nseg;
    // stage size: most rows in flight ((D - 1) stages ahead of the consumers), longer stages preferred on a tie
    // (fewer copies and barrier round trips)
    int SRb = 0, Db = 0;
    for (int SR : {8, 6, 4, 2}) {
        const size_t stage = 3 * chunk_bytes(SR, t.pos[J - 1].w);
        if (o + 64 + 2 * stage * G > kMaxDynSmem) continue;
        int D = (int)((kMaxDynSmem - o - 64) / (stage * G));
        D = std::min(D, 8);
        if (SRb == 0 || (D - 1) * SR > (Db - 1) * SRb) { SRb = SR; Db = D; }
    }
    if (SRb == 0) return false;
    if (D_req > 0) Db = std::max(2, std::min(Db, D_req));
    t.SR = SRb;
    t.D = Db;
    t.ring_band = (int)chunk_bytes(SRb, t.pos[J - 1].w);
    t.smem_bytes = (int)(o + 64 + (size_t)Db * 3 * t.ring_band * G);
    t.yl = l0.low;
    return true;
}

template <int L>
static int launch_sfb_tma_t(const SfbTmaParams& tp, cudaStream_t st) {
    using C = SfbT<L>;
    if (const cudaError_t e = allow_max_dyn_smem<sfb_tma_kernel<L>>()) return set_last_cuda_error(e);
#ifdef B200W_BOUNDS
    {
        BoundsList b;
        for (int c = 0; c < tp.J; ++c) {
            const SfbTmaPos& ps = tp.pos[c];
            b.add(ps.highs, sizeof(float) * (size_t)tp.planes * 3 * ps.h * ps.w);
            if (ps.y) b.add(ps.y, sizeof(float) * (size_t)tp.planes * ps.out_h * ps.out_w);
        }
        b.add(tp.yl, sizeof(float) * (size_t)tp.planes * tp.pos[0].h * tp.pos[0].w);
        bounds_set(b, st);
    }
#endif
    const cudaError_t le = launch_pdl(sfb_tma_kernel<L>, (unsigned)(tp.planes * tp.parts), C::NT, (size_t)tp.smem_bytes, st, tp);
    note_launch("sfb_tma_kernel");
    const cudaError_t e = le != cudaSuccess ? le : cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

bool sfb_tma_plan(const SfbParams& p, int L, int sms, bool force, int G, int D, SfbTmaParams& tp) {
    if (!tma_encode_fn()) return false;
#define X(LL) return sfb_tma_plan_t<LL>(p, sms, force, G, D, tp)
    B200W_FOR_EACH_L(X)
#undef X
    return false;
}

int launch_sfb_tma(const SfbTmaParams& tp, int L, cudaStream_t st) {
#define X(LL) return launch_sfb_tma_t<LL>(tp, st)
    B200W_FOR_EACH_L(X)
#undef X
    return B200W_ERR_BAD_TAPS;
}

}  // namespace b200w
