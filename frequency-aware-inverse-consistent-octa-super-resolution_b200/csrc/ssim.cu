// Gaussian-window SSIM, forward and backward, for sm_100a.
//
// Forward (replaces ssim.py:17-37: five dense 11x11 F.conv2d + ~15 pointwise kernels + mean): one
// streaming kernel.  A CTA owns a strip of TW output columns of one image plane and marches down it in
// chunks of 32 rows.  Per chunk: stage the two input row blocks (zero outside the image, i.e. the
// conv's zero padding), horizontal 11-tap pass of the FOUR moments x1, x2, x1^2 + x2^2, x1*x2 (the SSIM
// formula only uses sigma1^2 + sigma2^2, and the blur is linear, so the two squares share one blur;
// products formed in registers) into a shared-memory window of 42 rows, vertical 11-tap pass, SSIM
// map, running sum.  The last 10 horizontally-blurred rows are carried to the next chunk, so no row is
// filtered twice.  The 2-D window of ssim.py:11-15 is the outer product of the 1-D Gaussian, applied
// separably.  Both passes run on the packed FFMA2 (fma.rn.f32x2) pipe:
//   horizontal: a pair = two ADJACENT INPUT columns (as the 128-bit shared loads deliver them) times the tap
//               pair (w[d], w[d+1]); the two lanes are partial sums over the even / odd taps, added at the end;
//   vertical:   a pair = two CHANNELS of one pixel (the window holds (mu1, mu2) and (E[x1^2+x2^2], E[x1 x2]) as
//               float2) times (w[d], w[d]).
// Optionally the forward also stores the 3 (or 4) derivative maps the backward needs, so the backward
// is one more streaming kernel (3-4 blurs + combine) instead of autograd through ~25 kernels.
//
// Closed-form backward (SURVEY.md 8a-a10; oracle/ssim_oracle.py):
//   dx1 = W*(g M0) + 2 x1 W*(g M1) + x2 W*(g M2),   dx2 = W*(g M3) + 2 x2 W*(g M1) + x1 W*(g M2)
//   M0 = dS/dmu1, M1 = dS/dE[x1^2] = dS/dE[x2^2] = -S/B2, M2 = dS/dE[x1 x2] = 2 A1/(B1 B2), M3 = dS/dmu2
#include "common.cuh"

namespace b200w {

constexpr int kWin = B200W_SSIM_MAX_WINDOW;  // 11
constexpr int kHalo = kWin / 2;              // 5
constexpr int kTW = 64;                      // output columns per CTA
constexpr int kCR = 32;                      // rows per chunk
constexpr int kPW = kTW + 16;                // staged columns: image cols [C0-8, C0+72)
constexpr int kHR = kCR + 2 * kHalo;         // 42 horizontally-blurred rows resident
// forward: one staging buffer (63 KB per CTA, 3 CTAs/SM; the next chunk is fetched during the vertical pass);
// backward: two (its 3-4 staged maps are loaded a whole chunk ahead)
template <bool FWD> constexpr int kSsimStageBufs = FWD ? 1 : 2;

// options of the MS-SSIM scale instantiations (0: the plain SSIM kernels)
constexpr int kOptMs = 1;    // fwd: the map value by correctly rounded division, so identical images give exactly 1
constexpr int kOptCs = 2;    // fwd: the contrast-structure map cs = A2/B2 and its derivative maps instead of S
constexpr int kOptPool = 4;  // fwd: also write avg_pool2d(img1, 2) and avg_pool2d(img2, 2)
constexpr int kOptUp = 8;    // bwd: add 0.25 up[r/2][c/2] (the transpose of that pooling) to d1 / d2

struct SsimParams {
    const float* in[4];   // fwd: img1, img2 ; bwd: maps 0..3
    const float* img1;    // bwd epilogue
    const float* img2;
    const float* grad_out;
    float* out0;          // fwd: maps base (or null) ; bwd: d1
    float* out1;          // bwd: d2 (or null)
    float* partials;      // fwd: one float per CTA
    long long plane_elems;   // H*W
    long long map_stride;    // planes*H*W
    int planes, C, H, W;
    int strips, nseg, seg_rows;
    int n_maps, size_average;
    int vec_ok;           // 16 B staging copies allowed (W % 4 == 0 and every base 16 B aligned)
    float inv_count;      // 1/(N*C*H*W) or 1/(C*H*W)
    float win[kWin];
    // tap pairs of the packed passes (fill_window): wa[k] = (w[2k], w[2k+1]), wb[k] = (w[2k-1], w[2k]) with
    // w[-1] = w[11] = 0 (windows starting on an even / odd staged column), w2[d] = (w[d], w[d])
    float2 wa[6];
    float2 wb[6];
    float2 w2[kWin];
    // MS-SSIM scale fields, after the plain SSIM ones so that those keep their parameter offsets
    float* pooled1;       // fwd (kOptPool): (planes, Hp, Wp)
    float* pooled2;
    const float* up1;     // bwd (kOptUp): (planes, Hp, Wp) or null
    const float* up2;
    int Hp, Wp;           // H / 2, W / 2
};

// Stage rows [row0, row0+nrows) x cols [C0-8, C0+72) of one plane into dst[nrows][kPW] with cp.async, zero
// outside the image (= the conv's zero padding).  Thread = one vector column, walking down the rows.
template <int V>
__device__ __forceinline__ void stage_rows(unsigned dst_s, const float* __restrict__ src, int row0, int nrows, int C0,
                                           int H, int W, int tid) {
    constexpr int NVC = kPW / V;
    constexpr int NRG = kThreads / NVC;
    if (tid >= NVC * NRG) return;
    const int cv = tid % NVC;
    const int rg = tid / NVC;
    const int gc = C0 - 8 + V * cv;
    const bool col_in = gc >= 0 && gc + V <= W;   // V == 4 needs W % 4 == 0: a chunk is entirely in or out
    unsigned dst = dst_s + (unsigned)((rg * kPW + V * cv) * 4);
    const float* p = src + (long long)(row0 + rg) * W + gc;
    const long long step = (long long)NRG * W;
    for (int r = rg; r < nrows; r += NRG, dst += NRG * kPW * 4, p += step) {
        const int gr = row0 + r;
        if (col_in && gr >= 0 && gr < H) cp_async<V>(dst, p);
        else cp_async_zero<V>(dst, src);
    }
}

// shared-memory window of horizontally blurred rows: [pair][row][col] of float2, the 16-byte chunks (2 columns) of a
// row XOR-swizzled so that both the 128-bit stores of the horizontal pass (a lane owns 4 columns = 2 chunks, 32 B
// apart) and the 64-bit loads of the vertical pass (a lane owns 1 column) are bank-conflict free
__device__ __forceinline__ int hbuf_col(int c) { return ((((c >> 1) ^ ((c >> 4) & 1)) << 1) | (c & 1)); }

// FWD: 4 channels (x1, x2, x1^2 + x2^2, x1 x2) from NI = 2 staged inputs.  BWD: NC = NI = 3 or 4 staged maps.
// Either way the window holds 2 channel pairs (the fourth channel of the 3-map backward is a zero lane).
template <bool FWD, int NC, int OPT = 0>
__global__ void __launch_bounds__(kThreads, FWD ? 3 : 2) ssim_stream_kernel(const __grid_constant__ SsimParams p) {
    constexpr int NI = FWD ? 2 : NC;
    constexpr int NB = kSsimStageBufs<FWD>;    // staging buffers
    constexpr int NCH = FWD ? 4 : NC;          // channels of the horizontal pass
    constexpr int SB = NI * kCR * kPW;         // floats per staging buffer
    extern __shared__ __align__(16) float smem[];
    float2* hbuf = reinterpret_cast<float2*>(smem + NB * SB);  // [2][kHR][kTW] (the staging buffers [NI][kCR][kPW] first)
    __shared__ float red[kThreads / 32];
    const unsigned smem_s = (unsigned)__cvta_generic_to_shared(smem);

    const int tid = threadIdx.x;
    int bid = blockIdx.x;
    const int strip = bid % p.strips;
    bid /= p.strips;
    const int seg = bid % p.nseg;
    const int plane = bid / p.nseg;
    const int C0 = strip * kTW;
    const int S0 = seg * p.seg_rows;
    const int S1 = min(S0 + p.seg_rows, p.H);
    const int H = p.H, W = p.W;

    const float* src[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) src[i] = p.in[i] + (long long)plane * p.plane_elems;

    float g = 0.f;
    if (!FWD) g = __ldg(p.grad_out + (p.size_average ? 0 : plane / p.C)) * p.inv_count;
    float local_sum = 0.f;

    // chunk q covers horizontally-blurred rows [S0 + 32q + 5, +32); chunk -1 is the prologue [S0-5, S0+5)
    const int niter = (S1 - S0 + kCR - 1) / kCR;
    auto issue = [&](int q, int buf) {
        const int nrows = q < 0 ? 2 * kHalo : kCR;
        const int in_row0 = q < 0 ? S0 - kHalo : S0 + kCR * q + kHalo;
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const unsigned d = smem_s + (unsigned)((buf * SB + i * kCR * kPW) * 4);
            if (p.vec_ok) stage_rows<4>(d, src[i], in_row0, nrows, C0, H, W, tid);
            else stage_rows<1>(d, src[i], in_row0, nrows, C0, H, W, tid);
        }
    };
    issue(-1, 0);
    cp_async_commit();

    // backward epilogue inputs x1, x2 of this thread's 8 output rows of a chunk (thread = (column, strip), as in the
    // vertical pass), loaded a whole chunk ahead so that their DRAM latency hides behind a chunk of filtering
    float x1n[8], x2n[8];
    // kOptUp: 0.25 up of the 4 pooled rows under those 8 rows (row0 is even), fetched with them
    float u1n[4], u2n[4];
    auto fetch_x = [&](int qn) {
        const int col = C0 + tid % kTW;
        const int row0 = S0 + kCR * qn + 8 * (tid / kTW);
        const long long off = (long long)plane * p.plane_elems + (long long)row0 * W + col;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const bool ok = col < W && row0 + i < S1;
            x1n[i] = ok ? __ldg(p.img1 + off + (long long)i * W) : 0.f;
            x2n[i] = ok ? __ldg(p.img2 + off + (long long)i * W) : 0.f;
        }
        if constexpr ((OPT & kOptUp) != 0) {
            const int pr0 = row0 >> 1, pc = col >> 1;
            const long long uoff = ((long long)plane * p.Hp + pr0) * p.Wp + pc;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const bool ok = pc < p.Wp && pr0 + k < p.Hp;
                u1n[k] = ok && p.up1 ? 0.25f * __ldg(p.up1 + uoff + (long long)k * p.Wp) : 0.f;
                u2n[k] = ok && p.up2 ? 0.25f * __ldg(p.up2 + uoff + (long long)k * p.Wp) : 0.f;
            }
        }
    };
    if (!FWD) fetch_x(0);

    for (int q = -1; q < niter; ++q) {
        const int buf = NB == 2 ? (q + 1) & 1 : 0;
        if (NB == 2) {
            if (q + 1 < niter) issue(q + 1, buf ^ 1);   // prefetch the next chunk while this one is filtered
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const float* stage = smem + buf * SB;
        const int nrows = q < 0 ? 2 * kHalo : kCR;
        const int hrow0 = q < 0 ? 0 : 2 * kHalo;   // window row receiving staged row 0

        // ---- horizontal pass: item = (row, quad of 4 output columns); 128-bit shared loads and stores.
        //      Output o (0..3) of the quad is image col C0+4cq+o = staged col 4cq+o+8; its window is staged cols
        //      4cq+o+3 .. 4cq+o+13 = v[o+3 .. o+13].  The loads deliver the aligned pairs (v[j], v[j+1]), j even:
        //      an odd window start (o even) uses the tap pairs wb = (0,w0),(w1,w2)..(w9,w10) from j = o+2, an even
        //      one (o odd) wa = (w0,w1)..(w8,w9),(w10,0) from j = o+3.
        {
            const int cq = tid % (kTW / 4);
            int r = tid / (kTW / 4);
            const int sw = (cq >> 2) & 1;   // chunk swizzle of this lane's two 16-byte stores
            const float* sp0 = stage + r * kPW + 4 * cq;
            float4* hp = reinterpret_cast<float4*>(hbuf + (hrow0 + r) * kTW) + 2 * cq;
            constexpr int RSTEP = kThreads / (kTW / 4);
            for (; r < nrows; r += RSTEP, sp0 += RSTEP * kPW, hp += RSTEP * kTW / 2) {
                float2 v[NI][10];
#pragma unroll
                for (int i = 0; i < NI; ++i) {
#pragma unroll
                    for (int c = 0; c < 5; ++c) {
                        const float4 t = reinterpret_cast<const float4*>(sp0 + i * kCR * kPW)[c];
                        v[i][2 * c] = make_float2(t.x, t.y);
                        v[i][2 * c + 1] = make_float2(t.z, t.w);
                    }
                }
                float2 acc[NCH][4];
#pragma unroll
                for (int jj = 1; jj <= 8; ++jj) {      // pair jj = staged cols (2jj, 2jj+1) of this quad's window
                    float2 ch[NCH];
                    if (FWD) {
                        const float2 a = v[0][jj], b = v[1][jj];
                        ch[0] = a;
                        ch[1] = b;
                        ch[2 % NCH] = ffma2(b, b, fmul2(a, a));
                        ch[3 % NCH] = fmul2(a, b);
                    } else {
#pragma unroll
                        for (int m = 0; m < NCH; ++m) ch[m] = v[m][jj];
                    }
#pragma unroll
                    for (int o = 0; o < 4; ++o) {
                        const int j0 = (o & 1) ? o + 3 : o + 2;
                        const int k = jj - j0 / 2;
                        if (k >= 0 && k < 6) {
                            const float2 w = (o & 1) ? p.wa[k] : p.wb[k];
#pragma unroll
                            for (int m = 0; m < NCH; ++m) acc[m][o] = k == 0 ? fmul2(w, ch[m]) : ffma2(w, ch[m], acc[m][o]);
                        }
                    }
                }
                float a[4][4];
#pragma unroll
                for (int m = 0; m < 4; ++m)
#pragma unroll
                    for (int o = 0; o < 4; ++o) a[m][o] = m < NCH ? acc[m % NCH][o].x + acc[m % NCH][o].y : 0.f;
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                    float4* d = hp + pr * (kHR * kTW / 2);
                    d[sw] = make_float4(a[2 * pr][0], a[2 * pr + 1][0], a[2 * pr][1], a[2 * pr + 1][1]);
                    d[sw ^ 1] = make_float4(a[2 * pr][2], a[2 * pr + 1][2], a[2 * pr][3], a[2 * pr + 1][3]);
                }
            }
        }
        if constexpr (FWD && (OPT & kOptPool) != 0) {
            // ---- 2x2 average pools of the staged rows, before the staging buffer is reused.  A chunk stages rows
            //      [in_row0, in_row0 + nrows) with in_row0 odd (S0 is even) and nrows even: staged row r even is an odd
            //      image row, the bottom of pooled row (in_row0 + r - 1) / 2, whose top is staged row r - 1 or, for
            //      r = 0, the last row of the previous chunk, kept in a carry row (two of them, alternating by chunk)
            float* carry = smem + NB * SB + 2 * 2 * kHR * kTW;   // [2][NI][kTW]
            const float* cin = carry + (q & 1) * NI * kTW;
            float* cout = carry + ((q + 1) & 1) * NI * kTW;
            const int in_row0 = q < 0 ? S0 - kHalo : S0 + kCR * q + kHalo;
            const long long pplane = (long long)plane * p.Hp * p.Wp;
            for (int it = tid; it < (nrows / 2) * (kTW / 2); it += kThreads) {
                const int r = 2 * (it / (kTW / 2)), pc = it % (kTW / 2);
                const int gr = in_row0 + r;
                if (gr - 1 < S0 || gr >= S1 || C0 + 2 * pc + 1 >= W) continue;
                const long long o = pplane + (long long)((gr - 1) >> 1) * p.Wp + (C0 >> 1) + pc;
#pragma unroll
                for (int i = 0; i < NI; ++i) {
                    const float* sp = stage + i * kCR * kPW + 2 * pc + 8;
                    const float2 t = r == 0 ? *reinterpret_cast<const float2*>(cin + i * kTW + 2 * pc)
                                            : *reinterpret_cast<const float2*>(sp + (r - 1) * kPW);
                    const float2 b = *reinterpret_cast<const float2*>(sp + r * kPW);
                    (i == 0 ? p.pooled1 : p.pooled2)[o] = (((t.x + t.y) + b.x) + b.y) * 0.25f;   // avg_pool2d's order
                }
            }
            for (int it = tid; it < NI * kTW; it += kThreads)
                cout[it] = stage[(it / kTW) * kCR * kPW + (nrows - 1) * kPW + it % kTW + 8];
        }
        __syncthreads();
        if (NB == 1) {   // the one staging buffer is free again: the next chunk lands during the vertical pass
            if (q + 1 < niter) issue(q + 1, 0);
            cp_async_commit();
        }
        if (q < 0) continue;

        // ---- vertical pass: thread = (column, strip of 8 output rows); a pair = two channels of the pixel
        {
            const int c = tid % kTW;
            const int s = tid / kTW;  // 0..3
            const int col = C0 + c;
            const int row0 = S0 + kCR * q + 8 * s;
            const bool live = col < W && row0 < S1;
            const long long off = (long long)plane * p.plane_elems + (long long)row0 * W + col;
            float x1v[8], x2v[8], u1v[4], u2v[4];
            if (!FWD) {   // the epilogue's inputs were requested one chunk ago; request the next chunk's now
#pragma unroll
                for (int i = 0; i < 8; ++i) { x1v[i] = x1n[i]; x2v[i] = x2n[i]; }
                if constexpr ((OPT & kOptUp) != 0) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) { u1v[k] = u1n[k]; u2v[k] = u2n[k]; }
                }
                fetch_x(q + 1);
            }
            float2 acc[2][8];
            const float2* hb = hbuf + (8 * s) * kTW + hbuf_col(c);
#pragma unroll
            for (int rr = 0; rr < 8 + kWin - 1; ++rr) {
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {
                    const float2 t = hb[(pr * kHR + rr) * kTW];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int d = rr - i;
                        if (d >= 0 && d < kWin) acc[pr][i] = d == 0 ? fmul2(p.w2[0], t) : ffma2(p.w2[d], t, acc[pr][i]);
                    }
                }
            }
            if (live) {
                if (FWD) {
                    float* m0 = p.out0 + off;
                    const long long ms = p.map_stride;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        if (row0 + i < S1) {
                            const float C1 = 0.0001f, C2 = 0.0009f;
                            const float mu1 = acc[0][i].x, mu2 = acc[0][i].y;
                            // explicit roundings (no FMA contraction across these): for img1 == img2 the merged
                            // moment is exactly 2 E[x1 x2], so A1 == B1 and A2 == B2 bit for bit, as in the
                            // reference where the three product blurs are then the same numbers
                            const float mu12 = __fmul_rn(mu1, mu2);
                            const float msum = __fadd_rn(__fmul_rn(mu1, mu1), __fmul_rn(mu2, mu2));
                            const float s12 = __fsub_rn(acc[1][i].y, mu12);
                            const float ssum = __fsub_rn(acc[1][i].x, msum);   // sigma1^2 + sigma2^2
                            const float A1 = __fmaf_rn(2.f, mu12, C1), A2 = __fmaf_rn(2.f, s12, C2);
                            const float B1 = __fadd_rn(msum, C1), B2 = __fadd_rn(ssum, C2);
                            if constexpr ((OPT & kOptCs) != 0) {
                                const float cs = __fdiv_rn(A2, B2);   // exactly 1 where A2 == B2
                                local_sum += cs;
                                if (p.n_maps) {
                                    const float ib = __fdividef(1.f, B2);
                                    m0[0] = 2.f * (mu1 * cs - mu2) * ib;                       // M0 = dcs/dmu1
                                    m0[ms] = -cs * ib;                                         // M1 = -cs / B2
                                    m0[2 * ms] = 2.f * ib;                                     // M2 = 2 / B2
                                    if (p.n_maps == 4) m0[3 * ms] = 2.f * (mu2 * cs - mu1) * ib;   // M3 = dcs/dmu2
                                }
                                m0 += W;
                                continue;
                            }
                            const float inv = __fdividef(1.f, B1 * B2);   // B1, B2 >= ~1e-4: one MUFU.RCP, 2 ulp
                            // kOptMs: correctly rounded, exactly 1 where A1 == B1 and A2 == B2
                            const float S = (OPT & kOptMs) != 0 ? __fdiv_rn(__fmul_rn(A1, A2), __fmul_rn(B1, B2))
                                                                : (A1 * A2) * inv;
                            local_sum += S;
                            if (p.n_maps) {
                                const float k = 2.f * (A2 - A1) * inv;            // common factor of dS/dmu
                                const float e = 2.f * S * (B2 - B1) * inv;        // 2 S (1/B1 - 1/B2)
                                m0[0] = mu2 * k - mu1 * e;                        // M0 = dS/dmu1
                                m0[ms] = -S * B1 * inv;                           // M1 = -S / B2
                                m0[2 * ms] = 2.f * A1 * inv;                      // M2
                                if (p.n_maps == 4) m0[3 * ms] = mu1 * k - mu2 * e;  // M3 = dS/dmu2
                            }
                        }
                        m0 += W;
                    }
                } else {
                    float* d1 = p.out0 + off;
                    float* d2 = (NC == 4 && p.out1) ? p.out1 + off : nullptr;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        if (row0 + i < S1) {
                            const float x1 = x1v[i], x2 = x2v[i];
                            const float b0 = acc[0][i].x, b1 = acc[0][i].y, b2 = acc[1][i].x, b3 = acc[1][i].y;
                            if constexpr ((OPT & kOptUp) != 0) {
                                *d1 = g * (b0 + 2.f * x1 * b1 + x2 * b2) + u1v[i >> 1];
                                if (NC == 4 && d2) *d2 = g * (b3 + 2.f * x2 * b1 + x1 * b2) + u2v[i >> 1];
                            } else {
                                *d1 = g * (b0 + 2.f * x1 * b1 + x2 * b2);
                                if (NC == 4 && d2) *d2 = g * (b3 + 2.f * x2 * b1 + x1 * b2);
                            }
                        }
                        d1 += W;
                        if (NC == 4 && d2) d2 += W;
                    }
                }
            }
        }
        __syncthreads();
        // ---- carry the last 10 blurred rows to the top of the window (ordered before the next vertical pass by
        //      the barrier that follows the next cp.async wait)
        if (q + 1 < niter) {
            constexpr int RW4 = kTW / 2;                 // float4 per window row
            constexpr int N4 = 2 * 2 * kHalo * RW4;
            for (int idx = tid; idx < N4; idx += kThreads) {
                const int m = idx / (2 * kHalo * RW4);
                const int rem = idx - m * (2 * kHalo * RW4);
                float4* base = reinterpret_cast<float4*>(hbuf + m * kHR * kTW);
                base[rem] = base[kCR * RW4 + rem];
            }
        }
    }

    if (FWD) {
        float s = warp_sum(local_sum);
        if ((tid & 31) == 0) red[tid >> 5] = s;
        __syncthreads();
        if (tid < 32) {
            float t = tid < kThreads / 32 ? red[tid] : 0.f;
            t = warp_sum(t);
            if (tid == 0) p.partials[blockIdx.x] = t;
        }
    }
}

// deterministic final reduction: out[n] = (sum of the partials of sample n) * inv_count, in double
__global__ void __launch_bounds__(kThreads) ssim_finalize_kernel(const float* __restrict__ partials,
                                                                  int per_out, double inv_count,
                                                                  float* __restrict__ out) {
    __shared__ double red[kThreads / 32];
    const float* src = partials + (size_t)blockIdx.x * per_out;
    double s = 0.0;
    for (int i = threadIdx.x; i < per_out; i += kThreads) s += (double)src[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < kThreads / 32; ++i) t += red[i];
        out[blockIdx.x] = (float)(t * inv_count);
    }
}

static void plan_grid(int planes, int H, int W, int* strips, int* nseg, int* seg_rows) {
    *strips = (W + kTW - 1) / kTW;
    const int max_seg = (H + kCR - 1) / kCR;
    const long long base = (long long)planes * *strips;
    const long long target = 148LL * 3 * 4;  // a few waves at 3 CTAs/SM
    int n = (int)((target + base - 1) / base);
    if (n < 1) n = 1;
    if (n > max_seg) n = max_seg;
    int rows = (H + n - 1) / n;
    rows = (rows + kCR - 1) / kCR * kCR;
    *seg_rows = rows;
    *nseg = (H + rows - 1) / rows;
}

template <bool FWD, int NC, int OPT = 0>
static int launch_ssim(const SsimParams& p, cudaStream_t st) {
    constexpr int NI = FWD ? 2 : NC;
    constexpr int carry = (OPT & kOptPool) != 0 ? 2 * NI * kTW : 0;
    const size_t smem = sizeof(float) * (size_t)(kSsimStageBufs<FWD> * NI * kCR * kPW + 2 * 2 * kHR * kTW + carry);
    auto kern = ssim_stream_kernel<FWD, NC, OPT>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_last_cuda_error(e);
    const size_t grid = (size_t)p.planes * p.nseg * p.strips;
    kern<<<(unsigned)grid, kThreads, smem, st>>>(p);
    note_launch(FWD ? "ssim_stream_kernel<fwd>" : "ssim_stream_kernel<bwd>");
    e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

static bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; }

static int fill_window(SsimParams& p, const float* win, int ws) {
    if (!win || ws < 1 || ws > kWin || (ws % 2) == 0) return B200W_ERR_BAD_WINDOW;
    for (int i = 0; i < kWin; ++i) p.win[i] = 0.f;
    const int shift = (kWin - ws) / 2;  // a smaller odd window is the same "same" conv with zero outer taps
    for (int i = 0; i < ws; ++i) p.win[shift + i] = win[i];
    auto w = [&](int i) { return (i >= 0 && i < kWin) ? p.win[i] : 0.f; };
    for (int k = 0; k < 6; ++k) {
        p.wa[k] = make_float2(w(2 * k), w(2 * k + 1));
        p.wb[k] = make_float2(w(2 * k - 1), w(2 * k));
    }
    for (int d = 0; d < kWin; ++d) p.w2[d] = make_float2(p.win[d], p.win[d]);
    return B200W_OK;
}

}  // namespace b200w

using namespace b200w;

extern "C" size_t b200w_ssim_workspace_bytes(int N, int C, int H, int W) {
    if (N < 1 || C < 1 || H < 1 || W < 1) return 0;
    int strips, nseg, seg_rows;
    plan_grid(N * C, H, W, &strips, &nseg, &seg_rows);
    return sizeof(float) * (size_t)N * C * strips * nseg;
}

extern "C" int b200w_ssim_fwd_f32(const float* img1, const float* img2, int N, int C, int H, int W,
                                  const float* win, int ws, int size_average, int n_maps, float* maps, float* out,
                                  void* workspace, size_t workspace_bytes, void* stream) {
    if (!img1 || !img2 || !out) return B200W_ERR_NULL_POINTER;
    if (N < 1 || C < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!(n_maps == 0 || n_maps == 3 || n_maps == 4)) return B200W_ERR_BAD_SHAPE;
    if (n_maps && !maps) return B200W_ERR_NULL_POINTER;
    SsimParams p = {};
    int rc = fill_window(p, win, ws);
    if (rc) return rc;
    p.planes = N * C;
    p.C = C;
    p.H = H;
    p.W = W;
    plan_grid(p.planes, H, W, &p.strips, &p.nseg, &p.seg_rows);
    const size_t need = sizeof(float) * (size_t)p.planes * p.strips * p.nseg;
    if (!workspace || workspace_bytes < need) return B200W_ERR_WORKSPACE;
    p.in[0] = img1;
    p.in[1] = img2;
    p.out0 = maps;
    p.partials = (float*)workspace;
    p.plane_elems = (long long)H * W;
    p.map_stride = (long long)p.planes * H * W;
    p.n_maps = n_maps;
    p.size_average = size_average ? 1 : 0;
    p.vec_ok = ((W % 4) == 0 && aligned16(img1) && aligned16(img2)) ? 1 : 0;
    cudaStream_t st = (cudaStream_t)stream;
    rc = launch_ssim<true, 4>(p, st);
    if (rc) return rc;
    const int per_plane = p.strips * p.nseg;
    const int nout = size_average ? 1 : N;
    const int per_out = size_average ? p.planes * per_plane : C * per_plane;
    const double inv = size_average ? 1.0 / ((double)N * C * H * W) : 1.0 / ((double)C * H * W);
    ssim_finalize_kernel<<<nout, kThreads, 0, st>>>(p.partials, per_out, inv, out);
    note_launch("ssim_finalize_kernel");
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

extern "C" int b200w_ssim_bwd_f32(const float* img1, const float* img2, const float* maps, int n_maps,
                                  const float* grad_out, int N, int C, int H, int W, const float* win, int ws,
                                  int size_average, float* d1, float* d2, void* stream) {
    if (!img1 || !img2 || !maps || !grad_out || !d1) return B200W_ERR_NULL_POINTER;
    if (N < 1 || C < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!(n_maps == 3 || n_maps == 4) || (d2 && n_maps != 4)) return B200W_ERR_BAD_SHAPE;
    SsimParams p = {};
    int rc = fill_window(p, win, ws);
    if (rc) return rc;
    p.planes = N * C;
    p.C = C;
    p.H = H;
    p.W = W;
    plan_grid(p.planes, H, W, &p.strips, &p.nseg, &p.seg_rows);
    p.plane_elems = (long long)H * W;
    p.map_stride = (long long)p.planes * H * W;
    for (int i = 0; i < n_maps; ++i) p.in[i] = maps + (size_t)i * p.map_stride;
    p.img1 = img1;
    p.img2 = img2;
    p.grad_out = grad_out;
    p.out0 = d1;
    p.out1 = d2;
    p.n_maps = n_maps;
    p.size_average = size_average ? 1 : 0;
    p.inv_count = size_average ? (float)(1.0 / ((double)N * C * H * W)) : (float)(1.0 / ((double)C * H * W));
    p.vec_ok = ((W % 4) == 0 && aligned16(maps)) ? 1 : 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (d2) return launch_ssim<false, 4>(p, st);
    return launch_ssim<false, 3>(p, st);
}

// MS-SSIM, one scale: the SSIM kernels with the per-sample value of the SSIM map (cs == 0) or of the contrast-structure
// map (cs != 0), optionally the 2x2 average pools of both images (forward) and the pooling's transpose (backward)
extern "C" int b200w_msssim_scale_fwd_f32(const float* img1, const float* img2, int N, int C, int H, int W,
                                          const float* win, int ws, int cs, int n_maps, float* maps, float* out,
                                          float* pooled1, float* pooled2, void* workspace, size_t workspace_bytes,
                                          void* stream) {
    if (!img1 || !img2 || !out) return B200W_ERR_NULL_POINTER;
    if (N < 1 || C < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!(n_maps == 0 || n_maps == 3 || n_maps == 4)) return B200W_ERR_BAD_SHAPE;
    if (n_maps && !maps) return B200W_ERR_NULL_POINTER;
    if (!pooled1 != !pooled2) return B200W_ERR_NULL_POINTER;
    const bool pool = pooled1 != nullptr;
    if (pool && (H < 2 || W < 2)) return B200W_ERR_BAD_SHAPE;
    SsimParams p = {};
    int rc = fill_window(p, win, ws);
    if (rc) return rc;
    p.planes = N * C;
    p.C = C;
    p.H = H;
    p.W = W;
    plan_grid(p.planes, H, W, &p.strips, &p.nseg, &p.seg_rows);
    const size_t need = sizeof(float) * (size_t)p.planes * p.strips * p.nseg;
    if (!workspace || workspace_bytes < need) return B200W_ERR_WORKSPACE;
    p.in[0] = img1;
    p.in[1] = img2;
    p.out0 = maps;
    p.partials = (float*)workspace;
    p.plane_elems = (long long)H * W;
    p.map_stride = (long long)p.planes * H * W;
    p.n_maps = n_maps;
    p.vec_ok = ((W % 4) == 0 && aligned16(img1) && aligned16(img2)) ? 1 : 0;
    p.pooled1 = pooled1;
    p.pooled2 = pooled2;
    p.Hp = H / 2;
    p.Wp = W / 2;
    cudaStream_t st = (cudaStream_t)stream;
    if (cs) rc = pool ? launch_ssim<true, 4, kOptMs | kOptCs | kOptPool>(p, st) : launch_ssim<true, 4, kOptMs | kOptCs>(p, st);
    else rc = pool ? launch_ssim<true, 4, kOptMs | kOptPool>(p, st) : launch_ssim<true, 4, kOptMs>(p, st);
    if (rc) return rc;
    const int per_plane = p.strips * p.nseg;
    ssim_finalize_kernel<<<N, kThreads, 0, st>>>(p.partials, C * per_plane, 1.0 / ((double)C * H * W), out);
    note_launch("ssim_finalize_kernel");
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

extern "C" int b200w_msssim_scale_bwd_f32(const float* img1, const float* img2, const float* maps, int n_maps,
                                          const float* grad_out, int N, int C, int H, int W, const float* win, int ws,
                                          const float* up1, const float* up2, float* d1, float* d2, void* stream) {
    if (!img1 || !img2 || !maps || !grad_out || !d1) return B200W_ERR_NULL_POINTER;
    if (N < 1 || C < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!(n_maps == 3 || n_maps == 4) || (d2 && n_maps != 4)) return B200W_ERR_BAD_SHAPE;
    if (up2 && !d2) return B200W_ERR_BAD_SHAPE;
    const bool up = up1 || up2;
    if (up && (H < 2 || W < 2)) return B200W_ERR_BAD_SHAPE;
    SsimParams p = {};
    int rc = fill_window(p, win, ws);
    if (rc) return rc;
    p.planes = N * C;
    p.C = C;
    p.H = H;
    p.W = W;
    plan_grid(p.planes, H, W, &p.strips, &p.nseg, &p.seg_rows);
    p.plane_elems = (long long)H * W;
    p.map_stride = (long long)p.planes * H * W;
    for (int i = 0; i < n_maps; ++i) p.in[i] = maps + (size_t)i * p.map_stride;
    p.img1 = img1;
    p.img2 = img2;
    p.grad_out = grad_out;
    p.out0 = d1;
    p.out1 = d2;
    p.n_maps = n_maps;
    p.size_average = 0;
    p.inv_count = (float)(1.0 / ((double)C * H * W));
    p.vec_ok = ((W % 4) == 0 && aligned16(maps)) ? 1 : 0;
    p.up1 = up1;
    p.up2 = up2;
    p.Hp = H / 2;
    p.Wp = W / 2;
    cudaStream_t st = (cudaStream_t)stream;
    if (d2) return up ? launch_ssim<false, 4, kOptUp>(p, st) : launch_ssim<false, 4>(p, st);
    return up ? launch_ssim<false, 3, kOptUp>(p, st) : launch_ssim<false, 3>(p, st);
}
