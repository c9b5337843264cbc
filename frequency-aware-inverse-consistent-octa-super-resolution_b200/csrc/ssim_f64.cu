// Gaussian-window SSIM in double precision, forward and backward, for sm_100a: the reference's _ssim (ssim.py:17-37)
// on double images.
//
// Why not the separable fp32 kernel (ssim.cu) instantiated for double: in double the reference applies a window that
// is not separable.  ssim.py:7-15 builds it as the outer product of the 1-D Gaussian in the default dtype, rounds the
// 121 products to fp32 with .float() and casts them to the images' dtype (type_as).  A separable pass would differ from
// it by that fp32 rounding (~1e-8 relative), which is the precision this path exists to keep.  So these kernels apply
// the dense ws x ws window the caller passes, tap by tap.
//
// Forward (ssim_f64_kernel): a CTA owns a 32 x 64 output tile of one plane.  It stages the tile plus its 5-pixel halo
// of both images into shared memory as doubles (cp.async 8-byte copies, zero outside the image = the conv's zero
// padding), forms the two product channels x1^2 + x2^2 and x1 x2 in place (the SSIM formula only uses
// sigma1^2 + sigma2^2, so the two squares share one blur), and each thread correlates a column of 8 outputs with the
// 11 x 11 window for the 4 channels: 4 x 121 DFMA per pixel.  The window travels in the parameter block; per window
// column the 11 taps are read once into registers.  Epilogue as in ssim.cu, in double with explicit roundings: SSIM
// map, optional 3 / 4 derivative maps (same meaning and order as b200w_ssim_fwd_f32), per-CTA partial sum.
// ssim_f64_finalize_kernel reduces the partials in a fixed order: results are bit-reproducible.
//
// Backward (ssim_f64_bwd_kernel): the same tile machinery on the 3 or 4 saved maps, then
//   dx1 = g (W'*M0 + 2 x1 W'*M1 + x2 W'*M2),   dx2 = g (W'*M3 + 2 x2 W'*M1 + x1 W'*M2)
// with W' the window rotated by 180 degrees (the adjoint of a zero-padded correlation; the Gaussian window equals it).
// FP64-issue bound, not HBM bound.
#include "common.cuh"

namespace b200w {

namespace f64ssim {
constexpr int kWin = B200W_SSIM_MAX_WINDOW;   // 11
constexpr int kHalo = kWin / 2;               // 5
constexpr int kTW = 64;                       // output columns per CTA tile
constexpr int kR = 8;                         // output rows per thread
constexpr int kTH = kR * (kThreads / kTW);    // 32 output rows per CTA tile
constexpr int kSW = kTW + kWin - 1;           // 74 staged columns
constexpr int kSH = kTH + kWin - 1;           // 42 staged rows
constexpr int kPlaneS = kSW * kSH;            // doubles per staged channel
// options of the MS-SSIM scale instantiations (0: the plain SSIM kernels)
constexpr int kOptCs = 2;     // fwd: the contrast-structure map cs = A2/B2 and its derivative maps instead of S
constexpr int kOptPool = 4;   // fwd: also write avg_pool2d(img1, 2) and avg_pool2d(img2, 2)
constexpr int kOptUp = 8;     // bwd: add 0.25 up[r/2][c/2] (the transpose of that pooling) to d1 / d2
}  // namespace f64ssim

struct SsimF64Params {
    const double* in[4];     // fwd: img1, img2 ; bwd: maps 0..3
    const double* img1;      // bwd epilogue
    const double* img2;
    const double* grad_out;
    double* out0;            // fwd: maps base (or null) ; bwd: d1
    double* out1;            // bwd: d2 (or null)
    double* partials;        // fwd: one double per CTA
    long long plane_elems;   // H*W
    long long map_stride;    // planes*H*W
    int C, H, W, tiles_x, tiles_y;
    int n_maps, size_average;
    double inv_count;        // bwd: 1/(N*C*H*W) or 1/(C*H*W)
    double win[f64ssim::kWin * f64ssim::kWin];   // [dy][dx], a smaller window centred with zero outer taps
    // MS-SSIM scale fields, after the plain SSIM ones so that those keep their parameter offsets
    double* pooled1;         // fwd (kOptPool): (planes, Hp, Wp)
    double* pooled2;
    const double* up1;       // bwd (kOptUp): (planes, Hp, Wp) or null
    const double* up2;
    int Hp, Wp;              // H / 2, W / 2
};

// stage rows [Y0-5, Y0+37) x cols [X0-5, X0+69) of one plane into dst[kSH][kSW], zero outside the image
__device__ __forceinline__ void stage_tile_f64(unsigned dst_s, const double* __restrict__ src, int Y0, int X0, int H,
                                               int W, int tid) {
    using namespace f64ssim;
    for (int idx = tid; idx < kPlaneS; idx += kThreads) {
        const int r = idx / kSW, c = idx - r * kSW;
        const int gr = Y0 - kHalo + r, gc = X0 - kHalo + c;
        const unsigned d = dst_s + (unsigned)(idx * 8);
        const float* s = reinterpret_cast<const float*>(src + (long long)gr * W + gc);
        if (gr >= 0 && gr < H && gc >= 0 && gc < W) cp_async<2>(d, s);
        else cp_async_zero<2>(d, reinterpret_cast<const float*>(src));
    }
}

// acc[m][i] = sum_{dy,dx} win[dy][dx] * ch_m[row 8s + i + dy][col c + dx] for the NCH staged channels
template <int NCH>
__device__ __forceinline__ void blur_column(const double* sm, const SsimF64Params& p, int c, int s,
                                            double (&acc)[NCH][f64ssim::kR]) {
    using namespace f64ssim;
#pragma unroll
    for (int m = 0; m < NCH; ++m)
#pragma unroll
        for (int i = 0; i < kR; ++i) acc[m][i] = 0.0;
#pragma unroll 1
    for (int dx = 0; dx < kWin; ++dx) {
        double w[kWin];
#pragma unroll
        for (int d = 0; d < kWin; ++d) w[d] = p.win[d * kWin + dx];
#pragma unroll
        for (int m = 0; m < NCH; ++m) {
            const double* col = sm + m * kPlaneS + (kR * s) * kSW + c + dx;
#pragma unroll
            for (int j = 0; j < kR + kWin - 1; ++j) {
                const double v = col[j * kSW];
#pragma unroll
                for (int i = 0; i < kR; ++i) {
                    const int d = j - i;
                    if (d >= 0 && d < kWin) acc[m][i] = fma(w[d], v, acc[m][i]);
                }
            }
        }
    }
}

__device__ __forceinline__ double block_sum_f64(double v, double* red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < kThreads / 32; ++i) t += red[i];
    return t;
}

template <int OPT = 0>
__global__ void __launch_bounds__(kThreads, 2) ssim_f64_kernel(const __grid_constant__ SsimF64Params p) {
    using namespace f64ssim;
    extern __shared__ __align__(16) double sm[];   // [4][kSH][kSW]: x1, x2, x1^2 + x2^2, x1 x2
    __shared__ double red[kThreads / 32];
    const int tid = threadIdx.x;
    int bid = blockIdx.x;
    const int tx = bid % p.tiles_x;
    bid /= p.tiles_x;
    const int ty = bid % p.tiles_y;
    const int plane = bid / p.tiles_y;
    const int X0 = tx * kTW, Y0 = ty * kTH, H = p.H, W = p.W;
    const long long poff = (long long)plane * p.plane_elems;

    const unsigned sm_s = (unsigned)__cvta_generic_to_shared(sm);
    stage_tile_f64(sm_s, p.in[0] + poff, Y0, X0, H, W, tid);
    stage_tile_f64(sm_s + kPlaneS * 8, p.in[1] + poff, Y0, X0, H, W, tid);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    for (int idx = tid; idx < kPlaneS; idx += kThreads) {
        // explicit roundings: for img1 == img2 the merged channel is exactly 2 x1 x2, so A1 == B1 and A2 == B2 below
        const double a = sm[idx], b = sm[kPlaneS + idx];
        sm[2 * kPlaneS + idx] = __dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b));
        sm[3 * kPlaneS + idx] = __dmul_rn(a, b);
    }
    if constexpr ((OPT & kOptPool) != 0) {
        // 2x2 average pools of the tile (Y0, X0 even): pooled (Y0/2 + k, X0/2 + pc) from staged rows 2k+5, 2k+6 and
        // columns 2pc+5, 2pc+6, summed in avg_pool2d's order
        const long long pplane = (long long)plane * p.Hp * p.Wp;
        for (int it = tid; it < (kTH / 2) * (kTW / 2); it += kThreads) {
            const int k = it / (kTW / 2), pc = it % (kTW / 2);
            if (Y0 + 2 * k + 1 >= H || X0 + 2 * pc + 1 >= W) continue;
            const long long o = pplane + (long long)(Y0 / 2 + k) * p.Wp + X0 / 2 + pc;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const double* t = sm + i * kPlaneS + (2 * k + kHalo) * kSW + 2 * pc + kHalo;
                (i == 0 ? p.pooled1 : p.pooled2)[o] = (((t[0] + t[1]) + t[kSW]) + t[kSW + 1]) * 0.25;
            }
        }
    }
    __syncthreads();

    const int c = tid % kTW, s = tid / kTW;
    double acc[4][kR];
    blur_column<4>(sm, p, c, s, acc);

    double local = 0.0;
    const int col = X0 + c, row0 = Y0 + kR * s;
    if (col < W) {
        double* m0 = p.out0 ? p.out0 + poff + (long long)row0 * W + col : nullptr;
        const long long ms = p.map_stride;
#pragma unroll
        for (int i = 0; i < kR; ++i) {
            if (row0 + i < H) {
                const double C1 = 0.0001, C2 = 0.0009;   // 0.01^2, 0.03^2 (ssim.py:29-30) as the reference's doubles
                const double mu1 = acc[0][i], mu2 = acc[1][i];
                const double mu12 = __dmul_rn(mu1, mu2);
                const double msum = __dadd_rn(__dmul_rn(mu1, mu1), __dmul_rn(mu2, mu2));
                const double s12 = __dsub_rn(acc[3][i], mu12);
                const double ssum = __dsub_rn(acc[2][i], msum);   // sigma1^2 + sigma2^2
                const double A1 = __fma_rn(2.0, mu12, C1), A2 = __fma_rn(2.0, s12, C2);
                const double B1 = __dadd_rn(msum, C1), B2 = __dadd_rn(ssum, C2);
                if constexpr ((OPT & kOptCs) != 0) {
                    const double cs = __ddiv_rn(A2, B2);   // exactly 1 where A2 == B2
                    local += cs;
                    if (p.n_maps) {
                        const double ib = 1.0 / B2;
                        m0[0] = 2.0 * (mu1 * cs - mu2) * ib;                       // M0 = dcs/dmu1
                        m0[ms] = -cs * ib;                                         // M1 = -cs / B2
                        m0[2 * ms] = 2.0 * ib;                                     // M2 = 2 / B2
                        if (p.n_maps == 4) m0[3 * ms] = 2.0 * (mu2 * cs - mu1) * ib;   // M3 = dcs/dmu2
                    }
                    if (m0) m0 += W;
                    continue;
                }
                const double den = __dmul_rn(B1, B2);
                const double S = __ddiv_rn(__dmul_rn(A1, A2), den);
                local += S;
                if (p.n_maps) {
                    const double inv = 1.0 / den;
                    const double k = 2.0 * (A2 - A1) * inv;        // common factor of dS/dmu
                    const double e = 2.0 * S * (B2 - B1) * inv;    // 2 S (1/B1 - 1/B2)
                    m0[0] = mu2 * k - mu1 * e;                     // M0 = dS/dmu1
                    m0[ms] = -S * B1 * inv;                        // M1 = -S / B2
                    m0[2 * ms] = 2.0 * A1 * inv;                   // M2
                    if (p.n_maps == 4) m0[3 * ms] = mu1 * k - mu2 * e;   // M3 = dS/dmu2
                }
            }
            if (m0) m0 += W;
        }
    }
    const double t = block_sum_f64(local, red);
    if (tid == 0) p.partials[blockIdx.x] = t;
}

template <int NC, int OPT = 0>
__global__ void __launch_bounds__(kThreads, 2) ssim_f64_bwd_kernel(const __grid_constant__ SsimF64Params p) {
    using namespace f64ssim;
    extern __shared__ __align__(16) double sm[];   // [NC][kSH][kSW]: the saved maps
    const int tid = threadIdx.x;
    int bid = blockIdx.x;
    const int tx = bid % p.tiles_x;
    bid /= p.tiles_x;
    const int ty = bid % p.tiles_y;
    const int plane = bid / p.tiles_y;
    const int X0 = tx * kTW, Y0 = ty * kTH, H = p.H, W = p.W;
    const long long poff = (long long)plane * p.plane_elems;

    const unsigned sm_s = (unsigned)__cvta_generic_to_shared(sm);
#pragma unroll
    for (int m = 0; m < NC; ++m) stage_tile_f64(sm_s + m * kPlaneS * 8, p.in[m] + poff, Y0, X0, H, W, tid);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();

    const int c = tid % kTW, s = tid / kTW;
    double acc[NC][kR];
    blur_column<NC>(sm, p, c, s, acc);

    const int col = X0 + c, row0 = Y0 + kR * s;
    if (col >= W) return;
    const double g = __ldg(p.grad_out + (p.size_average ? 0 : plane / p.C)) * p.inv_count;
    const long long off = poff + (long long)row0 * W + col;
    double* d2 = NC == 4 ? p.out1 : nullptr;
#pragma unroll
    for (int i = 0; i < kR; ++i) {
        if (row0 + i < H) {
            const long long o = off + (long long)i * W;
            const double x1 = __ldg(p.img1 + o), x2 = __ldg(p.img2 + o);
            if constexpr ((OPT & kOptUp) != 0) {
                const int pr = (row0 + i) >> 1, pc = col >> 1;
                const bool in = pr < p.Hp && pc < p.Wp;
                const long long uo = ((long long)plane * p.Hp + pr) * p.Wp + pc;
                const double u1 = in && p.up1 ? 0.25 * __ldg(p.up1 + uo) : 0.0;
                const double u2 = in && p.up2 ? 0.25 * __ldg(p.up2 + uo) : 0.0;
                p.out0[o] = g * (acc[0][i] + 2.0 * x1 * acc[1][i] + x2 * acc[2][i]) + u1;
                if (NC == 4 && d2) d2[o] = g * (acc[NC - 1][i] + 2.0 * x2 * acc[1][i] + x1 * acc[2][i]) + u2;
            } else {
                p.out0[o] = g * (acc[0][i] + 2.0 * x1 * acc[1][i] + x2 * acc[2][i]);
                if (NC == 4 && d2) d2[o] = g * (acc[NC - 1][i] + 2.0 * x2 * acc[1][i] + x1 * acc[2][i]);
            }
        }
    }
}

// deterministic final reduction: out[n] = (sum of the partials of sample n) * inv_count
__global__ void __launch_bounds__(kThreads) ssim_f64_finalize_kernel(const double* __restrict__ partials, int per_out,
                                                                      double inv_count, double* __restrict__ out) {
    __shared__ double red[kThreads / 32];
    const double* src = partials + (size_t)blockIdx.x * per_out;
    double s = 0.0;
    for (int i = threadIdx.x; i < per_out; i += kThreads) s += src[i];
    const double t = block_sum_f64(s, red);
    if (threadIdx.x == 0) out[blockIdx.x] = t * inv_count;
}

static void tiles_f64(int H, int W, int* tx, int* ty) {
    *tx = (W + f64ssim::kTW - 1) / f64ssim::kTW;
    *ty = (H + f64ssim::kTH - 1) / f64ssim::kTH;
}

// ws x ws HOST doubles -> the 11 x 11 parameter window (centred; rotated by 180 degrees for the backward)
static int fill_window_f64(SsimF64Params& p, const double* win2d, int ws, bool rotate) {
    using namespace f64ssim;
    if (!win2d || ws < 1 || ws > kWin || (ws % 2) == 0) return B200W_ERR_BAD_WINDOW;
    for (int i = 0; i < kWin * kWin; ++i) p.win[i] = 0.0;
    const int shift = (kWin - ws) / 2;
    for (int i = 0; i < ws; ++i)
        for (int j = 0; j < ws; ++j) {
            const double v = rotate ? win2d[(ws - 1 - i) * ws + (ws - 1 - j)] : win2d[i * ws + j];
            p.win[(shift + i) * kWin + shift + j] = v;
        }
    return B200W_OK;
}

template <typename Kernel>
static int launch_f64(Kernel kern, int nch, const SsimF64Params& p, int planes, cudaStream_t st, const char* name) {
    using namespace f64ssim;
    const size_t smem = sizeof(double) * (size_t)nch * kPlaneS;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_last_cuda_error(e);
    const size_t grid = (size_t)planes * p.tiles_y * p.tiles_x;
    kern<<<(unsigned)grid, kThreads, smem, st>>>(p);
    note_launch(name);
    e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

}  // namespace b200w

using namespace b200w;

extern "C" size_t b200w_ssim_workspace_bytes_f64(int N, int C, int H, int W) {
    if (N < 1 || C < 1 || H < 1 || W < 1) return 0;
    int tx, ty;
    tiles_f64(H, W, &tx, &ty);
    return sizeof(double) * (size_t)N * C * tx * ty;
}

extern "C" int b200w_ssim_fwd_f64(const double* img1, const double* img2, int N, int C, int H, int W,
                                  const double* win2d, int ws, int size_average, int n_maps, double* maps, double* out,
                                  void* workspace, size_t workspace_bytes, void* stream) {
    if (!img1 || !img2 || !out) return B200W_ERR_NULL_POINTER;
    if (N < 1 || C < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!(n_maps == 0 || n_maps == 3 || n_maps == 4)) return B200W_ERR_BAD_SHAPE;
    if (n_maps && !maps) return B200W_ERR_NULL_POINTER;
    SsimF64Params p = {};
    int rc = fill_window_f64(p, win2d, ws, false);
    if (rc) return rc;
    const int planes = N * C;
    p.C = C;
    p.H = H;
    p.W = W;
    tiles_f64(H, W, &p.tiles_x, &p.tiles_y);
    const size_t need = b200w_ssim_workspace_bytes_f64(N, C, H, W);
    if (!workspace || workspace_bytes < need) return B200W_ERR_WORKSPACE;
    p.in[0] = img1;
    p.in[1] = img2;
    p.out0 = n_maps ? maps : nullptr;
    p.partials = (double*)workspace;
    p.plane_elems = (long long)H * W;
    p.map_stride = (long long)planes * H * W;
    p.n_maps = n_maps;
    p.size_average = size_average ? 1 : 0;
    cudaStream_t st = (cudaStream_t)stream;
    rc = launch_f64(ssim_f64_kernel<>, 4, p, planes, st, "ssim_f64_kernel");
    if (rc) return rc;
    const int per_plane = p.tiles_x * p.tiles_y;
    const int nout = size_average ? 1 : N;
    const int per_out = size_average ? planes * per_plane : C * per_plane;
    const double inv = size_average ? 1.0 / ((double)N * C * H * W) : 1.0 / ((double)C * H * W);
    ssim_f64_finalize_kernel<<<nout, kThreads, 0, st>>>(p.partials, per_out, inv, out);
    note_launch("ssim_f64_finalize_kernel");
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

extern "C" int b200w_ssim_bwd_f64(const double* img1, const double* img2, const double* maps, int n_maps,
                                  const double* grad_out, int N, int C, int H, int W, const double* win2d, int ws,
                                  int size_average, double* d1, double* d2, void* stream) {
    if (!img1 || !img2 || !maps || !grad_out || !d1) return B200W_ERR_NULL_POINTER;
    if (N < 1 || C < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!(n_maps == 3 || n_maps == 4) || (d2 && n_maps != 4)) return B200W_ERR_BAD_SHAPE;
    SsimF64Params p = {};
    int rc = fill_window_f64(p, win2d, ws, true);
    if (rc) return rc;
    const int planes = N * C;
    p.C = C;
    p.H = H;
    p.W = W;
    tiles_f64(H, W, &p.tiles_x, &p.tiles_y);
    p.plane_elems = (long long)H * W;
    p.map_stride = (long long)planes * H * W;
    // M3 is staged as channel 3 only when d2 is wanted; channels 0..2 are M0, M1, M2 either way
    const int nc = d2 ? 4 : 3;
    for (int i = 0; i < nc; ++i) p.in[i] = maps + (size_t)i * p.map_stride;
    p.img1 = img1;
    p.img2 = img2;
    p.grad_out = grad_out;
    p.out0 = d1;
    p.out1 = d2;
    p.n_maps = n_maps;
    p.size_average = size_average ? 1 : 0;
    p.inv_count = size_average ? 1.0 / ((double)N * C * H * W) : 1.0 / ((double)C * H * W);
    cudaStream_t st = (cudaStream_t)stream;
    if (d2) return launch_f64(ssim_f64_bwd_kernel<4>, 4, p, planes, st, "ssim_f64_bwd_kernel<4>");
    return launch_f64(ssim_f64_bwd_kernel<3>, 3, p, planes, st, "ssim_f64_bwd_kernel<3>");
}

// MS-SSIM, one scale (see b200w_msssim_scale_fwd_f32): the same checks in the same order
extern "C" int b200w_msssim_scale_fwd_f64(const double* img1, const double* img2, int N, int C, int H, int W,
                                          const double* win2d, int ws, int cs, int n_maps, double* maps, double* out,
                                          double* pooled1, double* pooled2, void* workspace, size_t workspace_bytes,
                                          void* stream) {
    if (!img1 || !img2 || !out) return B200W_ERR_NULL_POINTER;
    if (N < 1 || C < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!(n_maps == 0 || n_maps == 3 || n_maps == 4)) return B200W_ERR_BAD_SHAPE;
    if (n_maps && !maps) return B200W_ERR_NULL_POINTER;
    if (!pooled1 != !pooled2) return B200W_ERR_NULL_POINTER;
    const bool pool = pooled1 != nullptr;
    if (pool && (H < 2 || W < 2)) return B200W_ERR_BAD_SHAPE;
    SsimF64Params p = {};
    int rc = fill_window_f64(p, win2d, ws, false);
    if (rc) return rc;
    const int planes = N * C;
    p.C = C;
    p.H = H;
    p.W = W;
    tiles_f64(H, W, &p.tiles_x, &p.tiles_y);
    const size_t need = b200w_ssim_workspace_bytes_f64(N, C, H, W);
    if (!workspace || workspace_bytes < need) return B200W_ERR_WORKSPACE;
    p.in[0] = img1;
    p.in[1] = img2;
    p.out0 = n_maps ? maps : nullptr;
    p.partials = (double*)workspace;
    p.plane_elems = (long long)H * W;
    p.map_stride = (long long)planes * H * W;
    p.n_maps = n_maps;
    p.pooled1 = pooled1;
    p.pooled2 = pooled2;
    p.Hp = H / 2;
    p.Wp = W / 2;
    cudaStream_t st = (cudaStream_t)stream;
    using namespace f64ssim;
    if (cs) rc = pool ? launch_f64(ssim_f64_kernel<kOptCs | kOptPool>, 4, p, planes, st, "ssim_f64_kernel<cs,pool>")
                      : launch_f64(ssim_f64_kernel<kOptCs>, 4, p, planes, st, "ssim_f64_kernel<cs>");
    else rc = pool ? launch_f64(ssim_f64_kernel<kOptPool>, 4, p, planes, st, "ssim_f64_kernel<pool>")
                   : launch_f64(ssim_f64_kernel<>, 4, p, planes, st, "ssim_f64_kernel");
    if (rc) return rc;
    ssim_f64_finalize_kernel<<<N, kThreads, 0, st>>>(p.partials, C * p.tiles_x * p.tiles_y, 1.0 / ((double)C * H * W),
                                                      out);
    note_launch("ssim_f64_finalize_kernel");
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

extern "C" int b200w_msssim_scale_bwd_f64(const double* img1, const double* img2, const double* maps, int n_maps,
                                          const double* grad_out, int N, int C, int H, int W, const double* win2d,
                                          int ws, const double* up1, const double* up2, double* d1, double* d2,
                                          void* stream) {
    if (!img1 || !img2 || !maps || !grad_out || !d1) return B200W_ERR_NULL_POINTER;
    if (N < 1 || C < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!(n_maps == 3 || n_maps == 4) || (d2 && n_maps != 4)) return B200W_ERR_BAD_SHAPE;
    if (up2 && !d2) return B200W_ERR_BAD_SHAPE;
    const bool up = up1 || up2;
    if (up && (H < 2 || W < 2)) return B200W_ERR_BAD_SHAPE;
    SsimF64Params p = {};
    int rc = fill_window_f64(p, win2d, ws, true);
    if (rc) return rc;
    const int planes = N * C;
    p.C = C;
    p.H = H;
    p.W = W;
    tiles_f64(H, W, &p.tiles_x, &p.tiles_y);
    p.plane_elems = (long long)H * W;
    p.map_stride = (long long)planes * H * W;
    const int nc = d2 ? 4 : 3;
    for (int i = 0; i < nc; ++i) p.in[i] = maps + (size_t)i * p.map_stride;
    p.img1 = img1;
    p.img2 = img2;
    p.grad_out = grad_out;
    p.out0 = d1;
    p.out1 = d2;
    p.n_maps = n_maps;
    p.size_average = 0;
    p.inv_count = 1.0 / ((double)C * H * W);
    p.up1 = up1;
    p.up2 = up2;
    p.Hp = H / 2;
    p.Wp = W / 2;
    cudaStream_t st = (cudaStream_t)stream;
    using namespace f64ssim;
    if (d2) return up ? launch_f64(ssim_f64_bwd_kernel<4, kOptUp>, 4, p, planes, st, "ssim_f64_bwd_kernel<4,up>")
                      : launch_f64(ssim_f64_bwd_kernel<4>, 4, p, planes, st, "ssim_f64_bwd_kernel<4>");
    return up ? launch_f64(ssim_f64_bwd_kernel<3, kOptUp>, 3, p, planes, st, "ssim_f64_bwd_kernel<3,up>")
              : launch_f64(ssim_f64_bwd_kernel<3>, 3, p, planes, st, "ssim_f64_bwd_kernel<3>");
}
