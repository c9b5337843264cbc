// Total-variation loss (model.py:17-33, `TVLoss`; used at train.py:98): the two sums of squared forward differences
//     h_tv = sum (x[i+1][j] - x[i][j])^2,   w_tv = sum (x[i][j+1] - x[i][j])^2
// in ONE pass over x (the reference slices x four times, subtracts, squares and reduces: ~10 elementwise passes),
// and the gradient of  a*h_tv + b*w_tv  in one pass.  Bound: HBM (4 B/px forward, 8 B/px backward).
#include "common.cuh"

namespace b200w {

constexpr int kTvThreads = 256;
constexpr int kTvRows = 16;    // rows per CTA strip (one extra row above is re-read: 6 %)

// T = float, or double for the reference's fp64 mode; the per-CTA partials are a pair of T
template <typename T> struct TvPair;
template <> struct TvPair<float> { using type = float2; };
template <> struct TvPair<double> { using type = double2; };
template <typename T> using tv_pair_t = typename TvPair<T>::type;

// CTA = (plane, strip of kTvRows rows); a thread walks down columns j, j + 256, ...: coalesced row segments, the row
// above stays in a register, the rows of a strip are independent loads (unrolled).  Partial sums: warp shuffles, then
// one pair per CTA (reduced later in fixed order).
template <typename T>
__global__ void __launch_bounds__(kTvThreads) tv_fwd_kernel(const T* __restrict__ x, int H, int W, int strips,
                                                             tv_pair_t<T>* __restrict__ partials) {
    const int plane = blockIdx.x / strips, strip = blockIdx.x - plane * strips;
    const int i0 = strip * kTvRows;
    const int nr = min(kTvRows, H - i0);
    const T* xp = x + (size_t)plane * H * W + (size_t)i0 * W;
    T sh = 0, sw = 0;
    for (int j = threadIdx.x; j < W; j += kTvThreads) {
        const bool right = j + 1 < W;
        T v[kTvRows + 1], r[kTvRows];
        v[0] = i0 > 0 ? xp[j - W] : T(0);
#pragma unroll
        for (int k = 0; k < kTvRows; ++k) {
            v[k + 1] = k < nr ? xp[(size_t)k * W + j] : T(0);
            r[k] = (k < nr && right) ? xp[(size_t)k * W + j + 1] : T(0);
        }
#pragma unroll
        for (int k = 0; k < kTvRows; ++k) {
            if (k < nr) {
                if (i0 + k > 0) {
                    const T d = v[k + 1] - v[k];
                    sh = fma(d, d, sh);
                }
                if (right) {
                    const T d = r[k] - v[k + 1];
                    sw = fma(d, d, sw);
                }
            }
        }
    }
    sh = warp_sum(sh);
    sw = warp_sum(sw);
    __shared__ tv_pair_t<T> red[kTvThreads / 32];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = tv_pair_t<T>{sh, sw};
    __syncthreads();
    if (threadIdx.x == 0) {
        T a = 0, b = 0;
        for (int k = 0; k < kTvThreads / 32; ++k) {
            a += red[k].x;
            b += red[k].y;
        }
        partials[blockIdx.x] = tv_pair_t<T>{a, b};
    }
}

// one CTA: the partials in fixed order, in double (deterministic)
template <typename T>
__global__ void __launch_bounds__(kTvThreads) tv_finalize_kernel(const tv_pair_t<T>* __restrict__ partials, int n,
                                                                  T* __restrict__ out) {
    double a = 0.0, b = 0.0;
    for (int k = threadIdx.x; k < n; k += kTvThreads) {
        a += (double)partials[k].x;
        b += (double)partials[k].y;
    }
    __shared__ double ra[kTvThreads], rb[kTvThreads];
    ra[threadIdx.x] = a;
    rb[threadIdx.x] = b;
    __syncthreads();
    for (int s = kTvThreads / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            ra[threadIdx.x] += ra[threadIdx.x + s];
            rb[threadIdx.x] += rb[threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = (T)ra[0];
        out[1] = (T)rb[0];
    }
}

// dx = g * (ch * d h_tv/dx + cw * d w_tv/dx),  d h_tv/dx[i] = 2 (x[i]-x[i-1]) [i>0] - 2 (x[i+1]-x[i]) [i<H-1]
// Same strips as the forward kernel: the column of a thread is walked with the rows above / below in registers.
template <typename T>
__global__ void __launch_bounds__(kTvThreads) tv_bwd_kernel(const T* __restrict__ x, const T* __restrict__ g,
                                                             T ch, T cw, int H, int W, int strips,
                                                             T* __restrict__ dx) {
    const int plane = blockIdx.x / strips, strip = blockIdx.x - plane * strips;
    const int i0 = strip * kTvRows;
    const int nr = min(kTvRows, H - i0);
    const size_t base = (size_t)plane * H * W + (size_t)i0 * W;
    const T* xp = x + base;
    T* dp = dx + base;
    const T gs = g[0];
    const T a = T(2) * ch * gs, b = T(2) * cw * gs;
    for (int j = threadIdx.x; j < W; j += kTvThreads) {
        const bool hasl = j > 0, hasr = j + 1 < W;
        T v[kTvRows + 2], l[kTvRows], r[kTvRows];
        v[0] = i0 > 0 ? xp[j - W] : T(0);
#pragma unroll
        for (int k = 0; k < kTvRows + 1; ++k) v[k + 1] = (i0 + k < H && k <= nr) ? xp[(size_t)k * W + j] : T(0);
#pragma unroll
        for (int k = 0; k < kTvRows; ++k) {
            l[k] = (k < nr && hasl) ? xp[(size_t)k * W + j - 1] : T(0);
            r[k] = (k < nr && hasr) ? xp[(size_t)k * W + j + 1] : T(0);
        }
#pragma unroll
        for (int k = 0; k < kTvRows; ++k) {
            if (k < nr) {
                const int i = i0 + k;
                const T c = v[k + 1];
                T dh = 0, dw = 0;
                if (i > 0) dh += c - v[k];
                if (i + 1 < H) dh -= v[k + 2] - c;
                if (hasl) dw += c - l[k];
                if (hasr) dw -= r[k] - c;
                dp[(size_t)k * W + j] = fma(a, dh, b * dw);
            }
        }
    }
}

// the fp32 and fp64 entry points share their checks (same codes, same order) and their launches
template <typename T>
static int tv_fwd_run(const T* x, int planes, int H, int W, void* workspace, size_t workspace_bytes, T* out2,
                      void* stream, size_t need) {
    if (!x || !out2 || !workspace) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    const int strips = (H + kTvRows - 1) / kTvRows;
    const long long ctas = (long long)planes * strips;
    if (ctas > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    if (workspace_bytes < need) return B200W_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const bool f64 = sizeof(T) == 8;
    tv_fwd_kernel<T><<<(unsigned)ctas, kTvThreads, 0, st>>>(x, H, W, strips, (tv_pair_t<T>*)workspace);
    note_launch(f64 ? "tv_fwd_kernel<double>" : "tv_fwd_kernel");
    tv_finalize_kernel<T><<<1, kTvThreads, 0, st>>>((const tv_pair_t<T>*)workspace, (int)ctas, out2);
    note_launch(f64 ? "tv_finalize_kernel<double>" : "tv_finalize_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

template <typename T>
static int tv_bwd_run(const T* x, const T* grad_out, T ch, T cw, int planes, int H, int W, T* dx, void* stream) {
    if (!x || !grad_out || !dx) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    const int strips = (H + kTvRows - 1) / kTvRows;
    const long long ctas = (long long)planes * strips;
    if (ctas > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    tv_bwd_kernel<T><<<(unsigned)ctas, kTvThreads, 0, (cudaStream_t)stream>>>(x, grad_out, ch, cw, H, W, strips, dx);
    note_launch(sizeof(T) == 8 ? "tv_bwd_kernel<double>" : "tv_bwd_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

static size_t tv_strips_total(int planes, int H) { return (size_t)planes * ((H + kTvRows - 1) / kTvRows); }

}  // namespace b200w

using namespace b200w;

extern "C" size_t b200w_tv_workspace_bytes(int planes, int H) {
    if (planes < 1 || H < 1) return 0;
    return sizeof(float2) * tv_strips_total(planes, H);
}

extern "C" size_t b200w_tv_workspace_bytes_f64(int planes, int H) {
    if (planes < 1 || H < 1) return 0;
    return sizeof(double2) * tv_strips_total(planes, H);
}

extern "C" int b200w_tv_fwd_f32(const float* x, int planes, int H, int W, void* workspace, size_t workspace_bytes,
                                float* out2, void* stream) {
    return tv_fwd_run(x, planes, H, W, workspace, workspace_bytes, out2, stream, b200w_tv_workspace_bytes(planes, H));
}

extern "C" int b200w_tv_bwd_f32(const float* x, const float* grad_out, float ch, float cw, int planes, int H, int W,
                                float* dx, void* stream) {
    return tv_bwd_run(x, grad_out, ch, cw, planes, H, W, dx, stream);
}

extern "C" int b200w_tv_fwd_f64(const double* x, int planes, int H, int W, void* workspace, size_t workspace_bytes,
                                double* out2, void* stream) {
    return tv_fwd_run(x, planes, H, W, workspace, workspace_bytes, out2, stream,
                      b200w_tv_workspace_bytes_f64(planes, H));
}

extern "C" int b200w_tv_bwd_f64(const double* x, const double* grad_out, double ch, double cw, int planes, int H, int W,
                                double* dx, void* stream) {
    return tv_bwd_run(x, grad_out, ch, cw, planes, H, W, dx, stream);
}
