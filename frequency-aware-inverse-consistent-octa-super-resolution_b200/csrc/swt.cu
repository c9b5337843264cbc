// Undecimated ("a trous") 2-D analysis bank (SURVEY.md 8f row 3) for sm_100a: one level of SWTForward.
//
// Replaces afb2d_atrous (pw/dwt/lowlevel.py:475-521 = afb1d_atrous :175-223 along W, then along H: mypad + F.conv2d with
// `dilation`, no stride) and the adjoint autograd derives from it.  With L2 = (L * dilation) / 2 the reference pads
// L2 - dilation samples in front and L2 behind (:218-219), so the output has the input's size and
//     y_b[i][k] = sum_jh sum_jw hH_b[jh] hW_b[jw] x[ext(i + d jh - (L2 - d))][ext(k + d jw - (L2 - d))]
// for the four band combinations b = (lo,lo), (lo,hi) ... in the channel order the two grouped convolutions produce:
// out channel 4c + 2a + e = (row filter a in {lo, hi} along W, then column filter e in {lo, hi} along H) of channel c.
// mypad knows 'zero', 'symmetric', 'reflect' and 'periodic' here ('periodization', SWTForward's default, raises
// "Unkown pad type" in the reference and here).  One thread per output pixel evaluates the separable sum (2 L^2 + 4 L
// FMAs) from the read-only path; the 4 results are stored to the 4 band planes (coalesced along W).  The backward kernel
// is the exact adjoint in gather form: an input sample s collects, for every extended position t that the padding maps
// onto s (t = s itself, its mirror images / periodic images inside the padded range), the taps of all outputs that read
// t.  Both are rarely-used paths (the application does not call SWTForward): simple, correct, HBM-friendly, not tuned.
#include "common.cuh"

namespace b200w {

// T = float, or double for the reference's fp64 mode
template <typename T>
struct SwtParams {
    const T* in;         // forward: x (planes, H, W) ; backward: dy (planes, 4, H, W)
    T* out;              // forward: y (planes, 4, H, W) ; backward: dx (planes, H, W)
    int planes, H, W, L, d, pl, pr, mode;
    T w_lo[kMaxTaps], w_hi[kMaxTaps], h_lo[kMaxTaps], h_hi[kMaxTaps];
};

template <typename T>
__global__ void __launch_bounds__(kThreads) swt2d_fwd_kernel(const __grid_constant__ SwtParams<T> p) {
    const size_t plane_px = (size_t)p.H * p.W;
    // planes on grid.y, pixels of a plane on grid.x with 32-bit index arithmetic (H * W < 2^31 is checked by the host)
    for (int plane = blockIdx.y; plane < p.planes; plane += gridDim.y)
    for (unsigned px = blockIdx.x * blockDim.x + threadIdx.x; px < (unsigned)plane_px; px += gridDim.x * blockDim.x) {
        const int i = (int)(px / (unsigned)p.W);
        const int k = (int)(px - (unsigned)i * (unsigned)p.W);
        const T* __restrict__ xp = p.in + plane * plane_px;
        T ll = 0, lh = 0, hl = 0, hh = 0;   // (row lo, col lo), (row lo, col hi), (row hi, col lo), (row hi, col hi)
        const int r0 = i - p.pl, c0 = k - p.pl, span = p.d * (p.L - 1);
        if (r0 >= 0 && r0 + span < p.H && c0 >= 0 && c0 + span < p.W) {      // interior window: no index maps
            const T* __restrict__ xw = xp + (size_t)r0 * p.W + c0;
            for (int jh = 0; jh < p.L; ++jh) {
                const T* __restrict__ xr = xw + (size_t)(p.d * jh) * p.W;
                T lo = 0, hi = 0;
#pragma unroll 4
                for (int jw = 0; jw < p.L; ++jw) {
                    const T v = __ldg(xr + p.d * jw);
                    lo = fma(p.w_lo[jw], v, lo);
                    hi = fma(p.w_hi[jw], v, hi);
                }
                ll = fma(p.h_lo[jh], lo, ll);
                lh = fma(p.h_hi[jh], lo, lh);
                hl = fma(p.h_lo[jh], hi, hl);
                hh = fma(p.h_hi[jh], hi, hh);
            }
        } else {
            for (int jh = 0; jh < p.L; ++jh) {
                const int r = ext_index(r0 + p.d * jh, p.H, p.mode);
                if (r < 0) continue;
                const T* __restrict__ xr = xp + (size_t)r * p.W;
                T lo = 0, hi = 0;
                for (int jw = 0; jw < p.L; ++jw) {
                    const int c = ext_index(c0 + p.d * jw, p.W, p.mode);
                    if (c < 0) continue;
                    const T v = __ldg(xr + c);
                    lo = fma(p.w_lo[jw], v, lo);
                    hi = fma(p.w_hi[jw], v, hi);
                }
                ll = fma(p.h_lo[jh], lo, ll);
                lh = fma(p.h_hi[jh], lo, lh);
                hl = fma(p.h_lo[jh], hi, hl);
                hh = fma(p.h_hi[jh], hi, hh);
            }
        }
        T* o = p.out + plane * 4 * plane_px + (size_t)i * p.W + k;
        o[0] = ll;
        o[plane_px] = lh;
        o[2 * plane_px] = hl;
        o[3 * plane_px] = hh;
    }
}

// extended positions t in [-pl, n + pr) with ext_index(t, n, mode) == s; returns their count (<= kMaxPre)
constexpr int kMaxPre = 8;
__device__ __forceinline__ int preimages(int s, int n, int pl, int pr, int mode, int* t) {
    int cnt = 0;
    const int lo = -pl, hi = n + pr;   // [lo, hi)
    if (mode == B200W_MODE_ZERO) {
        t[cnt++] = s;
        return cnt;
    }
    int period, mirror;   // images: s + q * period and mirror - s + q * period
    bool has_mirror = true;
    if (mode == B200W_MODE_SYMMETRIC) { period = 2 * n; mirror = -1; }
    else if (mode == B200W_MODE_REFLECT) { period = 2 * n - 2; mirror = 0; if (n == 1) { t[cnt++] = s; return cnt; } }
    else { period = n; mirror = 0; has_mirror = false; }   // periodic
    for (int q = -4; q <= 4; ++q) {
        const int a = s + q * period;
        if (a >= lo && a < hi && cnt < kMaxPre) t[cnt++] = a;
        if (has_mirror) {
            const int b = mirror - s + q * period;
            // reflect: the end points 0 and n-1 are their own mirror images (b == a for some q): count them once
            bool dup = false;
            for (int u = 0; u < cnt; ++u) dup |= t[u] == b;
            if (!dup && b >= lo && b < hi && cnt < kMaxPre) t[cnt++] = b;
        }
    }
    return cnt;
}

template <typename T>
__global__ void __launch_bounds__(kThreads) swt2d_bwd_kernel(const __grid_constant__ SwtParams<T> p) {
    const size_t plane_px = (size_t)p.H * p.W;
    for (int plane = blockIdx.y; plane < p.planes; plane += gridDim.y)
    for (unsigned px = blockIdx.x * blockDim.x + threadIdx.x; px < (unsigned)plane_px; px += gridDim.x * blockDim.x) {
        const int r = (int)(px / (unsigned)p.W);
        const int c = (int)(px - (unsigned)r * (unsigned)p.W);
        const T* __restrict__ g = p.in + plane * 4 * plane_px;
        int tr[kMaxPre], tc[kMaxPre];
        const int nr = preimages(r, p.H, p.pl, p.pr, p.mode, tr);
        const int nc = preimages(c, p.W, p.pl, p.pr, p.mode, tc);
        T acc = 0;
        for (int a = 0; a < nr; ++a) {
            for (int jh = 0; jh < p.L; ++jh) {
                const int i = tr[a] + p.pl - p.d * jh;
                if (i < 0 || i >= p.H) continue;
                T s_lo = 0, s_hi = 0;   // sums over the W taps of (h_lo-weighted, h_hi-weighted) band gradients
                for (int b = 0; b < nc; ++b) {
                    for (int jw = 0; jw < p.L; ++jw) {
                        const int k = tc[b] + p.pl - p.d * jw;
                        if (k < 0 || k >= p.W) continue;
                        const T* q = g + (size_t)i * p.W + k;
                        const T gll = __ldg(q), glh = __ldg(q + plane_px), ghl = __ldg(q + 2 * plane_px),
                                    ghh = __ldg(q + 3 * plane_px);
                        s_lo = fma(p.w_lo[jw], gll, s_lo);
                        s_lo = fma(p.w_hi[jw], ghl, s_lo);
                        s_hi = fma(p.w_lo[jw], glh, s_hi);
                        s_hi = fma(p.w_hi[jw], ghh, s_hi);
                    }
                }
                acc = fma(p.h_lo[jh], s_lo, acc);
                acc = fma(p.h_hi[jh], s_hi, acc);
            }
        }
        p.out[plane * plane_px + px] = acc;
    }
}

static dim3 swt_grid(int planes, size_t plane_px) {
    unsigned gx = (unsigned)((plane_px + kThreads - 1) / kThreads);
    unsigned gy = (unsigned)planes;
    if (gy > 65535) gy = 65535;
    return dim3(gx < 1 ? 1 : gx, gy, 1);
}

template <typename T>
static int swt_fill(SwtParams<T>& p, int planes, int H, int W, const T* w_lo, const T* w_hi, const T* h_lo,
                    const T* h_hi, int L, int dilation, int mode) {
    if (!w_lo || !w_hi || !h_lo || !h_hi) return B200W_ERR_NULL_POINTER;
    if (!(mode == B200W_MODE_ZERO || mode == B200W_MODE_SYMMETRIC || mode == B200W_MODE_REFLECT ||
          mode == B200W_MODE_PERIODIC))
        return B200W_ERR_BAD_MODE;   // mypad has no 'periodization' (pw/dwt/lowlevel.py:28-88)
    if (planes < 1 || H < 1 || W < 1 || dilation < 1 || (long long)H * W > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    if (L < 1 || L > kMaxTaps) return B200W_ERR_BAD_TAPS;
    const int L2 = (L * dilation) / 2;
    p.pl = L2 - dilation;
    p.pr = L2;
    if (p.pl < 0) return B200W_ERR_BAD_TAPS;                       // a single tap: negative padding
    if (mode == B200W_MODE_REFLECT && (p.pr >= H || p.pr >= W)) return B200W_ERR_REFLECT_PAD;   // F.pad's rule
    if (p.pr > 3 * (H < W ? H : W)) return B200W_ERR_BAD_SHAPE;    // the backward enumerates at most 4 periods of images
    p.planes = planes;
    p.H = H;
    p.W = W;
    p.L = L;
    p.d = dilation;
    p.mode = mode;
    for (int j = 0; j < L; ++j) { p.w_lo[j] = w_lo[j]; p.w_hi[j] = w_hi[j]; p.h_lo[j] = h_lo[j]; p.h_hi[j] = h_hi[j]; }
    return B200W_OK;
}

// the fp32 and fp64 entry points share their checks (same codes, same order) and their launch
template <typename T>
static int swt2d_run(bool fwd, const T* in, int planes, int H, int W, const T* w_lo, const T* w_hi, const T* h_lo,
                     const T* h_hi, int L, int dilation, int mode, T* out, void* stream) {
    if (!in || !out) return B200W_ERR_NULL_POINTER;
    SwtParams<T> p = {};
    const int rc = swt_fill(p, planes, H, W, w_lo, w_hi, h_lo, h_hi, L, dilation, mode);
    if (rc) return rc;
    p.in = in;
    p.out = out;
    const dim3 grid = swt_grid(planes, (size_t)H * W);
    const bool f64 = sizeof(T) == 8;
    if (fwd) {
        swt2d_fwd_kernel<T><<<grid, kThreads, 0, (cudaStream_t)stream>>>(p);
        note_launch(f64 ? "swt2d_fwd_kernel<double>" : "swt2d_fwd_kernel");
    } else {
        swt2d_bwd_kernel<T><<<grid, kThreads, 0, (cudaStream_t)stream>>>(p);
        note_launch(f64 ? "swt2d_bwd_kernel<double>" : "swt2d_bwd_kernel");
    }
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

}  // namespace b200w

using namespace b200w;

extern "C" int b200w_swt2d_fwd_f32(const float* x, int planes, int H, int W, const float* w_lo, const float* w_hi,
                                   const float* h_lo, const float* h_hi, int L, int dilation, int mode, float* y,
                                   void* stream) {
    return swt2d_run(true, x, planes, H, W, w_lo, w_hi, h_lo, h_hi, L, dilation, mode, y, stream);
}

extern "C" int b200w_swt2d_bwd_f32(const float* dy, int planes, int H, int W, const float* w_lo, const float* w_hi,
                                   const float* h_lo, const float* h_hi, int L, int dilation, int mode, float* dx,
                                   void* stream) {
    return swt2d_run(false, dy, planes, H, W, w_lo, w_hi, h_lo, h_hi, L, dilation, mode, dx, stream);
}

extern "C" int b200w_swt2d_fwd_f64(const double* x, int planes, int H, int W, const double* w_lo, const double* w_hi,
                                   const double* h_lo, const double* h_hi, int L, int dilation, int mode, double* y,
                                   void* stream) {
    return swt2d_run(true, x, planes, H, W, w_lo, w_hi, h_lo, h_hi, L, dilation, mode, y, stream);
}

extern "C" int b200w_swt2d_bwd_f64(const double* dy, int planes, int H, int W, const double* w_lo, const double* w_hi,
                                   const double* h_lo, const double* h_hi, int L, int dilation, int mode, double* dx,
                                   void* stream) {
    return swt2d_run(false, dy, planes, H, W, w_lo, w_hi, h_lo, h_hi, L, dilation, mode, dx, stream);
}
