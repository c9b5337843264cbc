// 1-D analysis / synthesis filter banks (SURVEY.md 8f row 3) for sm_100a.
//
// Replace the bodies of AFB1D.forward / SFB1D.forward (pw/dwt/lowlevel.py:389-405, 719-730: afb1d / sfb1d, :91-172 and
// :226-271, on an (N, C, 1, L) view -- gather padding + F.conv2d with stride (1,2) + two strided .contiguous() copies /
// two F.conv_transpose2d + add) and, with the other bank's taps, each other's hand-written backward (:407-424,
// :732-743).  The 2-D kernels of this library always decimate both axes, so the 1-D transform has its own pair.
// Both are one pass over the data, HBM-bound: a thread owns one output position of one signal, reads its L-tap window
// through the read-only path (adjacent threads read windows that overlap by L - 2 samples: the loads coalesce and hit
// L1), and writes lo / hi (analysis) or y (synthesis) with coalesced 32-bit stores.  Windows that leave the signal take
// the same index maps as the 2-D kernels (ext_index / coef_index, common.cuh): zero, symmetric, reflect, periodic,
// periodization.  Algorithmic bytes: 8 B per input sample (4 read + 4 written) for either direction.
#include "common.cuh"

namespace b200w {

// T = float, or double for the reference's fp64 mode (modules built under torch.set_default_dtype(torch.float64))
template <typename T>
struct Dwt1dParams {
    const T* a;            // analysis: x ; synthesis: lo
    const T* b;            // synthesis: hi (or null = zeros)
    T* o0;                 // analysis: lo ; synthesis: y
    T* o1;                 // analysis: hi
    long long a_rs;        // row stride of `a` in elements (views: the 'unpad' crop of DWT1DInverse is free)
    int rows, n, m, off, mode, L, periodic;   // n = signal length (analysis in / synthesis out), m = coefficients
    T t0[kMaxTaps], t1[kMaxTaps];
};

template <typename T>
__global__ void __launch_bounds__(kThreads) afb1d_kernel(const __grid_constant__ Dwt1dParams<T> p) {
    // rows on grid.y, positions on grid.x: no 64-bit division per output
    for (int row = blockIdx.y; row < p.rows; row += gridDim.y)
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < p.m; k += gridDim.x * blockDim.x) {
        const size_t idx = (size_t)row * p.m + k;
        const T* __restrict__ xr = p.a + (long long)row * p.a_rs;
        const int s0 = 2 * k - p.off;
        T lo = 0, hi = 0;
        if (s0 >= 0 && s0 + p.L <= p.n) {            // interior window: no index maps
#pragma unroll 4
            for (int j = 0; j < p.L; ++j) {
                const T v = __ldg(xr + s0 + j);
                lo = fma(p.t0[j], v, lo);
                hi = fma(p.t1[j], v, hi);
            }
        } else {
            for (int j = 0; j < p.L; ++j) {
                const int s = ext_index(s0 + j, p.n, p.mode);
                if (s < 0) continue;
                const T v = __ldg(xr + s);
                lo = fma(p.t0[j], v, lo);
                hi = fma(p.t1[j], v, hi);
            }
        }
        p.o0[idx] = lo;
        p.o1[idx] = hi;
    }
}

// "A-space" as in the 2-D synthesis kernels: a = i + off, y[i] = sum_{t = a&1, a&1+2, ..} c[(a - t) / 2] g[t].
// The even output a = 2q and the odd output a = 2q + 1 read the same coefficients c[q - u], u = 0 .. L/2 (even taps /
// odd taps), so a thread owns the pair q: one set of loads, two outputs.
template <typename T>
__global__ void __launch_bounds__(kThreads) sfb1d_kernel(const __grid_constant__ Dwt1dParams<T> p) {
    const int q0 = p.off >> 1;                               // pair of output i = 0 (a = off)
    const int npairs = ((p.n - 1 + p.off) >> 1) - q0 + 1;    // pairs covering outputs 0 .. n-1
    const int H2 = (p.L + 1) / 2;
    for (int row = blockIdx.y; row < p.rows; row += gridDim.y)
    for (int pq = blockIdx.x * blockDim.x + threadIdx.x; pq < npairs; pq += gridDim.x * blockDim.x) {
        const int q = q0 + pq;
        const T* __restrict__ lo = p.a + (long long)row * p.a_rs;
        const T* __restrict__ hi = p.b ? p.b + (size_t)row * p.m : nullptr;
        T y0 = 0, y1 = 0;
        if (q - (H2 - 1) >= 0 && q < p.m) {                  // interior: every coefficient exists
            for (int u = 0; u < H2; ++u) {
                const T cl = __ldg(lo + q - u);
                const T g0e = p.t0[2 * u], g0o = 2 * u + 1 < p.L ? p.t0[2 * u + 1] : T(0);
                y0 = fma(cl, g0e, y0);
                y1 = fma(cl, g0o, y1);
                if (hi) {
                    const T ch = __ldg(hi + q - u);
                    const T g1e = p.t1[2 * u], g1o = 2 * u + 1 < p.L ? p.t1[2 * u + 1] : T(0);
                    y0 = fma(ch, g1e, y0);
                    y1 = fma(ch, g1o, y1);
                }
            }
        } else {
            for (int u = 0; u < H2; ++u) {
                const int k = coef_index(q - u, p.m, p.periodic != 0);
                if (k < 0) continue;
                const T cl = __ldg(lo + k);
                const T ch = hi ? __ldg(hi + k) : T(0);
                y0 = fma(cl, p.t0[2 * u], y0);
                y0 = fma(ch, p.t1[2 * u], y0);
                if (2 * u + 1 < p.L) {
                    y1 = fma(cl, p.t0[2 * u + 1], y1);
                    y1 = fma(ch, p.t1[2 * u + 1], y1);
                }
            }
        }
        const int i0 = 2 * q - p.off;
        T* yr = p.o0 + (size_t)row * p.n;
        if (i0 >= 0 && i0 < p.n) yr[i0] = y0;
        if (i0 + 1 >= 0 && i0 + 1 < p.n) yr[i0 + 1] = y1;
    }
}

// grid.x covers the positions of one signal, grid.y the signals (the kernels loop over what the limits cut off): many
// small CTAs balance better here than one resident wave of looping ones (measured: 136 vs 213 us at 64 x 2^20, db3)
static dim3 grid_1d(int positions, int rows) {
    unsigned gx = (unsigned)((positions + kThreads - 1) / kThreads);
    if (gx < 1) gx = 1;
    unsigned gy = (unsigned)rows;
    if (gy > 65535) gy = 65535;
    return dim3(gx, gy, 1);
}

static bool mode_ok(int mode) {
    return mode == B200W_MODE_ZERO || mode == B200W_MODE_SYMMETRIC || mode == B200W_MODE_PERIODIZATION ||
           mode == B200W_MODE_REFLECT || mode == B200W_MODE_PERIODIC;
}

// the fp32 and fp64 entry points share their checks (same codes, same order) and their launch
template <typename T>
static int afb1d_run(const T* x, int64_t x_rs, int rows, int n, const T* h0, const T* h1, int L, int mode, T* lo, T* hi,
                     void* stream) {
    if (!x || !h0 || !h1 || !lo || !hi) return B200W_ERR_NULL_POINTER;
    if (!mode_ok(mode)) return B200W_ERR_BAD_MODE;
    if (rows < 1 || n < 1) return B200W_ERR_BAD_SHAPE;
    if (L < 1 || L > kMaxTaps) return B200W_ERR_BAD_TAPS;
    Dwt1dParams<T> p = {};
    const bool per = mode == B200W_MODE_PERIODIZATION;
    if (per) {
        if (n + (n & 1) < L) return B200W_ERR_PER_TOO_SHORT;
        p.m = (n + 1) / 2;
        p.off = L - 1 - L / 2;
    } else {
        p.m = (n + L - 1) / 2;
        const int pad = 2 * (p.m - 1) - n + L;
        if (mode == B200W_MODE_REFLECT && pad > 0 && (pad + 1) / 2 >= n) return B200W_ERR_REFLECT_PAD;
        p.off = pad / 2;
    }
    if (p.m < 1) return B200W_ERR_BAD_SHAPE;
    p.a = x;
    p.a_rs = x_rs;
    p.o0 = lo;
    p.o1 = hi;
    p.rows = rows;
    p.n = n;
    p.mode = mode;
    p.L = L;
    p.periodic = per;
    for (int j = 0; j < L; ++j) { p.t0[j] = h0[j]; p.t1[j] = h1[j]; }
    afb1d_kernel<T><<<grid_1d(p.m, rows), kThreads, 0, (cudaStream_t)stream>>>(p);
    note_launch(sizeof(T) == 8 ? "afb1d_kernel<double>" : "afb1d_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

template <typename T>
static int sfb1d_run(const T* lo, int64_t lo_rs, const T* hi, int rows, int m, const T* g0, const T* g1, int L, int mode,
                     int out_len, T* y, void* stream) {
    if (!lo || !g0 || !g1 || !y) return B200W_ERR_NULL_POINTER;
    if (!mode_ok(mode)) return B200W_ERR_BAD_MODE;
    if (rows < 1 || m < 1 || out_len < 1) return B200W_ERR_BAD_SHAPE;
    if (L < 1 || L > kMaxTaps) return B200W_ERR_BAD_TAPS;
    const bool per = mode == B200W_MODE_PERIODIZATION;
    if (per && 2 * m < L) return B200W_ERR_PER_TOO_SHORT;
    if (out_len > (per ? 2 * m : 2 * m - L + 2)) return B200W_ERR_BAD_SHAPE;
    Dwt1dParams<T> p = {};
    p.a = lo;
    p.a_rs = lo_rs;
    p.b = hi;
    p.o0 = y;
    p.rows = rows;
    p.n = out_len;
    p.m = m;
    p.off = per ? L / 2 - 1 : L - 2;
    p.mode = mode;
    p.L = L;
    p.periodic = per;
    for (int j = 0; j < L; ++j) { p.t0[j] = g0[j]; p.t1[j] = g1[j]; }
    sfb1d_kernel<T><<<grid_1d(out_len / 2 + 2, rows), kThreads, 0, (cudaStream_t)stream>>>(p);
    note_launch(sizeof(T) == 8 ? "sfb1d_kernel<double>" : "sfb1d_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

}  // namespace b200w

using namespace b200w;

extern "C" int b200w_afb1d_f32(const float* x, int64_t x_rs, int rows, int n, const float* h0, const float* h1, int L,
                               int mode, float* lo, float* hi, void* stream) {
    return afb1d_run(x, x_rs, rows, n, h0, h1, L, mode, lo, hi, stream);
}

extern "C" int b200w_sfb1d_f32(const float* lo, int64_t lo_rs, const float* hi, int rows, int m, const float* g0,
                               const float* g1, int L, int mode, int out_len, float* y, void* stream) {
    return sfb1d_run(lo, lo_rs, hi, rows, m, g0, g1, L, mode, out_len, y, stream);
}

extern "C" int b200w_afb1d_f64(const double* x, int64_t x_rs, int rows, int n, const double* h0, const double* h1,
                               int L, int mode, double* lo, double* hi, void* stream) {
    return afb1d_run(x, x_rs, rows, n, h0, h1, L, mode, lo, hi, stream);
}

extern "C" int b200w_sfb1d_f64(const double* lo, int64_t lo_rs, const double* hi, int rows, int m, const double* g0,
                               const double* g1, int L, int mode, int out_len, double* y, void* stream) {
    return sfb1d_run(lo, lo_rs, hi, rows, m, g0, g1, L, mode, out_len, y, stream);
}
