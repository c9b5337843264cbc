// Fourier-domain Gaussian frequency split (SURVEY.md 8f row 1): the pointwise kernels around cuFFT.
//
// Replaces utils.py:71-117 of the reference: guais_low_pass / guais_high_pass build a rows x cols mask with two
// Python loops (one exp per pixel, on the host, every call), high_pass / low_pass do fft2 -> fftshift -> * mask ->
// ifftshift -> ifft2 -> abs on ONE image.  Here the mask is never materialised and nothing is shifted: in the
// unshifted layout the shifted index i holds frequency d = i - rows/2, so the mask at FFT bin (u, v) is
//     m = exp(-0.5 (du^2 + dv^2) / r^2),  du = u < rows - rows/2 ? u : u - rows   (same for dv)
// (1 - m for the high pass).  The mask is real and even, so the filtered spectrum of a real image stays Hermitian:
// the half spectrum of rfft2 / irfft2 is enough (half the bytes of the reference's complex fft2), batched over all
// planes.  The FFTs themselves are cuFFT (library); these kernels are the HBM-bound pointwise passes:
//   freq_mask   in place on the (planes, rows, cols/2+1) complex half spectrum: 16 B of traffic per bin
//   abs_sign    y = sign * |x| (low_pass returns -|.|, utils.py:117), optionally keeping sgn(x) for backward
//   sign_mul    backward of abs_sign: g * sign * sgn(x)
// The three are instantiated for float and, for the reference's double mode (complex128 spectra), for double.
#include <type_traits>

#include "common.cuh"

namespace b200w {

// The mask of one bin.  fp32: the fast exponential with 0.5 / r^2 folded into one factor.  fp64 (the reference's
// double mode): the mask is what utils.py stores -- built in numpy float64 as exp(-0.5 d^2 / r^2), 1 - that for the
// high pass, then rounded once to fp32 by torch.from_numpy(mask).float() -- and the complex128 spectrum is multiplied
// by that fp32 value in double.  `rp` is 0.5 / r^2 in fp32 and r^2 in fp64 (numpy divides by r^2).
__device__ __forceinline__ float gauss_mask(int du, int dv, float rp, int highpass) {
    const float m = __expf(-(float)(du * du + dv * dv) * rp);
    return highpass ? 1.f - m : m;
}
__device__ __forceinline__ double gauss_mask(int du, int dv, double rp, int highpass) {
    const double e = exp(-0.5 * ((double)du * du + (double)dv * dv) / rp);
    return (double)(float)(highpass ? 1.0 - e : e);
}

// flat grid-stride loop over the bins of all planes; the mask costs one exp and two small integer divisions per
// bin (an (u, v)-outer / plane-inner variant that evaluates the mask once per bin was slower: its plane-strided
// accesses and 129-bin rows used the memory system worse -- profiles/r01_notes.md).  Z = float2 / double2 bins.
template <class Z, class S>
__global__ void __launch_bounds__(256) freq_mask_kernel(Z* __restrict__ spec, int planes, int rows, int cols, int wh,
                                                        S rp, int highpass) {
    const unsigned per_plane = (unsigned)rows * (unsigned)wh;
    const size_t total = (size_t)per_plane * planes;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const unsigned rem = (unsigned)(idx % per_plane);
        const int u = (int)(rem / (unsigned)wh), v = (int)(rem - (unsigned)u * (unsigned)wh);
        const int du = u < rows - rows / 2 ? u : u - rows;
        const int dv = v < cols - cols / 2 ? v : v - cols;
        const S m = gauss_mask(du, dv, rp, highpass);
        Z z = spec[idx];
        z.x *= m;
        z.y *= m;
        spec[idx] = z;
    }
}

// 16-byte vectors of the abs pass: float4 / double2
template <class T>
using Vec16 = std::conditional_t<std::is_same<T, float>::value, float4, double2>;
__device__ __forceinline__ float4 scaled_abs(float4 a, float s) {
    return make_float4(s * fabsf(a.x), s * fabsf(a.y), s * fabsf(a.z), s * fabsf(a.w));
}
__device__ __forceinline__ double2 scaled_abs(double2 a, double s) { return make_double2(s * fabs(a.x), s * fabs(a.y)); }

template <class T>
__global__ void __launch_bounds__(256) abs_sign_kernel(const Vec16<T>* __restrict__ x, Vec16<T>* __restrict__ y,
                                                       size_t nv, const T* __restrict__ xt, T* __restrict__ yt, size_t n,
                                                       T sign) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (size_t)gridDim.x * blockDim.x)
        y[i] = scaled_abs(x[i], sign);
    if (blockIdx.x == 0)
        for (size_t i = (16 / sizeof(T)) * nv + threadIdx.x; i < n; i += blockDim.x) yt[i] = sign * fabs(xt[i]);
}

// fp32 reads scalars; fp64 reads double2 pairs when all three pointers are 16-byte aligned, and the odd last element
// (or every element of a misaligned call) in the scalar loop
template <class T>
__global__ void __launch_bounds__(256) sign_mul_kernel(const T* __restrict__ g, const T* __restrict__ x,
                                                       T* __restrict__ out, size_t n, T sign) {
    size_t i0 = 0;
    if constexpr (std::is_same<T, double>::value) {
        if ((((uintptr_t)g | (uintptr_t)x | (uintptr_t)out) & 15) == 0) {
            const size_t n2 = n / 2;
            for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (size_t)gridDim.x * blockDim.x) {
                const double2 a = ((const double2*)g)[i], v = ((const double2*)x)[i];
                ((double2*)out)[i] = make_double2(v.x > 0.0 ? sign * a.x : (v.x < 0.0 ? -sign * a.x : 0.0),
                                                  v.y > 0.0 ? sign * a.y : (v.y < 0.0 ? -sign * a.y : 0.0));
            }
            i0 = 2 * n2;
        }
    }
    for (size_t i = i0 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const T v = x[i];
        out[i] = v > T(0) ? sign * g[i] : (v < T(0) ? -sign * g[i] : T(0));
    }
}

// ---- phase_consistency_loss (model.py:36-58): -cos(a_x, a_y), a = m * log|fft2(.)| over one (C, rows, cols) image,
// m the radius-5 Gaussian high-pass mask.  The reference shifts both spectra the same way before flattening, which
// the cosine does not see; the inputs are real, so |F| is even and the half spectrum of rfft2 carries every term:
// a bin of column v stands for itself and its mirror (weight 2) unless it is its own mirror (v = 0, or v = cols/2
// with cols even: weight 1).  Kernel 1: the three sums <a_x,a_y>, <a_x,a_x>, <a_y,a_y> (per-CTA partials in double,
// fixed-order final reduction: bit-reproducible).  Kernel 2: the gradient w.r.t. both half spectra.
__device__ __forceinline__ float phase_mask(unsigned rem, int rows, int cols, int wh, float inv2r2, float* weight) {
    const int u = (int)(rem / (unsigned)wh), v = (int)(rem - (unsigned)u * (unsigned)wh);
    const int du = u < rows - rows / 2 ? u : u - rows;
    *weight = (v == 0 || 2 * v == cols) ? 1.f : 2.f;
    return 1.f - expf(-(float)(du * du + v * v) * inv2r2);
}

__global__ void __launch_bounds__(256) phase_sums_kernel(const float2* __restrict__ fx, const float2* __restrict__ fy,
                                                         int planes, int rows, int cols, int wh, float inv2r2,
                                                         double* __restrict__ partials) {
    const unsigned per_plane = (unsigned)rows * (unsigned)wh;
    const size_t total = (size_t)per_plane * planes;
    double sxy = 0.0, sxx = 0.0, syy = 0.0;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        float w;
        const float m = phase_mask((unsigned)(idx % per_plane), rows, cols, wh, inv2r2, &w);
        const float2 zx = fx[idx], zy = fy[idx];
        const float ax = m * logf(hypotf(zx.x, zx.y)), ay = m * logf(hypotf(zy.x, zy.y));
        sxy += (double)(w * ax * ay);
        sxx += (double)(w * ax * ax);
        syy += (double)(w * ay * ay);
    }
    __shared__ double red[3][8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sxy += __shfl_xor_sync(0xffffffffu, sxy, o);
        sxx += __shfl_xor_sync(0xffffffffu, sxx, o);
        syy += __shfl_xor_sync(0xffffffffu, syy, o);
    }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = sxy; red[1][threadIdx.x >> 5] = sxx; red[2][threadIdx.x >> 5] = syy; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int i = 0; i < 8; ++i) t += red[threadIdx.x][i];
        partials[3 * blockIdx.x + threadIdx.x] = t;
    }
}

__global__ void phase_finalize_kernel(const double* __restrict__ partials, int nblocks, float* __restrict__ out3) {
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int i = 0; i < nblocks; ++i) t += partials[3 * i + threadIdx.x];
        out3[threadIdx.x] = (float)t;
    }
}

// L = -sxy / (nx ny), nx = max(sqrt(sxx), eps): dL/da_x = -(a_y - (sxy / nx^2) a_x) / (nx ny) (the norm term only while
// nx > eps); a = m log|F| gives dL/dF = dL/da * m * F / |F|^2 in the (d/dRe + i d/dIm) convention autograd uses.
__global__ void __launch_bounds__(256) phase_grad_kernel(const float2* __restrict__ fx, const float2* __restrict__ fy,
                                                         int planes, int rows, int cols, int wh, float inv2r2,
                                                         const float* __restrict__ sums3, const float* __restrict__ grad_out,
                                                         float eps, float2* __restrict__ gx, float2* __restrict__ gy) {
    const unsigned per_plane = (unsigned)rows * (unsigned)wh;
    const size_t total = (size_t)per_plane * planes;
    const float sxy = sums3[0];
    const float rx = sqrtf(sums3[1]), ry = sqrtf(sums3[2]);
    const float nx = fmaxf(rx, eps), ny = fmaxf(ry, eps);
    const float c = -grad_out[0] / (nx * ny);
    const float kx = rx > eps ? sxy / (nx * nx) : 0.f, ky = ry > eps ? sxy / (ny * ny) : 0.f;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        float w;
        const float m = phase_mask((unsigned)(idx % per_plane), rows, cols, wh, inv2r2, &w);
        const float2 zx = fx[idx], zy = fy[idx];
        const float hx = hypotf(zx.x, zx.y), hy = hypotf(zy.x, zy.y);
        const float ax = m * logf(hx), ay = m * logf(hy);
        const float tx = c * w * m * (ay - kx * ax) / (hx * hx);
        const float ty = c * w * m * (ax - ky * ay) / (hy * hy);
        if (gx) gx[idx] = make_float2(tx * zx.x, tx * zx.y);
        if (gy) gy[idx] = make_float2(ty * zy.x, ty * zy.y);
    }
}

static unsigned pointwise_grid(size_t n) {
    size_t g = (n + 255) / 256;
    const size_t cap = 148 * 8;
    return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

// the fp32 and fp64 entry points: the same checks in the same order
template <class T>
static int freq_mask_run(void* spec, int planes, int rows, int cols, T radius, int highpass, cudaStream_t st) {
    constexpr bool f64 = std::is_same<T, double>::value;
    if (!spec) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || rows < 1 || cols < 1 || !(radius > T(0))) return B200W_ERR_BAD_SHAPE;
    const int wh = cols / 2 + 1;
    if ((long long)rows * wh > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    const size_t total = (size_t)planes * rows * wh;
    using Z = std::conditional_t<f64, double2, float2>;
    freq_mask_kernel<<<pointwise_grid(total), 256, 0, st>>>((Z*)spec, planes, rows, cols, wh,
                                                            f64 ? radius * radius : T(0.5) / (radius * radius),
                                                            highpass ? 1 : 0);
    b200w::note_launch(f64 ? "freq_mask_kernel<double2>" : "freq_mask_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

template <class T>
static int abs_sign_run(const T* x, T* y, size_t n, T sign, cudaStream_t st) {
    if (!x || !y) return B200W_ERR_NULL_POINTER;
    if (n == 0) return B200W_OK;
    const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
    const size_t nv = vec ? n / (16 / sizeof(T)) : 0;
    abs_sign_kernel<T><<<pointwise_grid(nv ? nv : n), 256, 0, st>>>((const Vec16<T>*)x, (Vec16<T>*)y, nv, x, y, n, sign);
    b200w::note_launch(sizeof(T) == 8 ? "abs_sign_kernel<double>" : "abs_sign_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

template <class T>
static int sign_mul_run(const T* g, const T* x, T* out, size_t n, T sign, cudaStream_t st) {
    if (!g || !x || !out) return B200W_ERR_NULL_POINTER;
    if (n == 0) return B200W_OK;
    sign_mul_kernel<T><<<pointwise_grid(sizeof(T) == 8 ? (n + 1) / 2 : n), 256, 0, st>>>(g, x, out, n, sign);
    b200w::note_launch(sizeof(T) == 8 ? "sign_mul_kernel<double>" : "sign_mul_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

}  // namespace b200w

using namespace b200w;

extern "C" int b200w_freq_mask_c64(void* spec, int planes, int rows, int cols, float radius, int highpass, void* stream) {
    return freq_mask_run(spec, planes, rows, cols, radius, highpass, (cudaStream_t)stream);
}

extern "C" int b200w_abs_sign_f32(const float* x, float* y, size_t n, float sign, void* stream) {
    return abs_sign_run(x, y, n, sign, (cudaStream_t)stream);
}

extern "C" int b200w_sign_mul_f32(const float* g, const float* x, float* out, size_t n, float sign, void* stream) {
    return sign_mul_run(g, x, out, n, sign, (cudaStream_t)stream);
}

extern "C" int b200w_freq_mask_c128(void* spec, int planes, int rows, int cols, double radius, int highpass,
                                    void* stream) {
    return freq_mask_run(spec, planes, rows, cols, radius, highpass, (cudaStream_t)stream);
}

extern "C" int b200w_abs_sign_f64(const double* x, double* y, size_t n, double sign, void* stream) {
    return abs_sign_run(x, y, n, sign, (cudaStream_t)stream);
}

extern "C" int b200w_sign_mul_f64(const double* g, const double* x, double* out, size_t n, double sign, void* stream) {
    return sign_mul_run(g, x, out, n, sign, (cudaStream_t)stream);
}

extern "C" size_t b200w_phase_workspace_bytes(int planes, int rows, int cols) {
    if (planes < 1 || rows < 1 || cols < 1) return 0;
    return sizeof(double) * 3 * pointwise_grid((size_t)planes * rows * (cols / 2 + 1));
}

extern "C" int b200w_phase_sums_c64(const void* fx, const void* fy, int planes, int rows, int cols, float radius,
                                    void* workspace, size_t workspace_bytes, float* out3, void* stream) {
    if (!fx || !fy || !out3) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || rows < 1 || cols < 1 || !(radius > 0.f)) return B200W_ERR_BAD_SHAPE;
    const int wh = cols / 2 + 1;
    if ((long long)rows * wh > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    const size_t total = (size_t)planes * rows * wh;
    const unsigned grid = pointwise_grid(total);
    if (!workspace || workspace_bytes < sizeof(double) * 3 * grid) return B200W_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    phase_sums_kernel<<<grid, 256, 0, st>>>((const float2*)fx, (const float2*)fy, planes, rows, cols, wh,
                                            0.5f / (radius * radius), (double*)workspace);
    b200w::note_launch("phase_sums_kernel");
    phase_finalize_kernel<<<1, 32, 0, st>>>((const double*)workspace, (int)grid, out3);
    b200w::note_launch("phase_finalize_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

extern "C" int b200w_phase_grad_c64(const void* fx, const void* fy, int planes, int rows, int cols, float radius,
                                    const float* sums3, const float* grad_out, float eps, void* gx, void* gy,
                                    void* stream) {
    if (!fx || !fy || !sums3 || !grad_out || (!gx && !gy)) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || rows < 1 || cols < 1 || !(radius > 0.f)) return B200W_ERR_BAD_SHAPE;
    const int wh = cols / 2 + 1;
    if ((long long)rows * wh > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    const size_t total = (size_t)planes * rows * wh;
    phase_grad_kernel<<<pointwise_grid(total), 256, 0, (cudaStream_t)stream>>>(
        (const float2*)fx, (const float2*)fy, planes, rows, cols, wh, 0.5f / (radius * radius), sums3, grad_out, eps,
        (float2*)gx, (float2*)gy);
    b200w::note_launch("phase_grad_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}
