// 2-D DWT analysis / synthesis filter banks for sm_100a: kernel selection, the C entry points and the direct kernels.
//
// What it replaces.  Per level the reference runs pad-gather + 2x F.conv2d + reshape + 2x .contiguous()
// (AFB2D, pw/dwt/lowlevel.py:336-347) resp. 6x F.conv_transpose2d + 3 adds (SFB2D, :671-680), and
// DWTForward / DWTInverse loop over the J levels in Python (pw/dwt/transform2d.py:66-74, 134-148).
// Here a J-level transform of up to 16 taps is ONE launch: an owner kernel for chains of small planes
// (dwt_tma_*.cu, dwt_stream_*.cu; analysis: 16-byte aligned rows), otherwise the ticketed stream chain
// (dwt_stream_*.cu), which takes rows of any alignment.
//
// Direct kernels: one thread per output of one level, any tap count, in fp32 and in fp64.
//
// Closed forms (SURVEY.md 8a, validated against the reference to 1e-15 by oracle/dwt_oracle.py):
//   analysis   y_c[k] = sum_j w_c[j] * x_ext[2k + j - off],  off = p//2 with p = 2(M-1) - N + L,
//              periodization: off = L-1 - L//2 on the (even-extended) N'-periodic signal
//   synthesis  y[n]   = sum_k lo[k] g0[t] + hi[k] g1[t],  t = n + off - 2k in [0,L),
//              off = L-2 (coefficients outside [0,M) are zero), periodization: off = L//2 - 1 and the
//              coefficient sequence is M-periodic
//
// These are HBM-bound stencils (8 B of traffic per pixel for 2L FMAs): the code keeps the instruction count
// per pixel low -- 128-bit shared loads feeding register-blocked FMAs whose coefficients come from the
// constant bank, 64-bit coalesced global stores, staging loops whose addresses advance by constants.
#include <type_traits>
#include "dwt_levels.cuh"
#include "dwt_tma.cuh"

namespace b200w {

__global__ void zero_words_kernel(unsigned* w, unsigned n) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) w[i] = 0u;
}

int zero_sync_words(unsigned* words, size_t n, cudaStream_t st) {
    zero_words_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(words, (unsigned)n);
    note_launch("zero_words_kernel");
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

// ------------------------------------------------------------------------------------------------
// direct kernels: one thread per output position of ONE level, no staging, any tap count up to kMaxTaps (odd or
// mixed lengths).  In fp32 they serve the tap counts the templated kernels are not instantiated for (and
// B200W_FORCE_DIRECT); in fp64 they are the whole path -- precision, not speed, is the point there.
// ------------------------------------------------------------------------------------------------
struct Taps64 {
    double w_lo[kMaxTaps], w_hi[kMaxTaps], h_lo[kMaxTaps], h_hi[kMaxTaps];
};
template <class T>
using DirectTaps = std::conditional_t<std::is_same<T, float>::value, Taps, Taps64>;

// The fp32 chain runners fill these from AfbLevel / SfbLevel, the fp64 entry points directly.
template <class T>
struct AfbDirectParams {
    const T* x;
    T* low;
    T* highs;                  // dense (planes,3,Ho,Wo)
    long long x_ps, x_rs, low_ps, low_rs;
    int H, W, Hreal, Wreal;    // as in AfbLevel
    int Ho, Wo, offH, offW;
    int st_low, st_hi;         // store epilogue of AfbLevel
    T hi_scale, hi_shift;
    int planes, mode, Lw, Lh;
    DirectTaps<T> t;
};

template <class T>
__global__ void __launch_bounds__(kThreads) afb2d_direct_kernel(const __grid_constant__ AfbDirectParams<T> p) {
    const size_t band = (size_t)p.Ho * p.Wo;
    const size_t total = band * p.planes;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(idx % p.Wo);
        const int i = (int)((idx / p.Wo) % p.Ho);
        const int plane = (int)(idx / band);
        const T* __restrict__ xp = p.x + (long long)plane * p.x_ps;
        T ll = 0, lh = 0, hl = 0, hh = 0;
        for (int jh = 0; jh < p.Lh; ++jh) {
            const int sr = ext_index(2 * i + jh - p.offH, p.H, p.mode);
            if (sr < 0 || sr >= p.Hreal) continue;
            T lo = 0, hi = 0;
            for (int jw = 0; jw < p.Lw; ++jw) {
                const int sc = ext_index(2 * k + jw - p.offW, p.W, p.mode);
                if (sc < 0 || sc >= p.Wreal) continue;
                const T v = __ldg(xp + (long long)sr * p.x_rs + sc);
                lo = fma(p.t.w_lo[jw], v, lo);
                hi = fma(p.t.w_hi[jw], v, hi);
            }
            ll = fma(p.t.h_lo[jh], lo, ll);
            lh = fma(p.t.h_hi[jh], lo, lh);
            hl = fma(p.t.h_lo[jh], hi, hl);
            hh = fma(p.t.h_hi[jh], hi, hh);
        }
        const size_t o = (size_t)i * p.Wo + k;
        if (p.st_low) p.low[(long long)plane * p.low_ps + (long long)i * p.low_rs + k] = ll;
        if (p.st_hi) {
            T* hip = p.highs + (size_t)plane * 3 * band + o;
            hip[0] = fma(lh, p.hi_scale, p.hi_shift);
            hip[band] = fma(hl, p.hi_scale, p.hi_shift);
            hip[2 * band] = fma(hh, p.hi_scale, p.hi_shift);
        }
    }
}

template <class T>
struct SfbDirectParams {
    const T* low;
    const T* highs;            // dense (planes,3,h,w); may be null (= zeros)
    T* y;
    long long low_ps, low_rs, y_ps, y_rs;
    int h, w, out_h, out_w, offH, offW;
    int planes, periodic, Lw, Lh;
    DirectTaps<T> t;
};

// "A-space" as in the other synthesis kernels: a = n + off; output a uses the taps of parity a & 1
template <class T>
__global__ void __launch_bounds__(kThreads) sfb2d_direct_kernel(const __grid_constant__ SfbDirectParams<T> p) {
    const size_t total = (size_t)p.planes * p.out_h * p.out_w;
    const size_t band = (size_t)p.h * p.w;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int nW = (int)(idx % p.out_w);
        const int nH = (int)((idx / p.out_w) % p.out_h);
        const int plane = (int)(idx / ((size_t)p.out_h * p.out_w));
        const T* __restrict__ lowp = p.low + (long long)plane * p.low_ps;
        const T* __restrict__ hip = p.highs ? p.highs + (size_t)plane * 3 * band : nullptr;
        const int AH = nH + p.offH, AW = nW + p.offW;
        T y = 0;
        for (int tH = AH & 1; tH < p.Lh; tH += 2) {
            const int kr = coef_index((AH - tH) / 2, p.h, p.periodic);
            if (kr < 0) continue;
            T lo = 0, hi = 0;  // W-synthesised values to be combined with h_lo / h_hi
            for (int tW = AW & 1; tW < p.Lw; tW += 2) {
                const int kc = coef_index((AW - tW) / 2, p.w, p.periodic);
                if (kc < 0) continue;
                const T ll = __ldg(lowp + (long long)kr * p.low_rs + kc);
                lo = fma(ll, p.t.w_lo[tW], lo);
                if (hip) {
                    const T* q = hip + (size_t)kr * p.w + kc;
                    hi = fma(__ldg(q), p.t.w_lo[tW], hi);               // LH
                    lo = fma(__ldg(q + band), p.t.w_hi[tW], lo);        // HL
                    hi = fma(__ldg(q + 2 * band), p.t.w_hi[tW], hi);    // HH
                }
            }
            y = fma(lo, p.t.h_lo[tH], y);
            y = fma(hi, p.t.h_hi[tH], y);
        }
        p.y[(long long)plane * p.y_ps + (long long)nH * p.y_rs + nW] = y;
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static bool mode_supported(int mode) {
    return mode == B200W_MODE_ZERO || mode == B200W_MODE_SYMMETRIC || mode == B200W_MODE_PERIODIZATION ||
           mode == B200W_MODE_REFLECT || mode == B200W_MODE_PERIODIC;
}

// copies the taps into a kernel's tap block, zero beyond Lw / Lh
template <class T>
static int fill_taps(DirectTaps<T>& t, const T* w_lo, const T* w_hi, int Lw, const T* h_lo, const T* h_hi, int Lh) {
    if (Lw < 1 || Lw > kMaxTaps || Lh < 1 || Lh > kMaxTaps || !w_lo || !w_hi || !h_lo || !h_hi)
        return B200W_ERR_BAD_TAPS;
    for (int i = 0; i < kMaxTaps; ++i) {
        t.w_lo[i] = i < Lw ? w_lo[i] : T(0);
        t.w_hi[i] = i < Lw ? w_hi[i] : T(0);
        t.h_lo[i] = i < Lh ? h_lo[i] : T(0);
        t.h_hi[i] = i < Lh ? h_hi[i] : T(0);
    }
    if constexpr (std::is_same<T, float>::value) {
        for (int i = 0; i < kMaxTemplTaps; ++i) {
            t.h_lo2[i] = make_float2(t.h_lo[i], t.h_lo[i]);
            t.h_hi2[i] = make_float2(t.h_hi[i], t.h_hi[i]);
        }
    }
    return B200W_OK;
}

static int coeff_len(int n, int l, int mode) { return mode == B200W_MODE_PERIODIZATION ? (n + 1) / 2 : (n + l - 1) / 2; }
static int idwt_len(int m, int l, int mode) { return mode == B200W_MODE_PERIODIZATION ? 2 * m : 2 * m - l + 2; }

// left padding of the analysis bank along one axis; also validates the axis
static int analysis_offset(int n, int l, int mode, int* off) {
    if (mode == B200W_MODE_PERIODIZATION) {
        if (n + (n & 1) < l) return B200W_ERR_PER_TOO_SHORT;
        *off = l - 1 - l / 2;
        return B200W_OK;
    }
    const int m = coeff_len(n, l, mode);
    const int p = 2 * (m - 1) - n + l;
    if (mode == B200W_MODE_REFLECT && p > 0 && (p + 1) / 2 >= n) return B200W_ERR_REFLECT_PAD;
    *off = p / 2;
    return B200W_OK;
}

// A-space offset of the synthesis bank along one axis
static int synthesis_offset(int l, int mode) { return mode == B200W_MODE_PERIODIZATION ? l / 2 - 1 : l - 2; }

constexpr int kMaxDevices = 64;

// SM count of the current device, queried once per device
static int device_sms() {
    static int sms[kMaxDevices] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 148;
    if (sms[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        sms[dev] = n;
    }
    return sms[dev];
}

// Workspace layout of a J-level chain: [ticket, done[J][planes]] (u32), then the intermediate low-pass images
// (planes x rows x pitch floats, pitch = columns rounded up to 4 so that every row is 16-byte aligned), each
// region rounded up to 256 bytes.  The caller's pointer must be 256-byte aligned (torch allocations are).
static size_t round256(size_t n) { return (n + 255) & ~(size_t)255; }
static size_t sync_bytes(int planes, int J) { return J > 1 ? round256(sizeof(unsigned) * ((size_t)J * planes + 1)) : 0; }
static int pitch4(int w) { return (w + 3) & ~3; }
static size_t scratch_bytes(int planes, int rows, int cols) {
    return round256(sizeof(float) * (size_t)planes * rows * pitch4(cols));
}

static size_t direct_grid(size_t total) {
    size_t g = (total + kThreads - 1) / kThreads;
    const size_t cap = 148 * 16;
    return g < 1 ? 1 : (g > cap ? cap : g);
}

// one launch of a direct kernel; `outputs` = output positions over all planes
template <class Params>
static int launch_direct(void (*kernel)(Params), const Params& d, size_t outputs, const char* name, cudaStream_t st) {
    kernel<<<(unsigned)direct_grid(outputs), kThreads, 0, st>>>(d);
    note_launch(name);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

static bool templated_taps(int Lw, int Lh) {
    return Lw == Lh && (Lw % 2) == 0 && Lw >= 2 && Lw <= 16 && !dwt_policy().force_direct;
}

// level sizes of the analysis chain; returns a status
static int afb_dims(int H, int W, int Lw, int Lh, int mode, int J, const int* pad_hw, int* Ho, int* Wo) {
    int h = H, w = W;
    for (int j = 0; j < J; ++j) {
        const int ph = (pad_hw && j > 0) ? pad_hw[2 * j] : 0, pw = (pad_hw && j > 0) ? pad_hw[2 * j + 1] : 0;
        if (ph < 0 || ph > 1 || pw < 0 || pw > 1) return B200W_ERR_BAD_SHAPE;
        h = coeff_len(h + ph, Lh, mode);
        w = coeff_len(w + pw, Lw, mode);
        if (h < 1 || w < 1) return B200W_ERR_BAD_SHAPE;
        Ho[j] = h;
        Wo[j] = w;
    }
    return B200W_OK;
}

static size_t afb_workspace_bytes(int planes, int H, int W, int Lw, int Lh, int mode, int J, const int* pad_hw) {
    if (planes < 1 || H < 1 || W < 1 || J < 1 || J > kMaxLevels || Lw < 1 || Lh < 1 || !mode_supported(mode)) return 0;
    int Ho[kMaxLevels], Wo[kMaxLevels];
    if (afb_dims(H, W, Lw, Lh, mode, J, pad_hw, Ho, Wo)) return 0;
    size_t n = sync_bytes(planes, J);
    for (int j = 0; j + 1 < J; ++j) n += scratch_bytes(planes, Ho[j], Wo[j]);
    return n;
}

static int run_afb_chain(const float* x, int64_t x_ps, int64_t x_rs, int planes, int H, int W, const float* w_lo,
                         const float* w_hi, int Lw, const float* h_lo, const float* h_hi, int Lh, int mode, int J,
                         const int* pad_hw, float* yl, float* const* highs, void* workspace, size_t workspace_bytes,
                         cudaStream_t st, float hi_scale = 1.f, float hi_shift = 0.f, bool allow_skip = false) {
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (J < 1 || J > kMaxLevels) return B200W_ERR_BAD_SHAPE;
    // the filter_wavelet entry point (single level) may leave out the low-pass or the detail output
    if (!x || !highs || (!allow_skip && !yl) || (allow_skip && !yl && !highs[0])) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    AfbParams p;
    int rc = fill_taps(p.t, w_lo, w_hi, Lw, h_lo, h_hi, Lh);
    if (rc) return rc;
    int Ho[kMaxLevels], Wo[kMaxLevels];
    if ((rc = afb_dims(H, W, Lw, Lh, mode, J, pad_hw, Ho, Wo))) return rc;
    if (J > 1) {
        if (!workspace || workspace_bytes < afb_workspace_bytes(planes, H, W, Lw, Lh, mode, J, pad_hw) ||
            !aligned_to(workspace, 256))
            return B200W_ERR_WORKSPACE;
    }
    p.J = J;
    p.planes = planes;
    p.mode = mode;
    p.ticket = J > 1 ? (unsigned*)workspace : nullptr;
    p.done = J > 1 ? p.ticket + 1 : nullptr;
    char* scratch = (char*)workspace + sync_bytes(planes, J);
    int h = H, w = W;  // real size of the level input
    for (int j = 0; j < J; ++j) {
        AfbLevel& lv = p.lv[j];
        if (!highs[j] && !allow_skip) return B200W_ERR_NULL_POINTER;
        const int ph = (pad_hw && j > 0) ? pad_hw[2 * j] : 0, pw = (pad_hw && j > 0) ? pad_hw[2 * j + 1] : 0;
        lv.st_low = (j < J - 1 || yl != nullptr) ? 1 : 0;
        lv.st_hi = highs[j] != nullptr ? 1 : 0;
        lv.hi_scale = hi_scale;
        lv.hi_shift = hi_shift;
        if (j == 0) {
            lv.x = x;
            lv.x_ps = x_ps;
            lv.x_rs = x_rs;
        } else {  // the previous level's low-pass image in the workspace
            lv.x = p.lv[j - 1].low;
            lv.x_ps = p.lv[j - 1].low_ps;
            lv.x_rs = p.lv[j - 1].low_rs;
        }
        lv.Hreal = h;
        lv.Wreal = w;
        lv.H = h + ph;
        lv.W = w + pw;
        if ((rc = analysis_offset(lv.W, Lw, mode, &lv.offW))) return rc;
        if ((rc = analysis_offset(lv.H, Lh, mode, &lv.offH))) return rc;
        lv.Ho = Ho[j];
        lv.Wo = Wo[j];
        if (j == J - 1) {
            lv.low = yl;
            lv.low_rs = lv.Wo;
            lv.low_ps = (long long)lv.Ho * lv.Wo;
        } else {
            lv.low = (float*)scratch;
            lv.low_rs = pitch4(lv.Wo);
            lv.low_ps = (long long)lv.Ho * lv.low_rs;
            scratch += scratch_bytes(planes, lv.Ho, lv.Wo);
        }
        lv.highs = highs[j];
        lv.out_vec2 = ((lv.Wo % 2) == 0 && lv.highs && aligned_to(lv.highs, 8)) ? 1 : 0;
        lv.low_vec2 = ((lv.low_rs % 2) == 0 && (lv.low_ps % 2) == 0 && lv.low && aligned_to(lv.low, 8)) ? 1 : 0;
        lv.cta_base = 0;
        lv.R = lv.ncp = lv.cpp = lv.cp0A = lv.ncpA = lv.itemsA = lv.cppA = lv.RB = lv.itemsB = 0;
        h = lv.Ho;
        w = lv.Wo;
    }
    if (templated_taps(Lw, Lh) && afb_stream_supported(p, Lw)) {
        // chains of small planes: one CTA owns a part of a plane for all levels (TMA-staged owner kernel first, the
        // cp.async owner kernel for the shapes it declines; both need 16-byte aligned rows); everything else goes
        // through the ticketed stream chain
        const DwtPolicy& pol = dwt_policy();
        const bool owner = J > 1 && pol.owner != 0, force = pol.owner == 2;
        if (owner && pol.tma) {
            AfbTmaParams tp;
            if (afb_tma_plan(p, Lw, device_sms(), force, pol.tma_G, pol.tma_D, pol.tma_noboxes, tp))
                return launch_afb_tma(tp, Lw, st);
        }
        if (owner) {
            AfbOwnerParams op;
            if (afb_owner_plan(p, Lw, device_sms(), force, op)) return launch_afb_owner(op, Lw, st);
        }
        return launch_afb_stream(p, Lw, device_sms(), st);
    }
    for (int j = 0; j < J; ++j) {  // other taps and row strides: level by level with the direct kernel
        const AfbLevel& lv = p.lv[j];
        const AfbDirectParams<float> d = {lv.x, lv.low, lv.highs, lv.x_ps, lv.x_rs, lv.low_ps, lv.low_rs, lv.H, lv.W,
                                          lv.Hreal, lv.Wreal, lv.Ho, lv.Wo, lv.offH, lv.offW, lv.st_low, lv.st_hi,
                                          lv.hi_scale, lv.hi_shift, planes, mode, Lw, Lh, p.t};
        if ((rc = launch_direct(afb2d_direct_kernel<float>, d, (size_t)planes * lv.Ho * lv.Wo, "afb2d_direct_kernel", st)))
            return rc;
    }
    return B200W_OK;
}

// ---- synthesis chain -------------------------------------------------------------------------------
static int sfb_check_dims(int planes, const int* hs, const int* ws, int Lw, int Lh, int mode, int J, const int* out_hs,
                          const int* out_ws) {
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (J < 1 || J > kMaxLevels) return B200W_ERR_BAD_SHAPE;
    if (!hs || !ws || !out_hs || !out_ws) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || Lw < 1 || Lh < 1) return B200W_ERR_BAD_SHAPE;
    const bool per = mode == B200W_MODE_PERIODIZATION;
    for (int j = 0; j < J; ++j) {
        if (hs[j] < 1 || ws[j] < 1 || out_hs[j] < 1 || out_ws[j] < 1) return B200W_ERR_BAD_SHAPE;
        if (per && (2 * hs[j] < Lh || 2 * ws[j] < Lw)) return B200W_ERR_PER_TOO_SHORT;
        if (out_hs[j] > idwt_len(hs[j], Lh, mode) || out_ws[j] > idwt_len(ws[j], Lw, mode)) return B200W_ERR_BAD_SHAPE;
        // level j < J-1 reads the top-left h[j] x w[j] block of the previous output ('unpad')
        if (j + 1 < J && (out_hs[j + 1] < hs[j] || out_ws[j + 1] < ws[j])) return B200W_ERR_BAD_SHAPE;
    }
    return B200W_OK;
}

static size_t sfb_workspace_bytes(int planes, int J, const int* out_hs, const int* out_ws) {
    size_t n = sync_bytes(planes, J);
    for (int j = 1; j < J; ++j) n += scratch_bytes(planes, out_hs[j], out_ws[j]);
    return n;
}

// levels are given finest first (index j like yh[j]); the chain runs j = J-1 .. 0
static int run_sfb_chain(const float* yl, int64_t yl_ps, int64_t yl_rs, const float* const* highs, int planes,
                         const int* hs, const int* ws, const float* w_lo, const float* w_hi, int Lw, const float* h_lo,
                         const float* h_hi, int Lh, int mode, int J, const int* out_hs, const int* out_ws, float* y,
                         void* workspace, size_t workspace_bytes, cudaStream_t st) {
    int rc = sfb_check_dims(planes, hs, ws, Lw, Lh, mode, J, out_hs, out_ws);
    if (rc) return rc;
    if (!yl || !y) return B200W_ERR_NULL_POINTER;
    SfbParams p;
    if ((rc = fill_taps(p.t, w_lo, w_hi, Lw, h_lo, h_hi, Lh))) return rc;
    if (J > 1) {
        if (!workspace || workspace_bytes < sfb_workspace_bytes(planes, J, out_hs, out_ws) || !aligned_to(workspace, 256))
            return B200W_ERR_WORKSPACE;
    }
    const bool per = mode == B200W_MODE_PERIODIZATION;
    p.J = J;
    p.planes = planes;
    p.periodic = per ? 1 : 0;
    p.ticket = J > 1 ? (unsigned*)workspace : nullptr;
    p.done = J > 1 ? p.ticket + 1 : nullptr;
    char* scratch = (char*)workspace + sync_bytes(planes, J);
    for (int c = 0; c < J; ++c) {  // chain position c handles level j = J-1-c
        const int j = J - 1 - c;
        SfbLevel& lv = p.lv[c];
        if (c == 0) {
            lv.low = yl;
            lv.low_ps = yl_ps;
            lv.low_rs = yl_rs;
        } else {  // the previous chain output, of which the top-left h x w block is used ('unpad')
            lv.low = p.lv[c - 1].y;
            lv.low_ps = p.lv[c - 1].y_ps;
            lv.low_rs = p.lv[c - 1].y_rs;
        }
        lv.highs = highs ? highs[j] : nullptr;
        lv.h = hs[j];
        lv.w = ws[j];
        lv.out_h = out_hs[j];
        lv.out_w = out_ws[j];
        if (j == 0) {
            lv.y = y;
            lv.y_rs = lv.out_w;
            lv.y_ps = (long long)lv.out_h * lv.out_w;
        } else {
            lv.y = (float*)scratch;
            lv.y_rs = pitch4(lv.out_w);
            lv.y_ps = (long long)lv.out_h * lv.y_rs;
            scratch += scratch_bytes(planes, lv.out_h, lv.out_w);
        }
        lv.offW = synthesis_offset(Lw, mode);
        lv.offH = synthesis_offset(Lh, mode);
        lv.cta_base = 0;
        lv.Rp = lv.cpp = lv.tA0 = lv.ntA = lv.itemsA = lv.cppA = 0;
        lv.nA0 = lv.nA1 = lv.itemsB = lv.n0_off = lv.kb_off = lv.m_lo = lv.vec2 = 0;
        lv.y_vec = 1;
    }
    if (templated_taps(Lw, Lh)) {
        // chains of small planes: one CTA owns a part of a plane for all positions (TMA-staged owner kernel first, the
        // cp.async owner kernel for the shapes it declines); everything else goes through the ticketed stream chain
        const DwtPolicy& pol = dwt_policy();
        const bool owner = J > 1 && pol.owner != 0, force = pol.owner == 2;
        if (owner && pol.tma) {
            SfbTmaParams tp;
            if (sfb_tma_plan(p, Lw, device_sms(), force, pol.tma_G, pol.tma_D, tp)) return launch_sfb_tma(tp, Lw, st);
        }
        if (owner) {
            SfbOwnerParams op;
            if (sfb_owner_plan(p, Lw, device_sms(), force, op)) return launch_sfb_owner(op, Lw, st);
        }
        return launch_sfb_stream(p, Lw, device_sms(), st);
    }
    for (int c = 0; c < J; ++c) {
        const SfbLevel& lv = p.lv[c];
        const SfbDirectParams<float> d = {lv.low, lv.highs, lv.y, lv.low_ps, lv.low_rs, lv.y_ps, lv.y_rs, lv.h, lv.w,
                                          lv.out_h, lv.out_w, lv.offH, lv.offW, planes, p.periodic, Lw, Lh, p.t};
        if ((rc = launch_direct(sfb2d_direct_kernel<float>, d, (size_t)planes * lv.out_h * lv.out_w, "sfb2d_direct_kernel",
                                st)))
            return rc;
    }
    return B200W_OK;
}

// one fp64 analysis level through the direct kernel; the caller has validated the arguments and set d.t, d.offH, d.offW,
// d.Ho and d.Wo
static int launch_afb2d_f64(AfbDirectParams<double>& d, const double* x, int64_t x_ps, int64_t x_rs, int planes, int H,
                            int W, int Lw, int Lh, int mode, double* low, double* highs, double hi_scale,
                            double hi_shift, cudaStream_t st) {
    d.x = x;
    d.x_ps = x_ps;
    d.x_rs = x_rs;
    d.low = low;
    d.low_rs = d.Wo;
    d.low_ps = (long long)d.Ho * d.Wo;
    d.highs = highs;
    d.H = d.Hreal = H;
    d.W = d.Wreal = W;
    d.st_low = low != nullptr;
    d.st_hi = highs != nullptr;
    d.hi_scale = hi_scale;
    d.hi_shift = hi_shift;
    d.planes = planes;
    d.mode = mode;
    d.Lw = Lw;
    d.Lh = Lh;
    return launch_direct(afb2d_direct_kernel<double>, d, (size_t)planes * d.Ho * d.Wo, "afb2d_f64_kernel", st);
}

}  // namespace b200w

using namespace b200w;

extern "C" int b200w_dwt_coeff_len(int n, int l, int mode) {
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (n < 1 || l < 1) return B200W_ERR_BAD_SHAPE;
    return coeff_len(n, l, mode);
}

extern "C" int b200w_idwt_len(int m, int l, int mode) {
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (m < 1 || l < 1) return B200W_ERR_BAD_SHAPE;
    return idwt_len(m, l, mode);
}

extern "C" size_t b200w_dwt2_workspace_bytes(int planes, int H, int W, int Lw, int Lh, int mode, int J,
                                             const int* pad_hw) {
    return afb_workspace_bytes(planes, H, W, Lw, Lh, mode, J, pad_hw);
}

extern "C" size_t b200w_idwt2_workspace_bytes(int planes, int J, const int* out_h, const int* out_w) {
    if (planes < 1 || J < 1 || J > kMaxLevels || !out_h || !out_w) return 0;
    for (int j = 0; j < J; ++j)
        if (out_h[j] < 1 || out_w[j] < 1) return 0;
    return sfb_workspace_bytes(planes, J, out_h, out_w);
}

extern "C" int b200w_afb2d_f32(const float* x, int64_t x_plane_stride, int64_t x_row_stride, int planes, int H,
                               int W, const float* w_lo, const float* w_hi, int Lw, const float* h_lo,
                               const float* h_hi, int Lh, int mode, float* low, float* highs, void* stream) {
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (!low || !highs) return B200W_ERR_NULL_POINTER;
    float* his[1] = {highs};
    return run_afb_chain(x, x_plane_stride, x_row_stride, planes, H, W, w_lo, w_hi, Lw, h_lo, h_hi, Lh, mode, 1,
                         nullptr, low, his, nullptr, 0, (cudaStream_t)stream);
}

extern "C" int b200w_afb2d_ex_f32(const float* x, int64_t x_plane_stride, int64_t x_row_stride, int planes, int H,
                                  int W, const float* w_lo, const float* w_hi, int Lw, const float* h_lo,
                                  const float* h_hi, int Lh, int mode, float* low, float* highs, float hi_scale,
                                  float hi_shift, void* stream) {
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    float* his[1] = {highs};
    return run_afb_chain(x, x_plane_stride, x_row_stride, planes, H, W, w_lo, w_hi, Lw, h_lo, h_hi, Lh, mode, 1,
                         nullptr, low, his, nullptr, 0, (cudaStream_t)stream, hi_scale, hi_shift, true);
}

extern "C" int b200w_dwt2_f32(const float* x, int64_t x_plane_stride, int64_t x_row_stride, int planes, int H, int W,
                              const float* w_lo, const float* w_hi, int Lw, const float* h_lo, const float* h_hi,
                              int Lh, int mode, int J, const int* pad_hw, float* yl, float* const* highs,
                              void* workspace, size_t workspace_bytes, void* stream) {
    return run_afb_chain(x, x_plane_stride, x_row_stride, planes, H, W, w_lo, w_hi, Lw, h_lo, h_hi, Lh, mode, J,
                         pad_hw, yl, highs, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int b200w_sfb2d_f32(const float* low, int64_t low_plane_stride, int64_t low_row_stride,
                               const float* highs, int planes, int h, int w, const float* w_lo, const float* w_hi,
                               int Lw, const float* h_lo, const float* h_hi, int Lh, int mode, float* y, int out_h,
                               int out_w, void* stream) {
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (!low || !y) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || h < 1 || w < 1 || out_h < 1 || out_w < 1) return B200W_ERR_BAD_SHAPE;
    const float* his[1] = {highs};
    return run_sfb_chain(low, low_plane_stride, low_row_stride, his, planes, &h, &w, w_lo, w_hi, Lw, h_lo, h_hi, Lh,
                         mode, 1, &out_h, &out_w, y, nullptr, 0, (cudaStream_t)stream);
}

// The reference's fp64 mode (modules built under torch.set_default_dtype(torch.float64)): one level through the direct
// kernels.  Unlike the fp32 entry points these check the data pointers before the mode, report null taps as
// B200W_ERR_NULL_POINTER and reject outputs of more than 2^31-1 pixels per plane (ABI status codes).  The detail bands
// pass the store epilogue with scale 1 and shift 0, which stores a -0 as +0.
extern "C" int b200w_afb2d_f64(const double* x, int64_t x_ps, int64_t x_rs, int planes, int H, int W, const double* w_lo,
                               const double* w_hi, int Lw, const double* h_lo, const double* h_hi, int Lh, int mode,
                               double* low, double* highs, void* stream) {
    if (!x || !low || !highs) return B200W_ERR_NULL_POINTER;
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (planes < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    if (!w_lo || !w_hi || !h_lo || !h_hi) return B200W_ERR_NULL_POINTER;
    AfbDirectParams<double> d = {};
    int rc = fill_taps(d.t, w_lo, w_hi, Lw, h_lo, h_hi, Lh);
    if (rc || (rc = analysis_offset(H, Lh, mode, &d.offH)) || (rc = analysis_offset(W, Lw, mode, &d.offW))) return rc;
    d.Ho = coeff_len(H, Lh, mode);
    d.Wo = coeff_len(W, Lw, mode);
    if (d.Ho < 1 || d.Wo < 1 || (long long)d.Ho * d.Wo > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    return launch_afb2d_f64(d, x, x_ps, x_rs, planes, H, W, Lw, Lh, mode, low, highs, 1.0, 0.0, (cudaStream_t)stream);
}

// FS_Discriminator.filter_wavelet in double: the checks of b200w_afb2d_ex_f32, in its order, then the direct kernel with
// the same store epilogue (a NULL output is not written; detail bands stored as hi_scale * v + hi_shift).
extern "C" int b200w_afb2d_ex_f64(const double* x, int64_t x_ps, int64_t x_rs, int planes, int H, int W,
                                  const double* w_lo, const double* w_hi, int Lw, const double* h_lo, const double* h_hi,
                                  int Lh, int mode, double* low, double* highs, double hi_scale, double hi_shift,
                                  void* stream) {
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (!x || (!low && !highs)) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || H < 1 || W < 1) return B200W_ERR_BAD_SHAPE;
    AfbDirectParams<double> d = {};
    int rc = fill_taps(d.t, w_lo, w_hi, Lw, h_lo, h_hi, Lh);
    if (rc || (rc = afb_dims(H, W, Lw, Lh, mode, 1, nullptr, &d.Ho, &d.Wo))) return rc;
    if ((rc = analysis_offset(W, Lw, mode, &d.offW)) || (rc = analysis_offset(H, Lh, mode, &d.offH))) return rc;
    return launch_afb2d_f64(d, x, x_ps, x_rs, planes, H, W, Lw, Lh, mode, low, highs, hi_scale, hi_shift,
                            (cudaStream_t)stream);
}

extern "C" int b200w_sfb2d_f64(const double* low, int64_t low_ps, int64_t low_rs, const double* highs, int planes, int h,
                               int w, const double* w_lo, const double* w_hi, int Lw, const double* h_lo,
                               const double* h_hi, int Lh, int mode, double* y, int out_h, int out_w, void* stream) {
    if (!low || !y) return B200W_ERR_NULL_POINTER;
    if (!mode_supported(mode)) return B200W_ERR_BAD_MODE;
    if (planes < 1 || h < 1 || w < 1 || out_h < 1 || out_w < 1) return B200W_ERR_BAD_SHAPE;
    if (!w_lo || !w_hi || !h_lo || !h_hi) return B200W_ERR_NULL_POINTER;
    SfbDirectParams<double> d = {};
    const int rc = fill_taps(d.t, w_lo, w_hi, Lw, h_lo, h_hi, Lh);
    if (rc) return rc;
    const bool per = mode == B200W_MODE_PERIODIZATION;
    if (per && (2 * h < Lh || 2 * w < Lw)) return B200W_ERR_PER_TOO_SHORT;
    if (out_h > idwt_len(h, Lh, mode) || out_w > idwt_len(w, Lw, mode) || (long long)out_h * out_w > 0x7fffffffLL)
        return B200W_ERR_BAD_SHAPE;
    d.low = low;
    d.low_ps = low_ps;
    d.low_rs = low_rs;
    d.highs = highs;
    d.y = y;
    d.y_rs = out_w;
    d.y_ps = (long long)out_h * out_w;
    d.h = h;
    d.w = w;
    d.out_h = out_h;
    d.out_w = out_w;
    d.offH = synthesis_offset(Lh, mode);
    d.offW = synthesis_offset(Lw, mode);
    d.planes = planes;
    d.periodic = per;
    d.Lw = Lw;
    d.Lh = Lh;
    return launch_direct(sfb2d_direct_kernel<double>, d, (size_t)planes * out_h * out_w, "sfb2d_f64_kernel",
                         (cudaStream_t)stream);
}

extern "C" int b200w_idwt2_f32(const float* yl, int64_t yl_plane_stride, int64_t yl_row_stride,
                               const float* const* highs, int planes, const int* h, const int* w, const float* w_lo,
                               const float* w_hi, int Lw, const float* h_lo, const float* h_hi, int Lh, int mode,
                               int J, const int* out_h, const int* out_w, float* y, void* workspace,
                               size_t workspace_bytes, void* stream) {
    return run_sfb_chain(yl, yl_plane_stride, yl_row_stride, highs, planes, h, w, w_lo, w_hi, Lw, h_lo, h_hi, Lh, mode,
                         J, out_h, out_w, y, workspace, workspace_bytes, (cudaStream_t)stream);
}
