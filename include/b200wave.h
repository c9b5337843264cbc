/*
 * b200wave -- C ABI of the B200-native (sm_100a) wavelet + SSIM hot path.
 *
 * The reference (KevynUtopia/Frequency-Aware-Inverse-Consistent-OCTA-Super-Resolution)
 * is pure Python and has no FFI seam of its own: the drop-in boundary is the pair of
 * torch.autograd Functions AFB2D / SFB2D and the free function _ssim.  Each entry
 * point below replaces the body of one of them; citations are relative to
 * /root/reference (pw = pytorch_wavelets/pytorch_wavelets):
 *
 *   b200w_afb2d_f32     pw/dwt/lowlevel.py:336-347  AFB2D.forward (afb1d dim=3 then dim=2, :91-172)
 *                       pw/dwt/lowlevel.py:682-694  SFB2D.backward (same arithmetic, synthesis taps as correlators)
 *   b200w_sfb2d_f32     pw/dwt/lowlevel.py:671-680  SFB2D.forward (sfb1d x3, :226-271)
 *                       pw/dwt/lowlevel.py:349-365  AFB2D.backward (same arithmetic + crop to the input H, W)
 *   b200w_ssim_fwd_f32  ssim.py:17-37               _ssim (five 11x11 Gaussian blurs, SSIM map, mean)
 *   b200w_ssim_bwd_f32  autograd through ssim.py:17-37 (closed form, SURVEY.md 8a-a10)
 *   b200w_msssim_scale_fwd_f32 / _bwd_f32 (and _f64)  one scale of MS-SSIM (no counterpart in the reference)
 *   b200w_dwt2_f32      pw/dwt/transform2d.py:66-74    the J-level loop of DWTForward.forward over AFB2D.apply,
 *                       and the backward of DWTInverse (J x SFB2D.backward through the 'unpad' crops) -- ONE launch
 *   b200w_idwt2_f32     pw/dwt/transform2d.py:134-148  the J-level loop of DWTInverse.forward over SFB2D.apply incl.
 *                       the 'unpad' crop, and the backward of DWTForward (J x AFB2D.backward) -- ONE launch
 *   b200w_afb2d_ex_f32  model.py:166-179, 222-235  FS_Discriminator.filter_wavelet: AFB2D + band selection + *0.5+0.5
 *                       fused into the analysis kernel's stores (SURVEY.md 8f row 2)
 *   b200w_dwt_coeff_len pywt.dwt_coeff_len as called at pw/dwt/lowlevel.py:153
 *   b200w_freq_mask_c64 / b200w_abs_sign_f32 / b200w_sign_mul_f32
 *                       utils.py:71-117  Gaussian low / high pass in the Fourier domain (SURVEY.md 8f row 1)
 *   b200w_afb1d_f32 / b200w_sfb1d_f32             pw/dwt/lowlevel.py:368-424, 697-743  AFB1D / SFB1D (SURVEY.md 8f row 3)
 *   b200w_swt2d_fwd_f32 / b200w_swt2d_bwd_f32     pw/dwt/lowlevel.py:175-223, 475-521  afb2d_atrous / SWTForward (8f row 3)
 *   b200w_iswt2d_f32 / b200w_iswt2d_f64           one level of SWTInverse, the periodic inverse of SWTForward (the
 *                       reference's pw/dwt/swt_inverse.py is unfinished and not exported: semantics in DESIGN.md K12)
 *   b200w_tv_fwd_f32 / b200w_tv_bwd_f32           model.py:17-33  TVLoss (SURVEY.md 8f row 4)
 *   b200w_phase_sums_c64 / b200w_phase_grad_c64   model.py:36-58  phase_consistency_loss (SURVEY.md 8f row 4)
 *   b200w_*_f64         the same bodies on double tensors (the reference's double mode): afb2d / sfb2d, afb2d_ex,
 *                       afb1d / sfb1d, swt2d, tv, abs_sign / sign_mul, and ssim (ssim.py:17-37 with the dense window of
 *                       ssim.py:7-15, see below); b200w_freq_mask_c128 on complex128 spectra
 *
 * Conventions
 *   - every image pointer is DEVICE memory owned by the caller (torch); the library never
 *     allocates or frees device memory and keeps no mutable global state => re-entrant.
 *   - filter taps are HOST pointers (<= B200W_MAX_TAPS floats each); they are copied into
 *     the kernel parameter block, so the call is asynchronous and CUDA-graph capturable.
 *     Analysis taps are the correlation kernels exactly as the reference's module buffers
 *     hold them (already time-reversed by prep_filt_afb1d, pw/dwt/lowlevel.py:970-971);
 *     synthesis taps are as-is (prep_filt_sfb1d, :918-922).
 *   - "w_*" taps filter along W (dim 3: the h*_row / g*_row *parameters* of AFB2D/SFB2D.forward),
 *     "h_*" taps along H (dim 2).
 *   - layout: fp32, planes = N*C images of H x W, unit stride along W.  Inputs take explicit
 *     plane / row strides (in elements) so a cropped view (transform2d.py:141-145) needs no copy;
 *     outputs are dense (the reference returns contiguous tensors, tests/test_dwt.py:47-50).
 *   - `stream` is a cudaStream_t (NULL = legacy default stream).  Nothing synchronises.
 *   - return value: B200W_OK (0) or a negative b200w_status; b200w_status_string() names it.
 *     An unsupported padding mode returns B200W_ERR_BAD_MODE, which the Python wrapper raises
 *     as ValueError("Unkown pad type: ...") like pw/dwt/lowlevel.py:88,170,290.
 */
#ifndef B200WAVE_H_
#define B200WAVE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200W_ABI_VERSION 1
#define B200W_MAX_TAPS 64
#define B200W_MAX_LEVELS 8

/* mode_to_int, pw/dwt/lowlevel.py:274-290 */
enum b200w_mode {
    B200W_MODE_ZERO = 0,
    B200W_MODE_SYMMETRIC = 1,
    B200W_MODE_PERIODIZATION = 2,
    B200W_MODE_CONSTANT = 3,   /* accepted by mode_to_int, rejected by afb1d/sfb1d: BAD_MODE */
    B200W_MODE_REFLECT = 4,
    B200W_MODE_REPLICATE = 5,  /* idem */
    B200W_MODE_PERIODIC = 6
};

enum b200w_status {
    B200W_OK = 0,
    B200W_ERR_BAD_MODE = -1,      /* "Unkown pad type" */
    B200W_ERR_BAD_TAPS = -2,      /* tap count < 1 or > B200W_MAX_TAPS, or null tap pointer */
    B200W_ERR_NULL_POINTER = -3,
    B200W_ERR_BAD_SHAPE = -4,     /* non-positive dimension, or out_h/out_w larger than the synthesis output */
    B200W_ERR_REFLECT_PAD = -5,   /* reflect padding needs pad < dimension (torch F.pad rule) */
    B200W_ERR_PER_TOO_SHORT = -6, /* periodization needs (even-extended) length >= tap count */
    B200W_ERR_LAUNCH = -7,        /* cudaGetLastError() after the launch was not cudaSuccess */
    B200W_ERR_WORKSPACE = -8,     /* workspace too small / null */
    B200W_ERR_BAD_WINDOW = -9     /* SSIM window size must be odd and <= B200W_SSIM_MAX_WINDOW */
};

#define B200W_SSIM_MAX_WINDOW 11

int b200w_abi_version(void);
const char* b200w_status_string(int status);
/* last cudaError_t seen by a failing launch on this thread (0 = none); for diagnostics only */
int b200w_last_cuda_error(void);
/* diagnostics: number of kernels this library has launched in the process, and the name of the `back`-th most
 * recent one ("" when out of range; the last 64 are kept).  bench.py counts its `gpu_launches` with these. */
unsigned long long b200w_kernel_launches(void);
const char* b200w_kernel_log(int back);
/* hash of the sources (csrc/, include/) and compiler flags this binary was built from: the Python side compares it
 * with the tree it runs in, so that numbers are never produced by kernels that do not match the committed sources */
const char* b200w_build_hash(void);

/* floor((n+l-1)/2), or ceil(n/2) for periodization; negative status for a bad mode */
int b200w_dwt_coeff_len(int n, int l, int mode);
/* length produced by one synthesis level from m coefficients: 2m-l+2, or 2m for periodization */
int b200w_idwt_len(int m, int l, int mode);

/*
 * One analysis level: x (planes,H,W) -> low (planes,Ho,Wo), highs (planes,3,Ho,Wo) with
 * Ho = b200w_dwt_coeff_len(H,Lh,mode), Wo = b200w_dwt_coeff_len(W,Lw,mode);
 * band order LH,HL,HH = (W-lo,H-hi),(W-hi,H-lo),(W-hi,H-hi)  (pw/dwt/lowlevel.py:343-347).
 */
int b200w_afb2d_f32(const float* x, int64_t x_plane_stride, int64_t x_row_stride,
                    int planes, int H, int W,
                    const float* w_lo, const float* w_hi, int Lw,
                    const float* h_lo, const float* h_hi, int Lh,
                    int mode, float* low, float* highs, void* stream);

/*
 * One analysis level with the store epilogue of FS_Discriminator.filter_wavelet (model.py:166-179, 222-235):
 * `low` or `highs` may be NULL (that output is not written: cs='sum' uses only LL, cs='cat' only the detail bands),
 * and the detail bands are stored as hi_scale * v + hi_shift (norm=True: 0.5, 0.5).  With C == 1 the (planes,3,Ho,Wo)
 * `highs` is exactly torch.cat((LH, HL, HH), 1).
 */
int b200w_afb2d_ex_f32(const float* x, int64_t x_plane_stride, int64_t x_row_stride,
                       int planes, int H, int W,
                       const float* w_lo, const float* w_hi, int Lw,
                       const float* h_lo, const float* h_hi, int Lh,
                       int mode, float* low, float* highs, float hi_scale, float hi_shift, void* stream);

/*
 * One synthesis level: low (planes,h,w) [strided], highs (planes,3,h,w) dense or NULL (= zeros,
 * transform2d.py:137-139) -> y (planes,out_h,out_w) dense, where out_h <= b200w_idwt_len(h,Lh,mode)
 * and out_w <= b200w_idwt_len(w,Lw,mode); a smaller out_h/out_w crops (pw/dwt/lowlevel.py:359-364).
 */
int b200w_sfb2d_f32(const float* low, int64_t low_plane_stride, int64_t low_row_stride,
                    const float* highs, int planes, int h, int w,
                    const float* w_lo, const float* w_hi, int Lw,
                    const float* h_lo, const float* h_hi, int Lh,
                    int mode, float* y, int out_h, int out_w, void* stream);

/*
 * J-level analysis in one launch (J <= B200W_MAX_LEVELS).  Level 0 reads x; level j > 0 reads the low-pass image
 * of level j-1, optionally extended by one zero row / column: pad_hw = 2*J ints (pad_h, pad_w per level, entry 0
 * ignored) or NULL.  The zero extension is what autograd's backward of the 'unpad' slice
 * (transform2d.py:141-145) feeds into SFB2D.backward.  yl: (planes,Ho_J,Wo_J) dense, highs[j]:
 * (planes,3,Ho_j,Wo_j) dense, with Ho_j = b200w_dwt_coeff_len(Ho_{j-1} + pad_h[j], Lh, mode); highs is a HOST
 * array of J device pointers.  The intermediate low-pass images live in `workspace` (DEVICE, 256-byte aligned, at
 * least b200w_dwt2_workspace_bytes(...) bytes, together with the per-plane completion counters; may be NULL
 * when J == 1) with rows padded to 16 bytes.
 */
size_t b200w_dwt2_workspace_bytes(int planes, int H, int W, int Lw, int Lh, int mode, int J, const int* pad_hw);
int b200w_dwt2_f32(const float* x, int64_t x_plane_stride, int64_t x_row_stride, int planes, int H, int W,
                   const float* w_lo, const float* w_hi, int Lw,
                   const float* h_lo, const float* h_hi, int Lh,
                   int mode, int J, const int* pad_hw, float* yl, float* const* highs,
                   void* workspace, size_t workspace_bytes, void* stream);

/*
 * J-level synthesis in one launch.  Levels are indexed like yh (j = 0 finest); the chain runs j = J-1 .. 0.
 * highs[j]: (planes,3,h[j],w[j]) dense or NULL (= zeros); highs itself may be NULL.  Level J-1 reads yl (strided,
 * at least h[J-1] x w[J-1]); level j < J-1 reads the top-left h[j] x w[j] block of the output of level j+1 (the
 * 'unpad'), whose size is out_h[j+1] x out_w[j+1] <= b200w_idwt_len(h[j+1],Lh,mode) (smaller = crop, as in
 * AFB2D.backward).  y: (planes,out_h[0],out_w[0]) dense, the result; the intermediate outputs live in `workspace`
 * (DEVICE, 256-byte aligned, at least b200w_idwt2_workspace_bytes(...) bytes; may be NULL when J == 1).
 * h, w, out_h, out_w and highs are HOST arrays of J entries.
 */
size_t b200w_idwt2_workspace_bytes(int planes, int J, const int* out_h, const int* out_w);
int b200w_idwt2_f32(const float* yl, int64_t yl_plane_stride, int64_t yl_row_stride,
                    const float* const* highs, int planes, const int* h, const int* w,
                    const float* w_lo, const float* w_hi, int Lw,
                    const float* h_lo, const float* h_hi, int Lh,
                    int mode, int J, const int* out_h, const int* out_w, float* y,
                    void* workspace, size_t workspace_bytes, void* stream);

/*
 * Fourier-domain Gaussian frequency split, utils.py:71-117 (guais_low_pass / guais_high_pass / high_pass / low_pass):
 * the pointwise passes around the FFTs (which the caller runs with cuFFT, e.g. torch.fft.rfft2 / irfft2).
 * b200w_freq_mask_c64: in place on the half spectrum of rfft2, (planes, rows, cols/2+1) interleaved complex64;
 *   multiplies bin (u,v) by exp(-0.5 (du^2+dv^2)/radius^2) (1 - that when highpass), du/dv the signed frequencies --
 *   the mask of utils.py:71-91 without materialising or shifting it.
 * b200w_abs_sign_f32: y = sign * |x|  (high_pass: +1, utils.py:103; low_pass: -1, utils.py:117).
 * b200w_sign_mul_f32: out = g * sign * sgn(x), the backward of abs_sign.
 */
int b200w_freq_mask_c64(void* spec, int planes, int rows, int cols, float radius, int highpass, void* stream);
int b200w_abs_sign_f32(const float* x, float* y, size_t n, float sign, void* stream);
int b200w_sign_mul_f32(const float* g, const float* x, float* out, size_t n, float sign, void* stream);

/*
 * SSIM forward.  img1,img2: (N,C,H,W) dense.  win: `ws` HOST floats, the normalised 1-D Gaussian
 * (ssim.py:7-9); the 2-D window of ssim.py:11-15 is its outer product and is applied separably.
 * out: DEVICE, 1 float (size_average != 0: mean over everything) or N floats (per-sample means,
 * ssim.py:34-37).  n_maps selects what is saved for the backward: 0 = nothing, 3 = dS/dmu1,
 * dS/dE[x^2], dS/dE[x1x2] (gradient w.r.t. img1), 4 = those + dS/dmu2 (both gradients);
 * maps: DEVICE (n_maps,N,C,H,W) or NULL when n_maps == 0.
 * workspace: DEVICE scratch of at least b200w_ssim_workspace_bytes() (per-CTA partial sums).
 */
size_t b200w_ssim_workspace_bytes(int N, int C, int H, int W);
int b200w_ssim_fwd_f32(const float* img1, const float* img2, int N, int C, int H, int W,
                       const float* win, int ws, int size_average,
                       int n_maps, float* maps, float* out,
                       void* workspace, size_t workspace_bytes, void* stream);

/*
 * SSIM backward.  grad_out: DEVICE, 1 float (size_average) or N floats.  d1 (and d2 if non-NULL,
 * which needs n_maps == 4): DEVICE (N,C,H,W).
 */
int b200w_ssim_bwd_f32(const float* img1, const float* img2, const float* maps, int n_maps,
                       const float* grad_out, int N, int C, int H, int W,
                       const float* win, int ws, int size_average,
                       float* d1, float* d2, void* stream);

/*
 * Total-variation loss, model.py:17-33 (`TVLoss`, train.py:98), SURVEY.md 8f row 4.
 * b200w_tv_fwd_f32: out2[0] = sum (x[i+1][j]-x[i][j])^2, out2[1] = sum (x[i][j+1]-x[i][j])^2 over all `planes`
 * dense H x W planes, one pass over x; `workspace` = b200w_tv_workspace_bytes(planes, H) bytes of per-CTA partials
 * (reduced in fixed order: deterministic).  The scalar loss is weight*2*(out2[0]/count_h + out2[1]/count_w)/batch.
 * b200w_tv_bwd_f32: dx = grad_out[0] * (ch * d out2[0]/dx + cw * d out2[1]/dx); grad_out is a device scalar.
 */
size_t b200w_tv_workspace_bytes(int planes, int H);
int b200w_tv_fwd_f32(const float* x, int planes, int H, int W, void* workspace, size_t workspace_bytes,
                     float* out2, void* stream);
int b200w_tv_bwd_f32(const float* x, const float* grad_out, float ch, float cw, int planes, int H, int W,
                     float* dx, void* stream);

/*
 * Double precision (the reference's fp64 mode: modules built under torch.set_default_dtype(torch.float64),
 * pw tests/test_dwt.py:132-160): single-level banks with the signatures of b200w_afb2d_f32 / b200w_sfb2d_f32 on
 * double data and double taps.  Simple one-thread-per-output kernels; the Python modules run multi-level fp64
 * transforms level by level through them.
 */
int b200w_afb2d_f64(const double* x, int64_t x_plane_stride, int64_t x_row_stride, int planes, int H, int W,
                    const double* w_lo, const double* w_hi, int Lw, const double* h_lo, const double* h_hi, int Lh,
                    int mode, double* low, double* highs, void* stream);
int b200w_sfb2d_f64(const double* low, int64_t low_plane_stride, int64_t low_row_stride, const double* highs, int planes,
                    int h, int w, const double* w_lo, const double* w_hi, int Lw, const double* h_lo, const double* h_hi,
                    int Lh, int mode, double* y, int out_h, int out_w, void* stream);

/*
 * Double twins of b200w_afb2d_ex_f32 and of the frequency-split passes (the reference's double mode: discriminators
 * built under torch.set_default_dtype(torch.float64), double images into utils.high_pass / low_pass): the same
 * arguments, status codes and order of the checks, on double data.
 * b200w_afb2d_ex_f64     model.py:166-179, 222-235  filter_wavelet; double taps, hi_scale and hi_shift (direct kernel)
 * b200w_freq_mask_c128   utils.py:71-91  in place on the complex128 half spectrum.  As in the reference, the mask is
 *   exp(-0.5 (du^2+dv^2) / radius^2) (1 - that when highpass) evaluated in double and rounded once to float
 *   (torch.from_numpy(mask).float()); each bin is multiplied by that float value in double.
 * b200w_abs_sign_f64 / b200w_sign_mul_f64   utils.py:103, 117  y = sign * |x| and its backward, on doubles.
 */
int b200w_afb2d_ex_f64(const double* x, int64_t x_plane_stride, int64_t x_row_stride, int planes, int H, int W,
                       const double* w_lo, const double* w_hi, int Lw, const double* h_lo, const double* h_hi, int Lh,
                       int mode, double* low, double* highs, double hi_scale, double hi_shift, void* stream);
int b200w_freq_mask_c128(void* spec, int planes, int rows, int cols, double radius, int highpass, void* stream);
int b200w_abs_sign_f64(const double* x, double* y, size_t n, double sign, void* stream);
int b200w_sign_mul_f64(const double* g, const double* x, double* out, size_t n, double sign, void* stream);

/*
 * 1-D analysis / synthesis banks, SURVEY.md 8f row 3: the bodies of AFB1D.forward / SFB1D.forward
 * (pw/dwt/lowlevel.py:389-405, 719-730 = afb1d / sfb1d of :91-172, :226-271 on an (N, C, 1, L) view) and, with the other
 * bank's taps, of each other's backward (:407-424, :732-743).  `rows` = N*C signals.
 * b200w_afb1d_f32: x (rows, n) with row stride x_rs -> lo, hi dense (rows, b200w_dwt_coeff_len(n, L, mode)); taps as the
 *   module stores them (prep_filt_afb1d: already time-reversed).
 * b200w_sfb1d_f32: lo (rows, m) with row stride lo_rs (the 'unpad' view of DWT1DInverse, transform1d.py:110-112, is
 *   free), hi dense (rows, m) or NULL (= zeros) -> y dense (rows, out_len), out_len <= b200w_idwt_len(m, L, mode)
 *   (the crop of AFB1D.backward, :421-422).
 */
int b200w_afb1d_f32(const float* x, int64_t x_rs, int rows, int n, const float* h0, const float* h1, int L, int mode,
                    float* lo, float* hi, void* stream);
int b200w_sfb1d_f32(const float* lo, int64_t lo_rs, const float* hi, int rows, int m, const float* g0, const float* g1,
                    int L, int mode, int out_len, float* y, void* stream);

/*
 * Undecimated (a trous) 2-D analysis bank, SURVEY.md 8f row 3: afb2d_atrous (pw/dwt/lowlevel.py:475-521, afb1d_atrous
 * :175-223 along W then along H) = one level of SWTForward (pw/dwt/transform2d.py:151-212), and its adjoint.
 * b200w_swt2d_fwd_f32: x dense (planes, H, W) -> y dense (planes, 4, H, W), band order (W-filter, H-filter) =
 *   (lo,lo), (lo,hi), (hi,lo), (hi,hi) -- the channel order of the reference's two grouped convolutions; taps as stored
 *   by prep_filt_afb2d (time-reversed), `w_*` along W (the reference's h*_row), `h_*` along H (h*_col); `dilation` = 2^level.
 *   Modes: zero, symmetric, reflect, periodic (mypad has no 'periodization': B200W_ERR_BAD_MODE, as the reference raises).
 * b200w_swt2d_bwd_f32: dx = adjoint applied to dy (planes, 4, H, W) -- what autograd derives from mypad + F.conv2d.
 */
int b200w_swt2d_fwd_f32(const float* x, int planes, int H, int W, const float* w_lo, const float* w_hi,
                        const float* h_lo, const float* h_hi, int L, int dilation, int mode, float* y, void* stream);
int b200w_swt2d_bwd_f32(const float* dy, int planes, int H, int W, const float* w_lo, const float* w_hi,
                        const float* h_lo, const float* h_hi, int L, int dilation, int mode, float* dx, void* stream);

/*
 * Undecimated (a trous) 2-D synthesis, one level of SWTInverse (DESIGN.md K12): the exact inverse of SWTForward with
 * mode 'periodic', the only extension for which an undecimated synthesis bank is exact (hence no mode argument).
 * With pl = floor(L * dilation / 2) - dilation,
 *   x[r][c] = sum_{a,e} sum_{jh,jw} (h_e[jh] / 2) (w_a[jw] / 2) y_{2a+e}[(r - d jh + pl) mod H][(c - d jw + pl) mod W]
 * where y_0 = ll and y_1..y_3 = bands 1..3 of `y`.
 *   ll: (planes, H, W), unit column stride, plane stride `ll_ps` elements (4 H W when ll is band 0 of the coarsest
 *       level's coefficients, H W for a reconstructed level); `y`: dense (planes, 4, H, W), band 0 is not read;
 *   x: dense (planes, H, W).  Taps: synthesis taps as prep_filt_sfb2d stores them (not reversed), `w_*` along W (g*_row),
 *   `h_*` along H (g*_col); the factor 1/2 per axis is applied inside.  The shapes are those b200w_swt2d_fwd_* accepts:
 *   2 <= L <= B200W_MAX_TAPS, dilation >= 1, H * W < 2^31, floor(L * dilation / 2) <= 3 * min(H, W).
 *   Both return the same codes, in the same order, before any launch.
 */
int b200w_iswt2d_f32(const float* ll, int64_t ll_ps, const float* y, int planes, int H, int W, const float* w_lo,
                     const float* w_hi, const float* h_lo, const float* h_hi, int L, int dilation, float* x, void* stream);
int b200w_iswt2d_f64(const double* ll, int64_t ll_ps, const double* y, int planes, int H, int W, const double* w_lo,
                     const double* w_hi, const double* h_lo, const double* h_hi, int L, int dilation, double* x,
                     void* stream);

/*
 * Double twins of the 1-D, a trous and TV entry points above (the reference's double mode: modules built under
 * torch.set_default_dtype(torch.float64), or double images for TVLoss): the same arguments, status codes and order of
 * the checks, on double data with double taps; the kernels are the fp32 ones instantiated for double.
 * b200w_afb1d_f64 / b200w_sfb1d_f64       pw/dwt/lowlevel.py:368-424, 697-743  AFB1D / SFB1D
 * b200w_swt2d_fwd_f64 / b200w_swt2d_bwd_f64 pw/dwt/lowlevel.py:175-223, 475-521 afb2d_atrous / SWTForward
 * b200w_tv_fwd_f64 / b200w_tv_bwd_f64     model.py:17-33  TVLoss; out2, grad_out (device), ch and cw are double, the
 *   workspace is b200w_tv_workspace_bytes_f64(planes, H) bytes (double partials).
 */
int b200w_afb1d_f64(const double* x, int64_t x_rs, int rows, int n, const double* h0, const double* h1, int L, int mode,
                    double* lo, double* hi, void* stream);
int b200w_sfb1d_f64(const double* lo, int64_t lo_rs, const double* hi, int rows, int m, const double* g0,
                    const double* g1, int L, int mode, int out_len, double* y, void* stream);
int b200w_swt2d_fwd_f64(const double* x, int planes, int H, int W, const double* w_lo, const double* w_hi,
                        const double* h_lo, const double* h_hi, int L, int dilation, int mode, double* y, void* stream);
int b200w_swt2d_bwd_f64(const double* dy, int planes, int H, int W, const double* w_lo, const double* w_hi,
                        const double* h_lo, const double* h_hi, int L, int dilation, int mode, double* dx, void* stream);
size_t b200w_tv_workspace_bytes_f64(int planes, int H);
int b200w_tv_fwd_f64(const double* x, int planes, int H, int W, void* workspace, size_t workspace_bytes,
                     double* out2, void* stream);
int b200w_tv_bwd_f64(const double* x, const double* grad_out, double ch, double cw, int planes, int H, int W,
                     double* dx, void* stream);

/*
 * SSIM in double precision, ssim.py:17-37 on double images (b200w_ssim_fwd_f64) and the closed form of autograd
 * through it (b200w_ssim_bwd_f64).  The arguments, status codes and order of the checks are those of
 * b200w_ssim_fwd_f32 / b200w_ssim_bwd_f32 except:
 *   - win2d: ws x ws HOST doubles, row-major, the DENSE 2-D window.  In double the reference applies the fp32 rounding
 *     of the outer product of the 1-D Gaussian (ssim.py:11-15: .float(), then type_as), which is not separable; the
 *     kernels apply the taps they are given.  They are copied into the parameter block.
 *   - img1, img2, maps, out, grad_out, d1, d2 are double; out is 1 or N doubles.
 *   - workspace: DEVICE scratch of at least b200w_ssim_workspace_bytes_f64() bytes (double per-CTA partials, reduced
 *     in a fixed order: bit-reproducible).
 */
size_t b200w_ssim_workspace_bytes_f64(int N, int C, int H, int W);
int b200w_ssim_fwd_f64(const double* img1, const double* img2, int N, int C, int H, int W,
                       const double* win2d, int ws, int size_average,
                       int n_maps, double* maps, double* out,
                       void* workspace, size_t workspace_bytes, void* stream);
int b200w_ssim_bwd_f64(const double* img1, const double* img2, const double* maps, int n_maps,
                       const double* grad_out, int N, int C, int H, int W,
                       const double* win2d, int ws, int size_average,
                       double* d1, double* d2, void* stream);

/*
 * MS-SSIM, one scale (b200wave.ms_ssim chains them).  The arguments, status codes and order of the checks are those of
 * b200w_ssim_fwd_f32 / b200w_ssim_bwd_f32 (and _f64, with the dense window), except:
 *   - out / grad_out: always N per-sample values (means over C, H, W); there is no size_average.
 *   - cs != 0: the value is the mean of the contrast-structure map cs = A2/B2 (= (2 sigma12 + C2) /
 *     (sigma1^2 + sigma2^2 + C2)) and maps hold its derivatives, in the same order (d/dmu1, d/dE[x^2], d/dE[x1x2],
 *     d/dmu2).  cs == 0: the SSIM map.  Either value is formed by correctly rounded division, so identical images
 *     give exactly 1.
 *   - pooled1, pooled2: DEVICE (N,C,H/2,W/2), written with avg_pool2d(img, 2) of img1 and img2 (an odd last row or
 *     column is dropped), or both NULL (no pooling).  One NULL and one not: B200W_ERR_NULL_POINTER; pooling with
 *     H < 2 or W < 2: B200W_ERR_BAD_SHAPE.
 *   - up1, up2: DEVICE (N,C,H/2,W/2) gradients of the pooled images, or NULL; the backward adds
 *     0.25 up[r/2][c/2] to d1 (d2) for r < 2 (H/2), c < 2 (W/2).  up2 without d2, or either with H < 2 or W < 2:
 *     B200W_ERR_BAD_SHAPE.
 * The workspace is that of b200w_ssim_fwd_f32 / _f64 (b200w_ssim_workspace_bytes / _f64).
 */
int b200w_msssim_scale_fwd_f32(const float* img1, const float* img2, int N, int C, int H, int W,
                               const float* win, int ws, int cs, int n_maps, float* maps, float* out,
                               float* pooled1, float* pooled2, void* workspace, size_t workspace_bytes, void* stream);
int b200w_msssim_scale_bwd_f32(const float* img1, const float* img2, const float* maps, int n_maps,
                               const float* grad_out, int N, int C, int H, int W, const float* win, int ws,
                               const float* up1, const float* up2, float* d1, float* d2, void* stream);
int b200w_msssim_scale_fwd_f64(const double* img1, const double* img2, int N, int C, int H, int W,
                               const double* win2d, int ws, int cs, int n_maps, double* maps, double* out,
                               double* pooled1, double* pooled2, void* workspace, size_t workspace_bytes,
                               void* stream);
int b200w_msssim_scale_bwd_f64(const double* img1, const double* img2, const double* maps, int n_maps,
                               const double* grad_out, int N, int C, int H, int W, const double* win2d, int ws,
                               const double* up1, const double* up2, double* d1, double* d2, void* stream);

/*
 * phase_consistency_loss, model.py:36-58 (constructed at train.py:94), SURVEY.md 8f row 4: minus the cosine
 * similarity of a_x = m * log|fft2(x[0])| and a_y = m * log|fft2(y[0])|, m = 1 - exp(-0.5 d^2 / radius^2) the Gaussian
 * high-pass mask around the spectrum centre (radius 5 in the reference).  `fx`, `fy`: HALF spectra of the real images
 * (rfft2 layout, (planes, rows, cols/2+1) interleaved complex64); mirrored bins are counted with weight 2.
 * b200w_phase_sums_c64: out3 = { <a_x,a_y>, <a_x,a_x>, <a_y,a_y> } (device floats; per-CTA partials in double in
 *   `workspace` = b200w_phase_workspace_bytes(...) bytes, reduced in fixed order).  The loss is
 *   -out3[0] / (max(sqrt(out3[1]), eps) * max(sqrt(out3[2]), eps))  (torch.cosine_similarity, eps = 1e-8).
 * b200w_phase_grad_c64: gx, gy (either may be NULL) = grad_out[0] * dLoss/d(fx), d(fy) in the d/dRe + i d/dIm convention
 *   of torch autograd, same layout as the spectra; `sums3` = out3 of the forward call.
 */
size_t b200w_phase_workspace_bytes(int planes, int rows, int cols);
int b200w_phase_sums_c64(const void* fx, const void* fy, int planes, int rows, int cols, float radius,
                         void* workspace, size_t workspace_bytes, float* out3, void* stream);
int b200w_phase_grad_c64(const void* fx, const void* fy, int planes, int rows, int cols, float radius,
                         const float* sums3, const float* grad_out, float eps, void* gx, void* gy, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200WAVE_H_ */
