// Undecimated ("a trous") 2-D synthesis bank for sm_100a: one level of SWTInverse, the inverse of SWTForward in
// periodic mode.  The reference has no usable inverse (pw/dwt/swt_inverse.py is unfinished and not exported), so the
// semantics are this library's (DESIGN.md K12).  With d = dilation and pl = floor(L d / 2) - d (the forward's front
// padding), one level reconstructs
//     x[r][c] = sum_{a,e} sum_{jh,jw} (gH_e[jh] / 2) (gW_a[jw] / 2) y_{2a+e}[(r - d jh + pl) mod H][(c - d jw + pl) mod W]
// from y_0 = ll (the low band of the coarser level) and bands 1..3 of this level's coefficients; gW = (g0_row, g1_row)
// runs along W, gH = (g0_col, g1_col) along H, the synthesis taps as prep_filt_sfb2d stores them.  Only periodic
// extension has an exact undecimated inverse, so there is no mode argument.
//
// Separable two-pass kernel.  A CTA owns output rows rho_r + d (m0 + m), m < kRows (one residue class mod d: the H
// halo is L - 1 staged rows at any dilation) and output columns c0 + rho + d (n0 + n), rho < R, n < TN.  R = min(d, 32)
// consecutive residues keep every warp's loads and stores on consecutive columns; for d <= 32 the tile is simply
// d * TN contiguous columns.  The W halo is then R (L - 1) staged columns, independent of d.
//   H pass: one thread per staged column walks the kRows + L - 1 staged rows (4 coalesced loads each: ll and bands
//     1..3, rows / columns taken mod H / W) and accumulates the two W-streams t_a = sum_e gH_e / 2 * y_{2a+e} of the
//     kRows output rows in registers, then stores them to shared memory.
//   W pass: out = sum_jw gW_0[jw] / 2 * t_0 + gW_1[jw] / 2 * t_1 at staged column n + L - 1 - jw, conflict-free
//     (consecutive threads read consecutive words), one coalesced store per output.
// About 6 L FMAs per output; HBM traffic is 4 planes read + 1 written (the staged halos are served by L1 / L2).
#include "common.cuh"

namespace b200w {

constexpr int kIswtRows = 8;                 // output rows per CTA (register accumulators per W-stream)
constexpr int kIswtCols = 512;               // output columns per CTA (R * TN)
constexpr int kIswtMaxRes = 32;              // residues per CTA when d > 1
constexpr size_t kIswtSmemBudget = 96 * 1024;

template <typename T>
struct IswtParams {
    const T* ll;          // (planes, H, W) with plane stride ll_ps
    const T* y;           // dense (planes, 4, H, W); bands 1..3 are read
    T* x;                 // dense (planes, H, W)
    long long ll_ps;
    int planes, H, W, L, d, pl;
    int R, TN;            // column tile: R residues x TN steps of d
    int n_res_blocks;     // column tiles per step block: ceil(min(d, W) / R)
    int n_col_tiles;      // n_res_blocks * ceil(ceil(W / d) / TN)
    int n_row_res;        // min(d, H): row residue classes
    int QS;               // staged columns: R * (TN + L - 1)
    T w_lo[kMaxTaps], w_hi[kMaxTaps], h_lo[kMaxTaps], h_hi[kMaxTaps];   // halved synthesis taps
};

__device__ __forceinline__ int pmod(long long a, int n) {
    long long m = a % n;
    return (int)(m < 0 ? m + n : m);
}

template <typename T>
__global__ void __launch_bounds__(kThreads) iswt2d_kernel(const __grid_constant__ IswtParams<T> p) {
    extern __shared__ __align__(16) unsigned char iswt_smem[];
    T* t = reinterpret_cast<T*>(iswt_smem);                                   // [2][kIswtRows][QS]
    int* srow = reinterpret_cast<int*>(t + 2 * kIswtRows * p.QS);             // [kIswtRows + L - 1] row offsets
    const int L = p.L, d = p.d, R = p.R, QS = p.QS;
    const int nstage = kIswtRows + L - 1;

    const int ct = (int)(blockIdx.x % (unsigned)p.n_col_tiles);
    const int rt = (int)(blockIdx.x / (unsigned)p.n_col_tiles);
    const int res0 = (ct % p.n_res_blocks) * R;                // first column residue of the tile
    const long long n0 = (long long)(ct / p.n_res_blocks) * p.TN;
    const int rho_r = rt % p.n_row_res;
    const long long m0 = (long long)(rt / p.n_row_res) * kIswtRows;
    const long long row0 = rho_r + d * m0;                     // first output row of the tile
    if (row0 >= p.H) return;
    // staged row v / column (rho, s) hold input row / column (output + pl) + d (v - (L - 1)) / d (s - (L - 1))
    const long long rbase = row0 + p.pl - (long long)d * (L - 1);
    const long long cbase = res0 + d * (n0 - (L - 1)) + p.pl;
    const size_t plane_px = (size_t)p.H * p.W;

    for (int i = threadIdx.x; i < nstage; i += blockDim.x) srow[i] = pmod(rbase + (long long)d * i, p.H) * p.W;
    __syncthreads();

    for (int plane = blockIdx.y; plane < p.planes; plane += gridDim.y) {
        const T* __restrict__ y0 = p.ll + plane * p.ll_ps;
        const T* __restrict__ yb = p.y + (size_t)plane * 4 * plane_px;
        for (int q = threadIdx.x; q < QS; q += blockDim.x) {
            const int rho = q % R, s = q / R;
            const int col = pmod(cbase + rho + (long long)d * s, p.W);
            T a0[kIswtRows], a1[kIswtRows];
#pragma unroll
            for (int m = 0; m < kIswtRows; ++m) a0[m] = a1[m] = T(0);
            for (int v = 0; v < nstage; ++v) {
                const int off = srow[v] + col;
                const T v0 = __ldg(y0 + off), v1 = __ldg(yb + plane_px + off), v2 = __ldg(yb + 2 * plane_px + off),
                        v3 = __ldg(yb + 3 * plane_px + off);
#pragma unroll
                for (int m = 0; m < kIswtRows; ++m) {
                    const int jh = m + L - 1 - v;
                    if ((unsigned)jh < (unsigned)L) {
                        a0[m] = fma(p.h_lo[jh], v0, fma(p.h_hi[jh], v1, a0[m]));
                        a1[m] = fma(p.h_lo[jh], v2, fma(p.h_hi[jh], v3, a1[m]));
                    }
                }
            }
#pragma unroll
            for (int m = 0; m < kIswtRows; ++m) {
                t[m * QS + q] = a0[m];
                t[(kIswtRows + m) * QS + q] = a1[m];
            }
        }
        __syncthreads();
        T* __restrict__ xp = p.x + (size_t)plane * plane_px;
        for (int rem = threadIdx.x; rem < R * p.TN; rem += blockDim.x) {
            const int rho = rem % R, n = rem / R;
            const long long col = res0 + rho + d * (n0 + n);
            if (res0 + rho >= d || col >= p.W) continue;
            const T* t0 = t + rem + R * (L - 1);
            for (int m = 0; m < kIswtRows; ++m) {
                const long long row = row0 + (long long)d * m;
                if (row >= p.H) break;
                const T* u0 = t0 + m * QS;
                const T* u1 = u0 + kIswtRows * QS;
                T acc = 0;
                for (int jw = 0; jw < L; ++jw) acc = fma(p.w_lo[jw], u0[-R * jw], fma(p.w_hi[jw], u1[-R * jw], acc));
                xp[row * p.W + col] = acc;
            }
        }
        __syncthreads();   // the next plane overwrites the staged streams
    }
}

template <typename T>
static size_t iswt_smem_bytes(int R, int TN, int L) {
    return sizeof(T) * 2 * kIswtRows * (size_t)R * (TN + L - 1) + sizeof(int) * (kIswtRows + L - 1);
}

// the fp32 and fp64 entry points share their checks (same codes, same order) and their launch
template <typename T>
static int iswt2d_run(const T* ll, int64_t ll_ps, const T* y, int planes, int H, int W, const T* w_lo, const T* w_hi,
                      const T* h_lo, const T* h_hi, int L, int dilation, T* x, void* stream) {
    if (!ll || !y || !x || !w_lo || !w_hi || !h_lo || !h_hi) return B200W_ERR_NULL_POINTER;
    if (planes < 1 || H < 1 || W < 1 || dilation < 1 || (long long)H * W > 0x7fffffffLL || ll_ps < (long long)H * W)
        return B200W_ERR_BAD_SHAPE;
    if (L < 1 || L > kMaxTaps) return B200W_ERR_BAD_TAPS;
    const long long L2 = ((long long)L * dilation) / 2;
    if (L2 - dilation < 0) return B200W_ERR_BAD_TAPS;            // a single tap: negative padding, as swt_fill
    if (L2 > 3LL * (H < W ? H : W)) return B200W_ERR_BAD_SHAPE;   // the shapes SWTForward (swt_fill) accepts
    IswtParams<T> p = {};
    p.ll = ll;
    p.y = y;
    p.x = x;
    p.ll_ps = ll_ps;
    p.planes = planes;
    p.H = H;
    p.W = W;
    p.L = L;
    p.d = dilation;
    p.pl = (int)(L2 - dilation);
    for (int j = 0; j < L; ++j) {   // halving is exact
        p.w_lo[j] = w_lo[j] / 2;
        p.w_hi[j] = w_hi[j] / 2;
        p.h_lo[j] = h_lo[j] / 2;
        p.h_hi[j] = h_hi[j] / 2;
    }
    // column tile: R residues x TN steps; fewer residues (less coalescing) only where long filters need the room
    int R = dilation < kIswtMaxRes ? dilation : kIswtMaxRes;
    const long long steps = (W + (long long)dilation - 1) / dilation;   // columns per residue, at most
    int TN = kIswtCols / R;
    if (TN > steps) TN = (int)steps;
    while (R > 1 && iswt_smem_bytes<T>(R, TN, L) > kIswtSmemBudget) R = (R + 1) / 2;
    p.R = R;
    p.TN = TN;
    p.QS = R * (TN + L - 1);
    const int res = dilation < W ? dilation : W;
    p.n_res_blocks = (res + R - 1) / R;
    const long long col_tiles = (long long)p.n_res_blocks * ((steps + TN - 1) / TN);
    p.n_row_res = dilation < H ? dilation : H;
    const long long row_steps = (H + (long long)dilation - 1) / dilation;
    const long long row_tiles = (long long)p.n_row_res * ((row_steps + kIswtRows - 1) / kIswtRows);
    if (col_tiles * row_tiles > 0x7fffffffLL) return B200W_ERR_BAD_SHAPE;
    p.n_col_tiles = (int)col_tiles;
    const size_t smem = iswt_smem_bytes<T>(R, TN, L);
    auto kern = iswt2d_kernel<T>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_last_cuda_error(e);
    const dim3 grid((unsigned)(col_tiles * row_tiles), (unsigned)(planes < 65535 ? planes : 65535), 1);
    kern<<<grid, kThreads, smem, (cudaStream_t)stream>>>(p);
    note_launch(sizeof(T) == 8 ? "iswt2d_kernel<double>" : "iswt2d_kernel");
    e = cudaGetLastError();
    return e == cudaSuccess ? B200W_OK : set_last_cuda_error(e);
}

}  // namespace b200w

using namespace b200w;

extern "C" int b200w_iswt2d_f32(const float* ll, int64_t ll_ps, const float* y, int planes, int H, int W,
                                const float* w_lo, const float* w_hi, const float* h_lo, const float* h_hi, int L,
                                int dilation, float* x, void* stream) {
    return iswt2d_run(ll, ll_ps, y, planes, H, W, w_lo, w_hi, h_lo, h_hi, L, dilation, x, stream);
}

extern "C" int b200w_iswt2d_f64(const double* ll, int64_t ll_ps, const double* y, int planes, int H, int W,
                                const double* w_lo, const double* w_hi, const double* h_lo, const double* h_hi, int L,
                                int dilation, double* x, void* stream) {
    return iswt2d_run(ll, ll_ps, y, planes, H, W, w_lo, w_hi, h_lo, h_hi, L, dilation, x, stream);
}
