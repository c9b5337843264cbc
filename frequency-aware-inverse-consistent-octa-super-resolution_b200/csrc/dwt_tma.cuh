// Parameter blocks of the TMA-staged owner kernels (dwt_tma_afb.cu / dwt_tma_sfb.cu).
//
// One CTA owns a horizontal part of one image plane for EVERY level of a multi-level transform (as the round-1 owner
// kernels did), but the rows it streams from global memory arrive through the copy engine: one elected producer lane
// per row stream issues cp.async.bulk.tensor tiles (several full-width rows per instruction) into an mbarrier-guarded
// ring, a patch warp writes the few extension columns of the padding mode next to the landed rows, and every consumer
// lane then runs the same border-free register march over 16-byte aligned shared-memory windows.  The intermediate
// low-pass images (analysis) / partial reconstructions (synthesis) stay in shared memory, stored WITH their extension
// columns, so the dependent levels have no border class either.
#pragma once
#include "dwt_levels.cuh"
#include "tma.cuh"

namespace b200w {

constexpr int kTmaMaxStreams = 8;    // row streams (segments of the streamed level) per CTA
constexpr int kTmaMaxStrips = 4;     // tiles per staged row (a tile is at most 256 floats wide)
constexpr int kAfbTabMax = 5120;     // ints of host-built tables in the analysis kernel's parameter block

// taps of the templated kernels (<= 16), W taps as constant-bank scalars, H taps once more as (t, t) pairs for FFMA2
struct TapsT {
    float w_lo[kMaxTemplTaps], w_hi[kMaxTemplTaps];
    float2 h_lo2[kMaxTemplTaps], h_hi2[kMaxTemplTaps];
};

struct AfbTmaLevel {
    float* low;            // global low-pass output (last level only)
    float* highs;          // global (planes, 3, Ho, Wo)
    int H, W;              // logical input size (including the zero extension of SFB2D.backward's 'unpad')
    int Hreal, Wreal;      // rows / columns >= these read as zero
    int Ho, Wo;
    int ncp;               // output column pairs = ceil(Wo / 2)
    int R, nseg;           // output rows per segment, segments (level 0: = row streams)
    int in_pitch;          // level >= 1: row pitch (floats, multiple of 4) of the input image in shared memory
    int in_off;            // level >= 1: byte offset of that image from the dynamic shared-memory base
    int in_rows;           // level >= 1: rows of that image (max over the parts)
    int rtab_off;          // int offset of the row table of this level's input rows inside the table area
    int cfix_off;          // level >= 1: int offset of the column-patch table (pairs dst, src) and of its counter
    int vec2, low_vec2;    // 64-bit global stores allowed
    int c0[kMaxParts], c1[kMaxParts];   // output rows a part computes
    int h0[kMaxParts], h1[kMaxParts];   // output rows a part stores to global memory (a partition of [0, Ho))
};

struct AfbTmaHead {   // everything of the analysis kernel's parameter block but the tables
    CUtensorMap map_full;  // level-0 input (W, H, planes), box {BW, SR, 1}
    CUtensorMap map_row;   // the same tensor, box {BW, 1, 1}: rows the padding mode maps somewhere else
    AfbTmaLevel lv[kMaxLevels];
    TapsT t;
    int J, planes, parts, mode;
    int D, nstrips, cps, BW;   // ring: stages, tiles per row, column pairs per tile, tile width (floats, multiple of 32)
    int boxes;                 // 1: every ring stage is one box of consecutive (virtual) rows (see the kernel)
    int rp0_off, rp0_stride;   // per-pair row-address table of the first level: int offset, int2 entries per stream
    int fix0_off, fix0_n;      // int offset of the ring's column-patch table (int2 per stage row x extension column) and
                               // the extension columns per stage row
    int bar_off, tab_off, zrow_off, ring_off;   // shared-memory layout (bytes from the dynamic base)
    int zrow_floats, tab_ints;
    int smem_bytes;
};
// the row / patch tables of every part, built on the host (part q's tab_ints entries start at q * tab_ints): a CTA
// only copies its part's share into shared memory instead of spending ~2 us of set-up on index arithmetic.
// The whole parameter block travels with every launch, and its size shows up between kernels: at cfg2 (1444 table
// ints) a 10.6 KB block instead of 22.9 KB makes the four-launch step 2.4 us shorter.  So the kernel is built for two
// table capacities and the launch picks the smaller one the plan fits in.
template <int N>
struct AfbTmaParamsN : AfbTmaHead {
    int tab[N];
};
constexpr int kAfbTabSmall = 2048;
using AfbTmaParams = AfbTmaParamsN<kAfbTabMax>;   // what the plan fills
static_assert(sizeof(AfbTmaParams) <= 32764, "kernel parameter block (CUDA 12.1+: 32764 bytes)");

// ---- synthesis ---------------------------------------------------------------------------------------------------
// Chain positions run coarsest first.  The detail rows a part needs are contiguous in global memory (dense
// (planes, 3, h, w) tensors), so they come in as plain bulk copies (cp.async.bulk, one per band): the copy covers the
// 16-byte aligned superset of the rows and the data sits 0..3 floats into the destination, rows dense at pitch w --
// any width, any row alignment.  Every position but the last is "resident" (all its rows fetched at kernel start); the
// last, finest position streams its rows through per-stream mbarrier rings.
struct SfbTmaPos {
    float* y;              // global output (last position only)
    const float* highs;    // global (planes, 3, h, w)
    int h, w, out_h, out_w;
    int nq;                // lanes per segment = ceil(out_w / 4)
    int Rp, nseg;          // output row pairs per segment, segments
    int v2;                // detail rows are 8-byte aligned in shared memory (even w): 64-bit window loads
    int res_off, res_band; // resident positions: byte offset of the detail rows, bytes reserved per band
    int y_off, y_pitch, y_rows;   // output image in shared memory (all positions but the last): byte offset, pitch, rows
    int vec4;              // 128-bit global stores allowed (last position)
    int n0[kMaxParts], n1[kMaxParts];   // output rows [n0, n1) a part computes
    int k0[kMaxParts], k1[kMaxParts];   // coefficient rows [k0, k1) it reads
};

struct SfbTmaParams {
    SfbTmaPos pos[kMaxLevels];
    TapsT t;
    const float* yl;                  // dense (planes, h, w) low-pass input of the first position
    int J, planes, parts;
    int D, SR;                        // ring stages of the last position, coefficient rows per stage
    int ring_band;                    // bytes reserved per band inside a ring stage
    int low_off;                      // resident yl rows (first position)
    int bar_off, ring_off;
    int smem_bytes;
};
static_assert(sizeof(SfbTmaParams) <= 4096, "kernel parameter block");

// G / D > 0 replace the plan's row streams of the last position / ring stages (DwtPolicy::tma_G / tma_D)
bool sfb_tma_plan(const SfbParams& p, int L, int sms, bool force, int G, int D, SfbTmaParams& tp);
int launch_sfb_tma(const SfbTmaParams& tp, int L, cudaStream_t st);

// planning + launch (dwt_tma_afb.cu).  afb_tma_plan returns false when the shapes do not qualify (unaligned rows, the
// low-pass images do not fit, the driver has no tensor-map entry point, ...): the caller then takes the other kernels.
// G / D > 0 replace the plan's row streams / ring stages; `noboxes` fetches every extension row from its source row.
bool afb_tma_plan(const AfbParams& p, int L, int sms, bool force, int G, int D, bool noboxes, AfbTmaParams& tp);
int launch_afb_tma(const AfbTmaParams& tp, int L, cudaStream_t st);

}  // namespace b200w
