// Internal launch interface of the tcgen05 implicit-GEMM kernels (igemm2.cu, wgrad.cu, wgrad3.cu).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cesm {

struct WgradParams {
    int32_t c0, c1;
    int32_t num_taps;
    int32_t tap_map[16];
    int32_t tap_dh[16];
    int32_t tap_dw[16];
    int32_t n, oh, ow;      // pixel grid contracted over
    int32_t bw, bh, bn;     // 64-pixel K tile box (bw*bh*bn == 64)
    uint32_t box_bytes;     // bytes of one 64-channel x 64-pixel TMA box
    int32_t cout;
    float* dw;              // fp32, accumulated with red.add at dw[co*so + ci*si + tap_off[tap]]
    long long so, si;
    int32_t tap_off[16];
};

// ---- 3x3 weight gradient with halo reuse (wgrad3.cu) -------------------------------------------------
struct Wgrad3Maps {
    CUtensorMap x[2];   // box {64 ci, bw + 2, bh + 2, 1}
    CUtensorMap y;      // box {64 co, bw, bh, 1}
};
struct Wgrad3Params {
    int32_t c0, c1;
    int32_t n, cout;
    int32_t bw, bh;              // pixel tile: bw * bh == 128, bw in {16, 32}
    int32_t tiles_w, tiles_h;
    uint32_t halo_box_bytes;     // (bw + 2) * (bh + 2) * 128
    uint32_t halo_stage_bytes;   // the same rounded up to 1024 (+ slack for the ghost tap's view)
    int32_t tap_row[10];         // halo row of pixel (0, 0) for each tap, ascending; [9] = ghost of the last pair
    int32_t tap_off[10];         // offset of that tap in dw
    float* dw;                   // fp32, red.add at dw[co*so + ci*si + tap_off[tap]]
    long long so, si;
};
cudaError_t wgrad3_launch(const Wgrad3Maps& maps, const Wgrad3Params& p, int cblk, int ksplit, cudaStream_t stream);

// ---- second-generation persistent kernel (igemm2.cu) ------------------------------------------
static constexpr size_t kIgemm2MaxSmem = 232448;  // 227 KB opt-in limit per CTA on sm_100

struct Igemm2Maps {
    CUtensorMap a[4];
    CUtensorMap b;
    CUtensorMap out;
};

struct Igemm2Params {
    int32_t c0, c1;
    int32_t num_taps, num_kb;          // num_kb = num_taps * (c0 + c1) / 64
    int32_t tap_map[16];
    int32_t tap_dh[16];
    int32_t tap_dw[16];
    int32_t n, oh, ow;                 // output pixel space
    int32_t bw, bh, bn;                // useful pixels of a tile (HALO: accumulator rows are (bw+2) wide)
    int32_t tiles_w, tiles_h, m_tiles, n_tiles;
    int32_t cout;
    // shared-memory plan
    int32_t a_stages, b_stages, b_resident;
    uint32_t a_stage_bytes, a_box_bytes;
    // epilogue
    int32_t out_h, out_w, o_sh, o_sw, o_h0, o_w0;   // residual addressing (same pixel map as the output)
    const float* bias;
    const void* residual;
    int32_t ldr;
    float* gn_sums;                    // [B][gn_groups][2] (sum, sum of squares) or null
    int32_t gn_groups, gn_cpg, gn_frames;
    int32_t epi_warp;                  // 1: every epilogue warp stores its own 32-row slab (see igemm2.cu)
    int32_t m_major;                   // 1: consecutive tiles are the column tiles of ONE row tile (resident weights)
    const float* ln_colsum;            // LayerNorm folded into a 64 -> 64 projection (see cesm_igemm_args) or null
    float ln_eps;
};

// pair: launch as clusters of two CTAs working as one cta_group::2 unit (halo mode only; grid must be even)
cudaError_t igemm2_launch(const Igemm2Maps& maps, const Igemm2Params& p, int block_n, bool halo, bool pair, int grid,
                          size_t smem, cudaStream_t stream);   // p.ln_colsum != null: the LayerNorm-fold epilogue (block_n 64)

// pair: clusters of two CTAs along the (tap, ci) blocks working as one cta_group::2 unit (block_n >= 128)
cudaError_t wgrad_launch(const CUtensorMap* xmaps, int n_xmaps, const CUtensorMap& ymap, const WgradParams& p,
                         int block_n, int ksplit, bool pair, cudaStream_t stream);

}  // namespace cesm
