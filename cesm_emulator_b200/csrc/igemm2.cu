// Persistent tcgen05 / TMEM / TMA implicit GEMM for sm_100a: every forward and data-gradient contraction.
//
//     out[pixel, co] = sum_{tap, ci} A[pixel + tap, ci] * Wt[co, tap, ci]   (+ bias) (+ residual)
//
// What bounds these contractions on B200 is not the tensor pipe but the L2 -> shared-memory feed:
// a 128 x 64 tile needs 24 KB of operands per 128 MMA cycles when every tap re-fetches its pixels
// and its weights (~190 B/clk/SM against ~42 B/clk/SM of L2 bandwidth per SM).  This kernel removes
// that traffic instead of hiding it:
//
//   * HALO mode (3x3, stride 1): the (bw+2) x (bh+2) pixel halo of a tile is fetched ONCE per 64
//     input channels; the nine taps are nine row-shifted views of it (UMMA descriptors whose start
//     address is advanced by whole 128-byte rows -- exact on B200, tools/probe_umma_desc.cu).  The
//     accumulator rows live on the padded (bw+2)-wide grid; the two pad columns are dropped by
//     the epilogue.  A traffic: 9 x -> ~1.6 x.
//   * resident weights: when cout x K fits, the whole weight matrix is loaded once per CTA and
//     stays in shared memory across the persistent tile loop; otherwise it is streamed through its
//     own mbarrier ring, decoupled from the activation ring.
//   * persistent CTAs (one per SM) with two TMEM accumulator stages: the epilogue of tile i overlaps
//     the MMAs of tile i+1; a stage is handed back as soon as tcgen05.ld has it in registers.
//   * the epilogue goes TMEM -> registers -> swizzled shared memory -> TMA store (full 128-byte
//     lines), fusing bias, residual add and -- for the convs that feed a GroupNorm -- the per-sample
//     per-group sum / sum-of-squares of the fp16-rounded outputs (video_net.py:216), kept in registers
//     across tiles and reduced once per (sample, column tile).
//   * (round 2) ONE elected thread runs the MMA issue loop: its instruction stream is the critical path
//     (a 128x64x16 MMA is 32 tensor clocks), so the loop carries no per-MMA predicate and no per-tap branch.
//   * (round 2) PAIR mode for the 3x3 convolutions: the two CTAs of a cluster work as one cta_group::2
//     unit on two row tiles of the same column tile (M = 256).  What bounds a 128 x N x 16 SS-mode MMA is
//     the shared-memory operand feed (~77-90 B/clk measured: 4 KB of A + N*32 B of B per MMA); in a pair
//     each CTA supplies its own A rows and HALF of the B rows.  Only the even CTA issues; TMA loads of
//     both CTAs report to its barriers (peer bit of the barrier address cleared), commits are multicast,
//     the epilogues of both return the accumulator stage to the leader's barrier.
//
// Warp roles (352 threads): 0 = activation TMA producer, 1 = weight TMA producer, 2 = MMA issuer
// (+ TMEM allocation), 3..10 = epilogue: two groups of four warps (warp w reads TMEM lanes
// 32*(w%4)..+31), the groups alternating over the 64-column chunks of a tile.

#include "api_common.h"
#include "common.cuh"
#include "igemm.h"

#include <type_traits>

namespace cesm {

static constexpr int kTileM = 128;
static constexpr int kKBlk = 64;
static constexpr int kStageRowBytes = 128;                       // 64 fp16
static constexpr int kOutStageBytes = kTileM * kStageRowBytes;   // one 64-column output chunk
static constexpr int kIgemm2Threads = 352;

__device__ __forceinline__ void tma_store_4d(const void* map, uint32_t smem_src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 :
                 : "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// named barrier of one epilogue group (4 warps): ids 1 and 2
__device__ __forceinline__ void epi_bar_sync(int group) {
    asm volatile("bar.sync %0, 128;" ::"r"(group + 1) : "memory");
}
__device__ __forceinline__ void epi_bar_sync_all() { asm volatile("bar.sync 3, 256;" ::: "memory"); }
// 32 lanes x 64 consecutive fp32 columns in one instruction
__device__ __forceinline__ void tmem_ld_32x64(uint32_t taddr, uint32_t (&v)[64]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
        "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
        "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]),
          "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]),
          "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]),
          "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]),
          "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
        : "r"(taddr)
        : "memory");
}

// PAIR (HALO only): the two CTAs of a cluster work as one cta_group::2 unit on TWO row tiles (CTA r takes row tile
// 2*pair + r) of the same column tile.  Each CTA loads its own activation halo and HALF of the weight rows, keeps
// its own 128 accumulator rows in its own TMEM and runs its own epilogue; the even CTA issues the M = 256 MMAs.
// LNF (64 -> 64, one tap, residual = the GEMM input x): the channel LayerNorm of x is folded into the epilogue,
// out = x + rstd(x) * (x W'^T - mean(x) * colsum(W')) -- a thread holds a whole 64-channel row of x as its
// residual, so the row statistics cost no extra pass (the temporal-attention block at one frame is this ONE kernel).
template <int BLOCK_N, bool HALO, bool GN, bool PAIR, bool LNF = false>
__global__ void __launch_bounds__(kIgemm2Threads, 1)
igemm2_kernel(const __grid_constant__ Igemm2Maps maps, const Igemm2Params p) {
    static_assert(!PAIR || HALO, "CTA pairs are wired for the 3x3 halo mode only");
    static_assert(!LNF || (BLOCK_N == 64 && !HALO && !GN && !PAIR), "the LayerNorm fold is a 64-column plain GEMM epilogue");
    pdl_trigger();  // pdl_wait() sits in the two TMA producers: everything else depends on their data
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

    const uint32_t a_base = smem_base;
    const uint32_t b_base = a_base + p.a_stages * p.a_stage_bytes;
    constexpr int kBRows = PAIR ? BLOCK_N / 2 : BLOCK_N;      // weight rows of a block held by THIS CTA
    const uint32_t b_blk_bytes = kBRows * kStageRowBytes;
    const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;  // 0 = leader (issues the MMAs, owns the full barriers)
    const int work_id = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;     // persistent loop: first unit ...
    const int work_stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;   // ... and stride (CTAs or CTA pairs)
    const uint32_t b_bytes = p.b_resident ? (uint32_t)p.n_tiles * p.num_kb * b_blk_bytes : p.b_stages * b_blk_bytes;
    const uint32_t o_base = b_base + b_bytes;                 // 2 output staging buffers
    const uint32_t bar_base = o_base + 2 * kOutStageBytes;
    // barrier map
    auto a_full = [&](int s) { return bar_base + 8u * s; };
    auto a_empty = [&](int s) { return bar_base + 8u * (8 + s); };
    auto b_full = [&](int s) { return bar_base + 8u * (16 + s); };
    auto b_empty = [&](int s) { return bar_base + 8u * (32 + s); };
    auto t_full = [&](int s) { return bar_base + 8u * (48 + s); };
    auto t_empty = [&](int s) { return bar_base + 8u * (50 + s); };
    const uint32_t b_all_bar = bar_base + 8u * 52;
    const uint32_t tmem_ptr_addr = bar_base + 8u * 53;
    const uint32_t gn_base = bar_base + 8u * 56;  // 2 x 64 floats: per-epilogue-group GroupNorm (sum, sumsq) accumulators
    volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_ptr_addr - smem_base));

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    const int cblk0 = p.c0 >> 6;
    const int cblk = (p.c0 + p.c1) >> 6;
    const int a_loads = HALO ? cblk : p.num_kb;    // activation loads per tile
    const int taps_per_a = HALO ? 9 : 1;
    const int pw = HALO ? p.bw + 2 : p.bw;         // accumulator rows per tile row
    const int m_units = PAIR ? (p.m_tiles + 1) >> 1 : p.m_tiles;   // row tiles, or pairs of row tiles
    const int total_tiles = m_units * p.n_tiles;
    constexpr uint32_t kTmemCols = (2 * BLOCK_N < 32) ? 32 : 2 * BLOCK_N;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&maps.a[0]);
        tma_prefetch_desc(&maps.b);
        tma_prefetch_desc(&maps.out);
        for (int s = 0; s < p.a_stages; ++s) {
            mbar_init(a_full(s), 1);
            mbar_init(a_empty(s), 1);
        }
        for (int s = 0; s < p.b_stages; ++s) {
            mbar_init(b_full(s), 1);
            mbar_init(b_empty(s), 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(t_full(s), 1);
            mbar_init(t_empty(s), (BLOCK_N == 64 ? 4 : 8) * (PAIR ? 2 : 1));   // PAIR: both CTAs' epilogues
        }
        mbar_init(b_all_bar, 1);
        fence_barrier_init();
    }
    if (threadIdx.x < 128) reinterpret_cast<float*>(smem_gen + (gn_base - smem_base))[threadIdx.x] = 0.f;
    if (warp == 2) {
        if (PAIR) tmem_alloc_pair(tmem_ptr_addr, kTmemCols);
        else tmem_alloc(tmem_ptr_addr, kTmemCols);
    }
    tc_fence_before();
    if (PAIR) cluster_sync_all();   // the peer's barriers are initialised before anything signals them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;

    auto tile_coords = [&](int tile, int& n_tile, int& n0, int& oh0, int& ow0) {
        // n-major (streamed weights): concurrently running CTAs share the weight tile.  m-major (resident
        // weights): neighbouring CTAs write the column tiles of the same rows at the same time, so every
        // output row is completed in one go instead of in n_tiles passes over the whole tensor.
        int t;
        if (p.m_major) {
            t = tile / p.n_tiles;
            n_tile = tile - t * p.n_tiles;
        } else {
            n_tile = tile / m_units;
            t = tile - n_tile * m_units;
        }
        if (PAIR) t = 2 * t + (int)cta_rank;   // may be == m_tiles (odd count): a ghost tile, all out of bounds
        const int tw = t % p.tiles_w;
        t /= p.tiles_w;
        const int th = t % p.tiles_h;
        const int tn = t / p.tiles_h;
        ow0 = tw * p.bw;
        oh0 = th * p.bh;
        n0 = tn * p.bn;
    };

    if (warp == 0 && lane == 0) {
        // ===== activation producer =====
        pdl_wait();  // the preceding kernel has completed: its outputs (our activations) are visible
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = work_id; tile < total_tiles; tile += work_stride) {
            int n_tile, n0, oh0, ow0;
            tile_coords(tile, n_tile, n0, oh0, ow0);
            for (int ai = 0; ai < a_loads; ++ai) {
                mbar_wait(a_empty(stage), phase ^ 1u, 11);
                const uint32_t dst = a_base + stage * p.a_stage_bytes;
                if (PAIR) {
                    // both halos report to the leader's barrier, which expects the bytes of both
                    if (cta_rank == 0) mbar_arrive_expect_tx(a_full(stage), 2 * p.a_box_bytes);
                    int midx = 0, c = ai << 6;
                    if (ai >= cblk0) {
                        midx = 1;
                        c = (ai - cblk0) << 6;
                    }
                    tma_load_4d_pair(dst, &maps.a[midx], a_full(stage), c, ow0 - 1, oh0 - 1, n0);
                    if (++stage == p.a_stages) {
                        stage = 0;
                        phase ^= 1u;
                    }
                    continue;
                }
                mbar_arrive_expect_tx(a_full(stage), p.a_box_bytes);
                if (HALO) {
                    int midx = 0, c = ai << 6;
                    if (ai >= cblk0) {
                        midx = 1;
                        c = (ai - cblk0) << 6;
                    }
                    tma_load_4d(dst, &maps.a[midx], a_full(stage), c, ow0 - 1, oh0 - 1, n0);
                } else {
                    const int tap = ai / cblk;
                    const int cb = ai - tap * cblk;
                    int midx = p.tap_map[tap], c = cb << 6;
                    if (cb >= cblk0) {
                        midx += 1;
                        c = (cb - cblk0) << 6;
                    }
                    tma_load_4d(dst, &maps.a[midx], a_full(stage), c, ow0 + p.tap_dw[tap], oh0 + p.tap_dh[tap], n0);
                }
                if (++stage == p.a_stages) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
        }
        if (PAIR) {
            // producer tail: the leader's multicast commits arrive on THIS CTA's empty barriers asynchronously; do
            // not leave (and let the shared memory be handed to another CTA) before the last of them has landed
            for (int k = 0; k < p.a_stages; ++k) {
                mbar_wait(a_empty(stage), phase ^ 1u, 18);
                if (++stage == p.a_stages) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ===== weight producer =====
        pdl_wait();
        const int row_off = (int)cta_rank * kBRows;   // PAIR: this CTA's half of a block's weight rows
        if (p.b_resident) {
            const uint32_t total_bytes = (uint32_t)p.n_tiles * p.num_kb * b_blk_bytes;
            if (cta_rank == 0) mbar_arrive_expect_tx(b_all_bar, (PAIR ? 2u : 1u) * total_bytes);
            for (int nt = 0; nt < p.n_tiles; ++nt)
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    const uint32_t dst = b_base + (nt * p.num_kb + kb) * b_blk_bytes;
                    if (PAIR) tma_load_2d_pair(dst, &maps.b, b_all_bar, kb * kKBlk, nt * BLOCK_N + row_off);
                    else tma_load_2d(dst, &maps.b, b_all_bar, kb * kKBlk, nt * BLOCK_N);
                }
        } else {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = work_id; tile < total_tiles; tile += work_stride) {
                const int n_tile = p.m_major ? tile % p.n_tiles : tile / m_units;
                for (int ai = 0; ai < a_loads; ++ai)
                    for (int ti = 0; ti < taps_per_a; ++ti) {
                        const int kb = HALO ? ti * cblk + ai : ai;
                        mbar_wait(b_empty(stage), phase ^ 1u, 12);
                        if (PAIR) {
                            if (cta_rank == 0) mbar_arrive_expect_tx(b_full(stage), 2 * b_blk_bytes);
                            tma_load_2d_pair(b_base + stage * b_blk_bytes, &maps.b, b_full(stage), kb * kKBlk,
                                             n_tile * BLOCK_N + row_off);
                            if (++stage == p.b_stages) {
                                stage = 0;
                                phase ^= 1u;
                            }
                            continue;
                        }
                        mbar_arrive_expect_tx(b_full(stage), b_blk_bytes);
                        tma_load_2d(b_base + stage * b_blk_bytes, &maps.b, b_full(stage), kb * kKBlk, n_tile * BLOCK_N);
                        if (++stage == p.b_stages) {
                            stage = 0;
                            phase ^= 1u;
                        }
                    }
            }
            if (PAIR) {   // producer tail (see the activation producer)
                for (int k = 0; k < p.b_stages; ++k) {
                    mbar_wait(b_empty(stage), phase ^ 1u, 19);
                    if (++stage == p.b_stages) {
                        stage = 0;
                        phase ^= 1u;
                    }
                }
            }
        }
    } else if (warp == 2) {
        // ===== MMA issuer: ONE elected thread runs the whole loop =====
        // A 128x64x16 MMA occupies the tensor pipe for 32 clocks, so the issuing thread's own instruction stream is
        // on the critical path (round 2: the previous loop -- all 32 lanes walking it, a predicate per MMA, the
        // resident / streamed and bisection branches re-evaluated per tap -- spent ~50 instructions per tap and
        // held every MMA to >= 90 clocks).  Here the resident and streamed variants are separate instantiations
        // of one generic lambda, descriptors are a constant upper word OR a 14-bit start-address field advanced by
        // adds (+2 per 16-element K step = 32 B, +8 per 128-byte row for the halo tap views), and only the first
        // MMA of a tile carries a run-time accumulate flag.
        if (cta_rank == 0 && elect_one()) {
            constexpr uint32_t idesc = make_idesc_f16(PAIR ? 2 * kTileM : kTileM, BLOCK_N, 0, 0);
            const uint64_t desc_hi = make_smem_desc_sw128(0, 0, 1024);   // start-address field = 0
            uint32_t tap_rows8[9];  // HALO: ((1+dh)*pw + (1+dw)) * 8 = row offset of the tap view in 16-byte units
#pragma unroll
            for (int ti = 0; ti < 9; ++ti)
                tap_rows8[ti] = HALO ? ((1 + p.tap_dh[ti]) * pw + (1 + p.tap_dw[ti])) * 8 : 0;
            const uint32_t b_blk16 = b_blk_bytes >> 4;
            const uint32_t a_stage16 = p.a_stage_bytes >> 4;
            const uint32_t a_base16 = a_base >> 4, b_base16 = b_base >> 4;
            const uint32_t tap_b16 = cblk * b_blk16;        // HALO, resident: weight-block stride between taps
            const uint32_t tile_b16 = p.num_kb * b_blk16;   // resident: stride between n tiles
            const int n_a_stages = p.a_stages, n_b_stages = p.b_stages, n_tiles = p.n_tiles;
            const bool m_major = p.m_major != 0;
            auto mma4 = [&](uint32_t d_tmem, uint32_t a16, uint32_t b16, uint32_t first_accum) {
#pragma unroll
                for (int k = 0; k < kKBlk / 16; ++k) {
                    const uint64_t da = desc_hi | (uint64_t)(a16 + 2 * k), db = desc_hi | (uint64_t)(b16 + 2 * k);
                    if (PAIR) umma_f16_pair(d_tmem, da, db, idesc, k == 0 ? first_accum : 1u);
                    else umma_f16(d_tmem, da, db, idesc, k == 0 ? first_accum : 1u);
                }
            };
            auto commit = [&](uint32_t bar) {
                if (PAIR) umma_commit_pair(bar);
                else umma_commit(bar);
            };
            auto run = [&](auto resident_tag) {
                constexpr bool RES = decltype(resident_tag)::value;
                int a_stage = 0, b_stage = 0, acc = 0;
                uint32_t a_phase = 0, b_phase = 0, acc_phase = 0;
                if (RES) mbar_wait(b_all_bar, 0, 13);
                for (int tile = work_id; tile < total_tiles; tile += work_stride) {
                    const int n_tile = m_major ? tile % n_tiles : tile / m_units;
                    mbar_wait(t_empty(acc), acc_phase ^ 1u, 14);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
                    uint32_t b_kb16 = b_base16 + n_tile * tile_b16;   // resident: weight block (n_tile, kb = ai)
                    for (int ai = 0; ai < a_loads; ++ai, b_kb16 += b_blk16) {
                        mbar_wait(a_full(a_stage), a_phase, 15);
                        tc_fence_after();
                        const uint32_t sa16 = a_base16 + a_stage * a_stage16;
                        const uint32_t first = ai != 0;
                        if (RES) {
                            if (HALO) {
                                uint32_t b16 = b_kb16;
#pragma unroll
                                for (int ti = 0; ti < 9; ++ti, b16 += tap_b16)   // kb = ti * cblk + ai
                                    mma4(d_tmem, sa16 + tap_rows8[ti], b16, ti == 0 ? first : 1u);
                            } else {
                                mma4(d_tmem, sa16, b_kb16, first);
                            }
                        } else {
#pragma unroll
                            for (int ti = 0; ti < (HALO ? 9 : 1); ++ti) {
                                mbar_wait(b_full(b_stage), b_phase, 16);
                                tc_fence_after();
                                mma4(d_tmem, sa16 + tap_rows8[ti], b_base16 + b_stage * b_blk16, ti == 0 ? first : 1u);
                                commit(b_empty(b_stage));
                                if (++b_stage == n_b_stages) {
                                    b_stage = 0;
                                    b_phase ^= 1u;
                                }
                            }
                        }
                        commit(a_empty(a_stage));
                        if (++a_stage == n_a_stages) {
                            a_stage = 0;
                            a_phase ^= 1u;
                        }
                    }
                    commit(t_full(acc));
                    if (++acc == 2) {
                        acc = 0;
                        acc_phase ^= 1u;
                    }
                }
            };
            if (p.b_resident) run(std::true_type{});
            else run(std::false_type{});
        }
        __syncwarp();
    } else if (warp >= 3) {
        // ===== epilogue: two groups of four warps; group g takes the 64-column chunks with index % 2 == g =====
        // Staging: "warp-private" (p.epi_warp) when the 32 accumulator rows of a warp are one storable
        // box (a 32-pixel run of an image row, or -- HALO with 32-wide padded rows -- one tile row): the
        // warp stages, fences and TMA-stores its own 4 KB slab with no block-level barrier.  Otherwise the
        // four warps of a group fill the group's 16 KB buffer and one thread stores the tile box.
        const int q = warp & 3;                 // TMEM lane quadrant this warp may read
        const int group = (warp - 3) >> 2;      // 0 or 1
        const int r = q * 32 + lane;            // accumulator row
        const bool grp_issuer = (lane == 0) && (warp == 3 || warp == 7);
        const bool warp_mode = p.epi_warp != 0;
        const uint32_t obuf = o_base + group * kOutStageBytes;
        const uint32_t my_row = obuf + r * kStageRowBytes;
        const uint32_t sw7 = (r & 7);
        float* gn_acc = reinterpret_cast<float*>(smem_gen + (gn_base - smem_base)) + 64 * group;  // per group
        int acc = 0;
        uint32_t acc_phase = 0;
        int cur_b = -1;
        auto gn_flush = [&](int b) {  // per group: no cross-group synchronisation
            epi_bar_sync(group);
            if (q == 3 && b >= 0) {   // warps 3 and 7: the first warp of each group
                for (int i = lane; i < 2 * p.gn_groups; i += 32) {
                    atomicAdd(p.gn_sums + (size_t)b * p.gn_groups * 2 + i, gn_acc[i]);
                    gn_acc[i] = 0.f;
                }
            }
            epi_bar_sync(group);
        };
        // 16 values x 32 rows -> 16 totals with a halving butterfly (16 shuffles): after the step for lane bit b a
        // lane keeps the half of its values selected by that bit; even lanes end up with total number
        // idx = bit-reversed (lane >> 1) in v[0] ([0..7] octet sums, [8..15] octet sums of squares).
        auto butterfly16 = [&](float (&v)[16]) -> int {
            {
                const bool up = lane & 16;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float recv = __shfl_xor_sync(0xffffffffu, up ? v[i] : v[i + 8], 16);
                    v[i] = (up ? v[i + 8] : v[i]) + recv;
                }
            }
            {
                const bool up = lane & 8;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float recv = __shfl_xor_sync(0xffffffffu, up ? v[i] : v[i + 4], 8);
                    v[i] = (up ? v[i + 4] : v[i]) + recv;
                }
            }
            {
                const bool up = lane & 4;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const float recv = __shfl_xor_sync(0xffffffffu, up ? v[i] : v[i + 2], 4);
                    v[i] = (up ? v[i + 2] : v[i]) + recv;
                }
            }
            {
                const bool up = lane & 2;
                const float recv = __shfl_xor_sync(0xffffffffu, up ? v[0] : v[1], 2);
                v[0] = (up ? v[1] : v[0]) + recv;
            }
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
            return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
        };
        // BLOCK_N <= 128: a thread meets ONE 64-column chunk per tile, always the same columns while the column
        // tile stays the same, so the 16 per-row partial sums are simply kept in registers across tiles and reduced
        // (butterfly + 16 global atomics per warp) only when the (sample, column tile) changes -- no shuffles, no
        // shared-memory atomics and no barrier per tile (round 2: they cost 8 us of a 34 us L0 convolution).
        constexpr bool kRunningStats = GN && BLOCK_N <= 128;
        float racc[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) racc[i] = 0.f;
        int run_key = -1;   // b * n_tiles + n_tile
        auto run_flush = [&]() {
            if (run_key < 0) return;
            const int b = run_key / p.n_tiles, nt = run_key - b * p.n_tiles;
            const int col = nt * BLOCK_N + (BLOCK_N == 64 ? 0 : group * 64);
            const int idx = butterfly16(racc);
            if ((lane & 1) == 0) {
                const int g = (col + 8 * (idx & 7)) / p.gn_cpg;
                atomicAdd(p.gn_sums + ((size_t)b * p.gn_groups + g) * 2 + (idx >> 3), racc[0]);
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) racc[i] = 0.f;
        };
        // per-tile constants of the row -> pixel map
        const int rw = r % pw;
        const int rh = (r / pw) % p.bh;
        const int rn = r / (pw * p.bh);
        // warp-private store box origin (relative to the tile)
        const int r0 = q * 32;
        const int st_w = HALO ? 0 : r0 % p.bw, st_h = HALO ? q : (r0 / p.bw) % p.bh, st_n = HALO ? 0 : r0 / (p.bw * p.bh);
        const bool st_ok = HALO ? (q < p.bh) : (st_n < p.bn);
        int tile_it = 0;
        for (int tile = work_id; tile < total_tiles; tile += work_stride, ++tile_it) {
            if (BLOCK_N == 64) {
                // one 64-column chunk per tile: the groups alternate over tiles instead (stage == group),
                // so each has two tile periods for its TMEM read-out, statistics and store
                if ((tile_it & 1) != group) continue;
                acc = group;
                acc_phase = (tile_it >> 1) & 1;  // k-th use of this stage
            }
            int n_tile, n0, oh0, ow0;
            tile_coords(tile, n_tile, n0, oh0, ow0);
            if (PAIR && n0 >= p.n) {
                // ghost tile of an odd row-tile count: nothing to store, but the accumulator hand-over still runs
                mbar_wait(t_full(acc), acc_phase, 17);
                tc_fence_after();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(t_empty(acc));
                if (BLOCK_N != 64 && ++acc == 2) {
                    acc = 0;
                    acc_phase ^= 1u;
                }
                continue;
            }
            const int n = n0 + rn, oh = oh0 + rh, ow = ow0 + rw;
            const bool valid = (rw < p.bw) && (rn < p.bn) && (n < p.n) && (oh < p.oh) && (ow < p.ow);
            const long long pix = (static_cast<long long>(n) * p.out_h + (oh * p.o_sh + p.o_h0)) * p.out_w +
                                  (ow * p.o_sw + p.o_w0);
            if (GN) {
                const int b = n0 / p.gn_frames;  // the tile lies within one sample (host guarantees)
                if (kRunningStats) {
                    const int key = b * p.n_tiles + n_tile;
                    if (key != run_key) {
                        run_flush();
                        run_key = key;
                    }
                } else if (b != cur_b) {
                    if (cur_b >= 0) gn_flush(cur_b);
                    cur_b = b;
                }
            }
            mbar_wait(t_full(acc), acc_phase, 17);
            tc_fence_after();
            const uint32_t taddr = tmem_base + acc * BLOCK_N + (static_cast<uint32_t>(q * 32) << 16);
            const int last_cc = BLOCK_N == 64 ? 0 : group * 64 + (BLOCK_N > 128 ? 128 : 0);   // this group's last chunk
            bool released = false;
#pragma unroll 1
            for (int cc = (BLOCK_N == 64 ? 0 : group * 64); cc < BLOCK_N; cc += 128) {
                uint32_t v[64];
                tmem_ld_32x64(taddr + cc, v);
                // the store that last read this group's staging buffer must have drained
                if (warp_mode) {
                    if (lane == 0) tma_store_wait_read<0>();
                    __syncwarp();
                } else {
                    if (grp_issuer) tma_store_wait_read<0>();
                    epi_bar_sync(group);
                }
                const int col = n_tile * BLOCK_N + cc;
                const float4* bp = reinterpret_cast<const float4*>(p.bias + col);
                const bool has_res = p.residual != nullptr;
                const uint4* rp = reinterpret_cast<const uint4*>(
                    reinterpret_cast<const h16*>(p.residual) + (valid ? pix : 0) * p.ldr + col);
                tmem_ld_wait();
                if (cc == last_cc) {
                    // the accumulator stage is in registers now: hand it back BEFORE the arithmetic, staging and
                    // store of this chunk, so the MMAs of the tile after next never wait for the epilogue's tail
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (PAIR) mbar_arrive_leader(t_empty(acc));   // the leader's MMA warp waits for both epilogues
                        else mbar_arrive(t_empty(acc));
                    }
                    released = true;
                }
                float sv[16];  // GN: [0..7] per 8-column octet sums of this row, [8..15] sums of squares
                uint4 xrow[LNF ? 8 : 1];   // LNF: the row of x (= the residual) whose LayerNorm is folded in
                float ln_mean = 0.f, ln_rstd = 0.f;
                if (LNF) {
                    float s1 = 0.f, s2 = 0.f;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        xrow[j] = valid ? __ldg(rp + j) : make_uint4(0u, 0u, 0u, 0u);
                        const float2 a = unpack_h2(xrow[j].x), b = unpack_h2(xrow[j].y), c2 = unpack_h2(xrow[j].z),
                                     d = unpack_h2(xrow[j].w);
                        s1 += ((a.x + a.y) + (b.x + b.y)) + ((c2.x + c2.y) + (d.x + d.y));
                        s2 = fmaf(a.x, a.x, fmaf(a.y, a.y, fmaf(b.x, b.x, fmaf(b.y, b.y, fmaf(c2.x, c2.x,
                             fmaf(c2.y, c2.y, fmaf(d.x, d.x, fmaf(d.y, d.y, s2))))))));
                    }
                    ln_mean = s1 * (1.f / 64.f);
                    ln_rstd = rsqrtf(fmaxf(s2 * (1.f / 64.f) - ln_mean * ln_mean, 0.f) + p.ln_eps);
                }
                const float4* cp = reinterpret_cast<const float4*>(p.ln_colsum + (LNF ? col : 0));
#pragma unroll
                for (int j = 0; j < 8; ++j) {  // 8 columns = one 16-byte unit
                    float f[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[8 * j + i]);
                    if (LNF) {
                        const float4 c0 = __ldg(cp + 2 * j), c1 = __ldg(cp + 2 * j + 1);
                        const float cs[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
                        for (int i = 0; i < 8; ++i) f[i] = ln_rstd * fmaf(-ln_mean, cs[i], f[i]);
                    }
                    if (p.bias) {
                        const float4 b0 = __ldg(bp + 2 * j), b1 = __ldg(bp + 2 * j + 1);
                        f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
                        f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
                    }
                    if (has_res && valid) {
                        const uint4 rr = LNF ? xrow[j] : __ldg(rp + j);
                        const float2 a = unpack_h2(rr.x), b = unpack_h2(rr.y),
                                     c2 = unpack_h2(rr.z), d = unpack_h2(rr.w);
                        f[0] += a.x; f[1] += a.y; f[2] += b.x; f[3] += b.y;
                        f[4] += c2.x; f[5] += c2.y; f[6] += d.x; f[7] += d.y;
                    }
                    uint4 u;
                    u.x = pack_h2(f[0], f[1]);
                    u.y = pack_h2(f[2], f[3]);
                    u.z = pack_h2(f[4], f[5]);
                    u.w = pack_h2(f[6], f[7]);
                    const uint32_t addr = my_row + ((j ^ sw7) << 4);
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(u.x), "r"(u.y), "r"(u.z),
                                 "r"(u.w)
                                 : "memory");
                    if (GN) {
                        // statistics of what the consumer will read: the fp16-rounded values
                        const float2 a = unpack_h2(u.x), b = unpack_h2(u.y), c2 = unpack_h2(u.z),
                                     d = unpack_h2(u.w);
                        const float s = ((a.x + a.y) + (b.x + b.y)) + ((c2.x + c2.y) + (d.x + d.y));
                        const float qq = fmaf(a.x, a.x, fmaf(a.y, a.y, fmaf(b.x, b.x, fmaf(b.y, b.y, fmaf(c2.x, c2.x,
                                         fmaf(c2.y, c2.y, fmaf(d.x, d.x, d.y * d.y)))))));
                        if (kRunningStats) {
                            racc[j] += valid ? s : 0.f;
                            racc[8 + j] += valid ? qq : 0.f;
                        } else {
                            sv[j] = valid ? s : 0.f;
                            sv[8 + j] = valid ? qq : 0.f;
                        }
                    }
                }
                if (GN && !kRunningStats) {
                    const int idx = butterfly16(sv);
                    if ((lane & 1) == 0) {
                        const int g = (col + 8 * (idx & 7)) / p.gn_cpg;
                        atomicAdd(gn_acc + 2 * g + (idx >> 3), sv[0]);
                    }
                }
                fence_proxy_async();
                if (warp_mode) {
                    __syncwarp();
                    if (lane == 0) {
                        const uint32_t slab = obuf + q * 32 * kStageRowBytes;
                        if (st_ok && (!HALO || oh0 + st_h < p.oh))
                            tma_store_4d(&maps.out, slab, col, ow0 + st_w, oh0 + st_h, n0 + st_n);
                        tma_store_commit();
                    }
                } else {
                    epi_bar_sync(group);
                    if (grp_issuer) {
                        if (HALO) {
                            // one store per tile row: the bw useful pixels of each padded accumulator row
                            for (int h = 0; h < p.bh; ++h)
                                if (oh0 + h < p.oh)
                                    tma_store_4d(&maps.out, obuf + h * pw * kStageRowBytes, col, ow0, oh0 + h, n0);
                        } else {
                            tma_store_4d(&maps.out, obuf, col, ow0, oh0, n0);
                        }
                        tma_store_commit();
                    }
                }
            }
            if (!released) {   // not reached (every group's loop ends at last_cc); dropping it reschedules the
                               // kernel and moves its spills (profiles/r07_env_switch_removal.txt)
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (PAIR) mbar_arrive_leader(t_empty(acc));
                    else mbar_arrive(t_empty(acc));
                }
            }
            if (BLOCK_N != 64 && ++acc == 2) {
                acc = 0;
                acc_phase ^= 1u;
            }
        }
        if (kRunningStats) run_flush();
        else if (GN) gn_flush(cur_b);
        if (lane == 0) tma_store_wait_all();
    }

    tc_fence_before();
    if (PAIR) cluster_sync_all();   // neither CTA may free its half while the pair's MMAs / barriers are in use
    else __syncthreads();
    if (warp == 2) {
        if (PAIR) tmem_dealloc_pair(tmem_base, kTmemCols);
        else tmem_dealloc(tmem_base, kTmemCols);
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <int BLOCK_N, bool HALO, bool GN, bool PAIR, bool LNF = false>
static cudaError_t launch_igemm2(const Igemm2Maps& maps, const Igemm2Params& p, int grid, size_t smem,
                                 cudaStream_t stream) {
    static bool configured = false;  // benign race: attribute set is idempotent
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(igemm2_kernel<BLOCK_N, HALO, GN, PAIR, LNF>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kIgemm2MaxSmem);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    launch_pdl_cluster(igemm2_kernel<BLOCK_N, HALO, GN, PAIR, LNF>, grid, kIgemm2Threads, smem, stream, PAIR ? 2 : 1, maps,
                       p);
    return cudaGetLastError();
}

template <int BLOCK_N>
static cudaError_t launch_igemm2_n(const Igemm2Maps& maps, const Igemm2Params& p, bool halo, bool pair, int grid,
                                   size_t smem, cudaStream_t stream) {
    const bool gn = p.gn_sums != nullptr;
    if (halo && pair)
        return gn ? launch_igemm2<BLOCK_N, true, true, true>(maps, p, grid, smem, stream)
                  : launch_igemm2<BLOCK_N, true, false, true>(maps, p, grid, smem, stream);
    if (halo) return gn ? launch_igemm2<BLOCK_N, true, true, false>(maps, p, grid, smem, stream)
                        : launch_igemm2<BLOCK_N, true, false, false>(maps, p, grid, smem, stream);
    return gn ? launch_igemm2<BLOCK_N, false, true, false>(maps, p, grid, smem, stream)
              : launch_igemm2<BLOCK_N, false, false, false>(maps, p, grid, smem, stream);
}

cudaError_t igemm2_launch(const Igemm2Maps& maps, const Igemm2Params& p, int block_n, bool halo, bool pair, int grid,
                          size_t smem, cudaStream_t stream) {
    if (p.ln_colsum != nullptr) {
        if (block_n != 64 || halo || pair || p.gn_sums != nullptr) return cudaErrorInvalidValue;
        return launch_igemm2<64, false, false, false, true>(maps, p, grid, smem, stream);
    }
    switch (block_n) {
        case 64: return launch_igemm2_n<64>(maps, p, halo, pair, grid, smem, stream);
        case 128: return launch_igemm2_n<128>(maps, p, halo, pair, grid, smem, stream);
        case 256: return launch_igemm2_n<256>(maps, p, halo, pair, grid, smem, stream);
    }
    return cudaErrorInvalidValue;
}

}  // namespace cesm
