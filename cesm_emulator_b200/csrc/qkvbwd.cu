// Backward of the q/k/v projection (to_qkv: 1x1 conv / Linear C -> cout, no bias; video_net.py:322, :380)
// for C = 64: the data gradient and the weight gradient in ONE pass over dqkv.
//
//     dX[p][ci]  = sum_co dY[p][co] * W[co][ci]           (contraction over the cout = 768 output channels)
//     dW[co][ci] += sum_p  dY[p][co] * X[p][ci]            (contraction over pixels)
//
// dY (fp16 [rows][cout], 1.5 KB per row at cout = 768) is by far the largest operand of both; as two
// kernels it was streamed from HBM twice (84 + 87 us at 192x288, each at its own bandwidth roofline).
// Here a persistent CTA walks 128-pixel row tiles; a tile's dY arrives in 128-channel chunks
// ([128 px][128 co], two SWIZZLE_128B sub-tiles of 64 channels) and every chunk feeds two tcgen05 MMA
// streams from the same shared-memory bytes:
//     data gradient  : the chunk as a K-major A operand (M = pixels, K = co) x W^T chunk (K-major B),
//                      accumulating D1[128 px][64 ci] over the six chunks of the tile;
//     weight gradient: the chunk as an MN-major A operand (M = co, K = pixels) x the X tile (MN-major B),
//                      accumulating D2[chunk][128 co][64 ci] over ALL tiles of the CTA.
// TMEM: D1 double-buffered (2 x 64 columns) + D2 (6 x 64 columns) = 512 columns exactly.
// Warps: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocation, 4..7 = epilogue (D1 -> fp16 dX rows per
// tile; D2 -> red.add into dW once at the end).
#include "api_common.h"
#include "common.cuh"

namespace cesm {

static constexpr int QB_C = 64;                  // input channels (ci)
static constexpr int QB_TILE = 128;              // pixels per row tile
static constexpr int QB_CHUNK = 128;             // output channels (co) per chunk
static constexpr int QB_STAGES = 3;
static constexpr int QB_SUB = QB_TILE * 128;     // one [128 px][64 ch] SWIZZLE_128B sub-tile: 16 KB
static constexpr int QB_WSUB = QB_C * 128;       // one [64 ci][64 co] weight sub-tile: 8 KB
static constexpr int QB_STAGE = 2 * QB_SUB + 2 * QB_WSUB;   // 48 KB
static constexpr int QB_XSTAGES = 2;
static constexpr int QB_SMEM = 1024 + QB_STAGES * QB_STAGE + QB_XSTAGES * QB_SUB + 1024;
static constexpr int QB_THREADS = 256;

struct QkvBwdMaps {
    CUtensorMap dy;   // [rows][cout], box {64 co, 128 px}
    CUtensorMap x;    // [rows][64],   box {64 ci, 128 px}
    CUtensorMap w;    // [64 ci][cout] (W^T, K-major for the data gradient), box {64 co, 64 ci}
};
struct QkvBwdParams {
    long long rows;
    int tiles, chunks;          // row tiles; cout / 128
    h16* dx;          // [rows][64]
    float* dw;                  // dW[co * so + ci] (+=)
    long long so;
};

__global__ void __launch_bounds__(QB_THREADS, 1)
qkv_bwd_kernel(const __grid_constant__ QkvBwdMaps maps, const QkvBwdParams p) {
    pdl_trigger();  // pdl_wait() sits in the TMA producer: MMA and epilogue depend on its data
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t x_base = smem_base + QB_STAGES * QB_STAGE;
    const uint32_t bar_base = x_base + QB_XSTAGES * QB_SUB;
    auto s_full = [&](int s) { return bar_base + 8u * s; };
    auto s_empty = [&](int s) { return bar_base + 8u * (QB_STAGES + s); };
    auto x_full = [&](int s) { return bar_base + 8u * (2 * QB_STAGES + s); };
    auto x_empty = [&](int s) { return bar_base + 8u * (2 * QB_STAGES + 2 + s); };
    auto d1_full = [&](int s) { return bar_base + 8u * (2 * QB_STAGES + 4 + s); };
    auto d1_empty = [&](int s) { return bar_base + 8u * (2 * QB_STAGES + 6 + s); };
    const uint32_t d2_full = bar_base + 8u * (2 * QB_STAGES + 8);
    const uint32_t tmem_ptr_addr = bar_base + 8u * (2 * QB_STAGES + 9);
    volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_ptr_addr - smem_base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&maps.dy);
        tma_prefetch_desc(&maps.x);
        tma_prefetch_desc(&maps.w);
        for (int s = 0; s < QB_STAGES; ++s) {
            mbar_init(s_full(s), 1);
            mbar_init(s_empty(s), 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(x_full(s), 1);
            mbar_init(x_empty(s), 1);
            mbar_init(d1_full(s), 1);
            mbar_init(d1_empty(s), 4);
        }
        mbar_init(d2_full, 1);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(tmem_ptr_addr, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_gen;
    const uint32_t tmem_d1 = tmem_base;            // 2 x 64 columns
    const uint32_t tmem_d2 = tmem_base + 128;      // chunks x 64 columns

    if (warp == 0 && lane == 0) {
        // ===== TMA producer =====
        pdl_wait();
        int st = 0, xs = 0;
        uint32_t ph = 0, xph = 0;
        for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
            const int row0 = tile * QB_TILE;
            mbar_wait(x_empty(xs), xph ^ 1u, 31);
            mbar_arrive_expect_tx(x_full(xs), QB_SUB);
            tma_load_2d(x_base + xs * QB_SUB, &maps.x, x_full(xs), 0, row0);
            if (++xs == QB_XSTAGES) {
                xs = 0;
                xph ^= 1u;
            }
            for (int c = 0; c < p.chunks; ++c) {
                mbar_wait(s_empty(st), ph ^ 1u, 32);
                const uint32_t sb = smem_base + st * QB_STAGE;
                mbar_arrive_expect_tx(s_full(st), QB_STAGE);
                tma_load_2d(sb, &maps.dy, s_full(st), c * QB_CHUNK, row0);
                tma_load_2d(sb + QB_SUB, &maps.dy, s_full(st), c * QB_CHUNK + 64, row0);
                tma_load_2d(sb + 2 * QB_SUB, &maps.w, s_full(st), c * QB_CHUNK, 0);
                tma_load_2d(sb + 2 * QB_SUB + QB_WSUB, &maps.w, s_full(st), c * QB_CHUNK + 64, 0);
                if (++st == QB_STAGES) {
                    st = 0;
                    ph ^= 1u;
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one elected thread runs the loops =====
        constexpr uint32_t idesc_dg = make_idesc_f16(QB_TILE, QB_C, 0, 0);    // K-major A, B
        constexpr uint32_t idesc_wg = make_idesc_f16(QB_CHUNK, QB_C, 1, 1);   // MN-major A, B
        if (elect_one()) {
            const uint64_t dk = make_smem_desc_sw128(0, 0, 1024);              // K-major SW128
            const uint64_t dmn = make_smem_desc_sw128(0, QB_SUB, 1024);        // MN-major: 64-channel atoms QB_SUB apart
            const int chunks = p.chunks;
            int st = 0, xs = 0, acc = 0, it = 0;
            uint32_t ph = 0, xph = 0, accph = 0;
            for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++it) {
                mbar_wait(d1_empty(acc), accph ^ 1u, 33);
                mbar_wait(x_full(xs), xph, 34);
                tc_fence_after();
                const uint32_t x16 = (x_base + xs * QB_SUB) >> 4;
                const uint32_t d1 = tmem_d1 + acc * 64;
                for (int c = 0; c < chunks; ++c) {
                    mbar_wait(s_full(st), ph, 35);
                    tc_fence_after();
                    const uint32_t a16 = (smem_base + st * QB_STAGE) >> 4;
                    const uint32_t w16 = a16 + ((2 * QB_SUB) >> 4);
                    // data gradient: K = 128 co = 8 steps of 16 (32 B inside a 128-byte row; second sub-tile after 4)
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const uint32_t ao = a16 + (k >> 2) * (QB_SUB >> 4) + (k & 3) * 2;
                        const uint32_t bo = w16 + (k >> 2) * (QB_WSUB >> 4) + (k & 3) * 2;
                        umma_f16(d1, dk | (uint64_t)ao, dk | (uint64_t)bo, idesc_dg, k == 0 ? (uint32_t)(c != 0) : 1u);
                    }
                    // weight gradient: K = 128 pixels = 8 steps of 16 pixels (2048 B)
                    const uint32_t d2 = tmem_d2 + c * 64;
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        umma_f16(d2, dmn | (uint64_t)(a16 + k * 128), dmn | (uint64_t)(x16 + k * 128), idesc_wg,
                                 k == 0 ? (uint32_t)(it != 0) : 1u);
                    umma_commit(s_empty(st));
                    if (++st == QB_STAGES) {
                        st = 0;
                        ph ^= 1u;
                    }
                }
                umma_commit(x_empty(xs));
                umma_commit(d1_full(acc));
                if (++xs == QB_XSTAGES) {
                    xs = 0;
                    xph ^= 1u;
                }
                if (++acc == 2) {
                    acc = 0;
                    accph ^= 1u;
                }
            }
            umma_commit(d2_full);
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===== epilogue =====
        const int q = warp & 3;
        const uint32_t lane_base = static_cast<uint32_t>(q * 32) << 16;
        int acc = 0;
        uint32_t accph = 0;
        for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
            mbar_wait(d1_full(acc), accph, 36);
            tc_fence_after();
            const long long row = (long long)tile * QB_TILE + q * 32 + lane;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                uint32_t v[32];
                tmem_ld_32x32(tmem_d1 + acc * 64 + half * 32 + lane_base, v);
                tmem_ld_wait();
                if (row < p.rows) {
                    uint4* dst = reinterpret_cast<uint4*>(p.dx + row * QB_C + half * 32);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint4 u;
                        u.x = pack_h2(__uint_as_float(v[8 * j + 0]), __uint_as_float(v[8 * j + 1]));
                        u.y = pack_h2(__uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3]));
                        u.z = pack_h2(__uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
                        u.w = pack_h2(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7]));
                        dst[j] = u;
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(d1_empty(acc));
            if (++acc == 2) {
                acc = 0;
                accph ^= 1u;
            }
        }
        // weight gradient: TMEM lane = output channel of the chunk, columns = the 64 input channels.  The
        // parameter layout is [co][ci], so a lane-per-co red.add would scatter 32 requests per instruction;
        // each 32 x 32 block goes through a warp-private shared-memory tile (the operand ring is idle by now)
        // and is added with lanes along ci: one 128-byte request per instruction.
        if (blockIdx.x < p.tiles) {
            mbar_wait(d2_full, 0, 37);
            tc_fence_after();
            float* tr = reinterpret_cast<float*>(smem_gen) + q * (32 * 33);
            for (int c = 0; c < p.chunks; ++c) {
                float* base = p.dw + (long long)(c * QB_CHUNK + q * 32) * p.so;
#pragma unroll 1
                for (int half = 0; half < 2; ++half) {
                    uint32_t v[32];
                    tmem_ld_32x32(tmem_d2 + c * 64 + half * 32 + lane_base, v);
                    tmem_ld_wait();
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 32; ++i) tr[lane * 33 + i] = __uint_as_float(v[i]);
                    __syncwarp();
#pragma unroll 8
                    for (int co = 0; co < 32; ++co) atomicAdd(base + (long long)co * p.so + half * 32 + lane, tr[co * 33 + lane]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

}  // namespace cesm

using namespace cesm;

extern "C" int cesm_qkv_bwd(const void* dy, const void* x, const void* wt, void* dx, float* dw, long long dw_so,
                            long long rows, int cin, int cout, void* stream) {
    CESM_REQUIRE(cin == QB_C, "qkv_bwd is specialised for 64 input channels (cin=%d)", cin);
    CESM_REQUIRE(cout % QB_CHUNK == 0 && cout >= QB_CHUNK && cout <= 6 * QB_CHUNK,
                 "qkv_bwd needs cout in {128..768} and a multiple of 128 (cout=%d)", cout);
    CESM_REQUIRE(rows > 0 && dw_so >= cin, "bad rows / dw stride");
    QkvBwdMaps maps;
    {
        const uint64_t dims[2] = {(uint64_t)cout, (uint64_t)rows};
        const uint64_t str[1] = {(uint64_t)cout * 2};
        const uint32_t box[2] = {64u, (uint32_t)QB_TILE};
        int rc = get_tensor_map_h16(&maps.dy, dy, 2, dims, str, box);
        if (rc) return rc;
    }
    {
        const uint64_t dims[2] = {(uint64_t)cin, (uint64_t)rows};
        const uint64_t str[1] = {(uint64_t)cin * 2};
        const uint32_t box[2] = {64u, (uint32_t)QB_TILE};
        int rc = get_tensor_map_h16(&maps.x, x, 2, dims, str, box);
        if (rc) return rc;
    }
    {
        const uint64_t dims[2] = {(uint64_t)cout, (uint64_t)cin};
        const uint64_t str[1] = {(uint64_t)cout * 2};
        const uint32_t box[2] = {64u, (uint32_t)QB_C};
        int rc = get_tensor_map_h16(&maps.w, wt, 2, dims, str, box);
        if (rc) return rc;
    }
    QkvBwdParams p;
    p.rows = rows;
    p.tiles = (int)((rows + QB_TILE - 1) / QB_TILE);
    p.chunks = cout / QB_CHUNK;
    p.dx = (h16*)dx;
    p.dw = dw;
    p.so = dw_so;
    static bool cfg = false;
    if (!cfg) {
        CESM_CHECK_CUDA(cudaFuncSetAttribute(qkv_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, QB_SMEM));
        cfg = true;
    }
    int sms = 148, dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = p.tiles < sms ? p.tiles : sms;
    launch_pdl(qkv_bwd_kernel, grid, QB_THREADS, QB_SMEM, as_stream(stream), maps, p);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}
