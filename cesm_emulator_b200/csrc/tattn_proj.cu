// Temporal attention for short windows (F <= 3) FUSED WITH ITS q/k/v PROJECTION, for 64 input channels (the three
// full-resolution blocks and the level-1 up block of config/baseline), forward only -- calls without gradients:
//
//     o = attention(LN(x) Wq^T, LN(x) Wk^T, LN(x) Wv^T)            video_net.py:403-453, rotary_embedding.py:29-48
//
// Unfused, the projection writes a 768-wide q|k|v tensor (510 MB per block at 192x288, B = 2) and the attention core
// reads it back.  Here q, k and v never reach HBM: a warp owns 16 pixel columns (all F frames): LN(x) rows -> mma.sync
// A fragments (registers, loaded once); per head, q|k (then v) = A * W_h^T with W resident in shared memory; RoPE,
// scores, softmax and P.V run on the accumulator fragments (a pixel row's 32 head features live in one quad: dot
// products are quad shuffles); o leaves through a warp-private staging tile as 64-byte row segments.
//
// Roofline: tensor / issue.
#include "api_common.h"
#include "common.cuh"

namespace cesm {
namespace tp {

static constexpr int D = 32, C = 64, HEADS = 8, HID = HEADS * D;
static constexpr int WP = C + 8;          // pitch (halfs) of W rows and of staged LN(x) rows: 144 B, conflict-free ldmatrix
static constexpr int OP = D + 8;          // pitch of staged [16][32] head tiles: 80 B
static constexpr int WARPS = 8;

__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr));
}
__device__ __forceinline__ void mma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
        "{%0, %1, %2, %3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ float quad_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v + __shfl_xor_sync(0xffffffffu, v, 2);
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// acc[f][nt] (16 pixels x 8 output channels, F frames) for NTILES consecutive 8-row blocks of W starting at `wrow`
// (shared memory, pitch WP): every B fragment is loaded once and used for all F frames.
template <int F, int NTILES>
__device__ __forceinline__ void project(float (&acc)[F][NTILES][4], const uint32_t (&a)[F][4][4], uint32_t wbase, int lane) {
#pragma unroll
    for (int nt = 0; nt < NTILES; ++nt) {
        uint32_t b0[4], b1[4];
        const uint32_t addr = wbase + (uint32_t)((nt * 8 + (lane & 7)) * WP + (lane >> 3) * 8) * 2u;
        ldsm4(b0, addr);        // k steps 0, 1
        ldsm4(b1, addr + 64u);  // k steps 2, 3
#pragma unroll
        for (int f = 0; f < F; ++f) {
            acc[f][nt][0] = acc[f][nt][1] = acc[f][nt][2] = acc[f][nt][3] = 0.f;
            mma(acc[f][nt], a[f][0], b0[0], b0[1]);
            mma(acc[f][nt], a[f][1], b0[2], b0[3]);
            mma(acc[f][nt], a[f][2], b1[0], b1[1]);
            mma(acc[f][nt], a[f][3], b1[2], b1[3]);
        }
    }
}

// stage the F x 16 LN(x) rows of one pixel group (warp-private, pitch WP) and load them as A fragments
template <int F>
__device__ __forceinline__ void load_group(uint32_t (&a)[F][4][4], uint32_t xs, const h16* __restrict__ xn, long long b, long long p0,
                                           int HW, int lane) {
#pragma unroll
    for (int i = 0; i < F * 4; ++i) {   // F*16 rows x 8 chunks of 16 bytes = F*128 chunks, 32 per trip
        const int c = lane + 32 * i, row = c >> 3, ch = c & 7;
        const int f = row >> 4, px = row & 15;
        cp16(xs + (uint32_t)(row * WP + ch * 8) * 2u, xn + ((b * F + f) * HW + p0 + px) * C + ch * 8);
    }
    cp_commit();
    cp_wait_all();
    __syncwarp();
#pragma unroll
    for (int f = 0; f < F; ++f)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
            ldsm4(a[f][ks], xs + (uint32_t)((f * 16 + (lane & 15)) * WP + ks * 16 + (lane >> 4) * 8) * 2u);
    __syncwarp();
}

// RoPE on accumulator fragments: columns (2t, 2t+1) of n-tile nt are the pair m = nt*4 + t
template <int F>
__device__ __forceinline__ void rotate(float (&x)[F][4][4], const float (&cf)[F][4], const float (&sf)[F][4], float scale) {
#pragma unroll
    for (int f = 0; f < F; ++f)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const float x0 = x[f][nt][2 * r] * scale, x1 = x[f][nt][2 * r + 1] * scale;
                x[f][nt][2 * r] = x0 * cf[f][nt] - x1 * sf[f][nt];
                x[f][nt][2 * r + 1] = x1 * cf[f][nt] + x0 * sf[f][nt];
            }
}

// p[r][i][j]: softmax over j of q_i . k_j + bias[i][j] for the two pixel rows (g, g + 8) of this lane's quad
template <int F>
__device__ __forceinline__ void scores_softmax(float (&p)[2][F][F], const float (&q)[F][4][4], const float (&k)[F][4][4],
                                               const float* __restrict__ bs /* [F][F] of this head */) {
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int i = 0; i < F; ++i) {
            float m = -INFINITY;
#pragma unroll
            for (int j = 0; j < F; ++j) {
                float s = 0.f;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt)
                    s = fmaf(q[i][nt][2 * r], k[j][nt][2 * r], fmaf(q[i][nt][2 * r + 1], k[j][nt][2 * r + 1], s));
                s = quad_sum(s) + bs[i * F + j];
                p[r][i][j] = s;
                m = fmaxf(m, s);
            }
            float l = 0.f;
#pragma unroll
            for (int j = 0; j < F; ++j) {
                p[r][i][j] = __expf(p[r][i][j] - m);
                l += p[r][i][j];
            }
            const float inv = 1.f / l;
#pragma unroll
            for (int j = 0; j < F; ++j) p[r][i][j] *= inv;
        }
}

// write a [F][16][32] fragment set (fp32 accumulators) into a warp-private staging tile (pitch OP) as fp16
template <int F>
__device__ __forceinline__ void stage_frag(const float (&x)[F][4][4], uint32_t base, int lane) {
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int f = 0; f < F; ++f)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            const uint32_t a = base + (uint32_t)((f * 16 + g) * OP + nt * 8 + 2 * t) * 2u;
            sts32(a, pack_h2(x[f][nt][0], x[f][nt][1]));
            sts32(a + (uint32_t)(8 * OP) * 2u, pack_h2(x[f][nt][2], x[f][nt][3]));
        }
}

// copy a staged [F][16][32] tile to global rows: 64 contiguous bytes per (frame, pixel) at `dst` + row * ld
template <int F>
__device__ __forceinline__ void flush_tile(uint32_t base, h16* __restrict__ dst, long long b, long long p0, int HW, int ld, int lane) {
#pragma unroll
    for (int i = 0; i < (F * 64 + 31) / 32; ++i) {
        const int c = lane + 32 * i;
        if (c < F * 64) {
            const int row = c >> 2, ch = c & 3, f = row >> 4, px = row & 15;
            uint4 v;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                         : "r"(base + (uint32_t)(row * OP + ch * 8) * 2u));
            *reinterpret_cast<uint4*>(dst + ((b * F + f) * HW + p0 + px) * ld + ch * 8) = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// forward: W (all 768 rows) resident in shared memory
// ------------------------------------------------------------------------------------------------
template <int F>
__global__ void __launch_bounds__(32 * WARPS, 1)
tattn_proj_fwd_kernel(const h16* __restrict__ xn, const h16* __restrict__ wqkv /* [768][64] */, const float* __restrict__ bias,
                      const float* __restrict__ cs, const float* __restrict__ sn, h16* __restrict__ out, long long groups, int HW,
                      float scale) {
    pdl_trigger();
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t ws = smem_u32(smem);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, t = lane & 3;
    const uint32_t xs = ws + (uint32_t)(3 * HID * WP) * 2u + (uint32_t)w * (F * 16 * WP) * 2u;   // also the o staging tile
    float* sb = reinterpret_cast<float*>(smem + (size_t)3 * HID * WP * 2 + (size_t)WARPS * F * 16 * WP * 2);  // bias [H][F][F]
    // the packed weights were written at the top of the step: fetch them while the preceding kernel drains
    for (int c = threadIdx.x; c < 3 * HID * 8; c += blockDim.x) cp16(ws + (uint32_t)((c >> 3) * WP + (c & 7) * 8) * 2u, wqkv + c * 8);
    cp_commit();
    pdl_wait();
    for (int i = threadIdx.x; i < HEADS * F * F; i += blockDim.x) sb[i] = bias[i];
    float cf[F][4], sf[F][4];
#pragma unroll
    for (int f = 0; f < F; ++f)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            cf[f][nt] = __ldg(cs + f * 16 + nt * 4 + t);
            sf[f][nt] = __ldg(sn + f * 16 + nt * 4 + t);
        }
    cp_wait_all();
    __syncthreads();
    const int gpp = HW / 16;  // groups per image
    for (long long grp = (long long)blockIdx.x * WARPS + w; grp < groups; grp += (long long)gridDim.x * WARPS) {
        const long long b = grp / gpp, p0 = (grp - b * gpp) * 16;
        uint32_t a[F][4][4];
        load_group<F>(a, xs, xn, b, p0, HW, lane);
#pragma unroll 1
        for (int h = 0; h < HEADS; ++h) {
            float p[2][F][F];
            {
                float q[F][4][4], k[F][4][4];
                project<F, 4>(q, a, ws + (uint32_t)((h * D) * WP) * 2u, lane);
                project<F, 4>(k, a, ws + (uint32_t)((HID + h * D) * WP) * 2u, lane);
                rotate<F>(q, cf, sf, scale);
                rotate<F>(k, cf, sf, 1.f);
                scores_softmax<F>(p, q, k, sb + h * F * F);
            }
            float v[F][4][4], o[F][4][4];
            project<F, 4>(v, a, ws + (uint32_t)((2 * HID + h * D) * WP) * 2u, lane);
#pragma unroll
            for (int i = 0; i < F; ++i)
#pragma unroll
                for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float acc = 0.f;
#pragma unroll
                        for (int j = 0; j < F; ++j) acc = fmaf(p[e >> 1][i][j], v[j][nt][e], acc);
                        o[i][nt][e] = acc;
                    }
            __syncwarp();  // the previous head's staged rows have been copied out
            stage_frag<F>(o, xs, lane);
            __syncwarp();
            flush_tile<F>(xs, out + h * D, b, p0, HW, HID, lane);
        }
        __syncwarp();
    }
}

template <int F>
static constexpr size_t fwd_smem() {
    return (size_t)3 * HID * WP * 2 + (size_t)WARPS * F * 16 * WP * 2 + (size_t)HEADS * F * F * 4;
}

}  // namespace tp
}  // namespace cesm

using namespace cesm;

static int tp_check(int B, int F, int HW, int H, int dim_head, int cin) {
    CESM_REQUIRE(dim_head == tp::D && H == tp::HEADS && cin == tp::C,
                 "fused projection + temporal attention needs 8 heads of 32 and 64 input channels (H=%d D=%d C=%d)", H, dim_head, cin);
    CESM_REQUIRE(F >= 1 && F <= 3, "fused projection + temporal attention supports 1..3 frames (F=%d)", F);
    CESM_REQUIRE(HW % 16 == 0 && B > 0, "fused projection + temporal attention needs H*W divisible by 16 (HW=%d)", HW);
    return CESM_OK;
}

extern "C" int cesm_tattn_proj_fwd(const void* xn, const void* wqkv, const float* bias, const float* cs, const float* sn, void* out,
                                   int B, int F, int HW, int H, int dim_head, int cin, float scale, void* stream) {
    if (int rc = tp_check(B, F, HW, H, dim_head, cin)) return rc;
    const long long groups = (long long)B * HW / 16;
    int sms = 148, dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long want = (groups + tp::WARPS - 1) / tp::WARPS;
    const int grid = (int)(want < sms ? want : sms);
    cudaStream_t st = as_stream(stream);
#define TP_FWD(FF)                                                                                                         \
    {                                                                                                                      \
        static bool cfg = false;                                                                                           \
        if (!cfg) {                                                                                                        \
            CESM_CHECK_CUDA(cudaFuncSetAttribute(tp::tattn_proj_fwd_kernel<FF>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                                 (int)tp::fwd_smem<FF>()));                                                \
            cfg = true;                                                                                                    \
        }                                                                                                                  \
        launch_pdl(tp::tattn_proj_fwd_kernel<FF>, grid, 32 * tp::WARPS, tp::fwd_smem<FF>(), st, (const h16*)xn, (const h16*)wqkv, \
                   bias, cs, sn, (h16*)out, groups, HW, scale);                                                            \
    }
    switch (F) {
        case 1: TP_FWD(1) break;
        case 2: TP_FWD(2) break;
        default: TP_FWD(3) break;
    }
#undef TP_FWD
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}
