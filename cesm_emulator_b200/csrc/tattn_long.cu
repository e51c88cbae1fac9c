// Temporal attention for LONG windows (F > 4 frames; BASELINE.json configs[4], video_net.py:413-453 +
// rotary_embedding.py:29-48 + the relative-position bias of video_net.py:302-310), flash style.
//
// Sequences are short (tens to a few hundred frames) but there are B*H*W*heads of them, and the frames of
// one pixel column are H*W rows apart in the channels-last q|k|v tensor.  The generic kernel (attn.cu) gave
// every (query, head) a thread that re-read all keys and values from global memory: F x the traffic.  Here a
// CTA stages ALL frames of one pixel column (for a group of heads) in shared memory once -- each row is one
// contiguous run of the q, k and v slices of those heads -- and one WARP per head does the whole
// (F x F) attention on the tensor cores with mma.sync.m16n8k16 (fp16 in, fp32 accumulate):
//
//   forward : RoPE(q * scale), RoPE(k) in place as fp16 hi + lo pairs (rotate_qk);  per 16-query tile
//             S = Q K^T (+ bias) from the pairs -> softmax in the
//             accumulator registers -> O = P V;  O overwrites the dead q rows and leaves with 16-byte stores.
//   backward: recomputes S from q, k and the saved log-sum-exp.  Pass B (per query tile): dP = dO V^T,
//             dS = P (dP - delta), dQ = dS K.  Pass A (per key tile, everything transposed so that no
//             accumulator outlives a tile): S^T = K Q^T, dP^T = V dO^T, dV = P^T dO, dK = dS^T Q, written over
//             the k / v rows they belong to.  RoPE is undone on dQ / dK in registers (pairs are adjacent columns
//             of an accumulator fragment).
//
// The position bias is Toeplitz (it depends on key - query only), so it travels as one (2F-1)-entry table per
// head and its gradient is accumulated per diagonal in shared memory: 2F-1 floats per head instead of F*F.
// Roofline: HBM (q|k|v read once: 1.5 KB per row forward; + dout, out, dq|dk|dv backward = 4 KB per row).
#include "api_common.h"
#include "common.cuh"

namespace cesm {
namespace tl {

static constexpr int D = 32;

__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr));
}
__device__ __forceinline__ void ldsm4_t(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
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
__device__ __forceinline__ void cp_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ float quad_max(float v) {
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
    return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v + __shfl_xor_sync(0xffffffffu, v, 2);
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

struct Geo {
    int F, Fp, HW, H, HG;      // frames, frames padded to 16, pixels per frame, heads, heads per CTA
    int pq;                    // row pitch of the staged q|k|v|q_lo|k_lo tile in halfs: 5*HG*32 + 8
    int po;                    // row pitch of a staged [Fp][HG*32] tile (dout, dq) in halfs: HG*32 + 8
};

// Stage rows r < F of one pixel column: `parts` runs of HG*64 bytes per row, `part_stride` halfs apart in global.
// One warp per row (rows strided over the warps), lanes over the row's 16-byte chunks: no integer divisions.
__device__ __forceinline__ void stage_rows(uint32_t dst, int pitch_h, const h16* __restrict__ src, long long row0,
                                           long long row_stride, int ld, int parts, int part_stride, int HG, int F, int Fp) {
    const int cpr = HG * 4;                       // 16-byte chunks per part per row
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int r = warp; r < Fp; r += nw) {
        const uint32_t drow = dst + (uint32_t)(r * pitch_h) * 2u;
        if (r < F) {
            const h16* srow = src + (row0 + (long long)r * row_stride) * ld;
            for (int part = 0; part < parts; ++part)
                for (int ch = lane; ch < cpr; ch += 32)
                    cp16(drow + (uint32_t)(part * HG * 32 + ch * 8) * 2u, srow + part * part_stride + ch * 8);
        } else {
            for (int part = 0; part < parts; ++part)
                for (int ch = lane; ch < cpr; ch += 32)
                    asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(drow + (uint32_t)(part * HG * 32 + ch * 8) * 2u), "r"(0u)
                                 : "memory");
        }
    }
}

// In-place RoPE of this warp's q (times `scale`) and k columns: (x0, x1) -> (x0 c - x1 s, x1 c + x0 s).  The rotated
// values are stored as fp16 hi + lo pairs (lo = fp32 value - hi, in the q_lo / k_lo parts of the tile): logits are
// formed as Q_hi K_hi^T + Q_lo K_hi^T + Q_hi K_lo^T, to fp32 accuracy.  With hi alone, a logit carries an absolute
// error of ~2^-12 |logit|, which at sharp (trained) logits of standard deviation 10 moved the output by 3.5e-3.
// Padded rows get zero lo parts (their hi parts are zeroed by stage_rows).
__device__ __forceinline__ void rotate_qk(uint32_t tile, const Geo& g, int w, int lane, const float* __restrict__ cs,
                                          const float* __restrict__ sn, float scale) {
    for (int idx = lane; idx < g.Fp * 16; idx += 32) {
        const int r = idx >> 4, m = idx & 15;
        const uint32_t aq = tile + (uint32_t)(r * g.pq + w * D + 2 * m) * 2u;
        const uint32_t ak = aq + (uint32_t)(g.HG * D) * 2u;
        const uint32_t aql = aq + (uint32_t)(3 * g.HG * D) * 2u, akl = aq + (uint32_t)(4 * g.HG * D) * 2u;
        if (r >= g.F) {
            sts32(aql, 0u);
            sts32(akl, 0u);
            continue;
        }
        const float c = __ldg(cs + idx), s = __ldg(sn + idx);
        float2 q = unpack_h2(lds32(aq)), k = unpack_h2(lds32(ak));
        q.x *= scale;
        q.y *= scale;
        const float2 qr = make_float2(q.x * c - q.y * s, q.y * c + q.x * s), kr = make_float2(k.x * c - k.y * s, k.y * c + k.x * s);
        const uint32_t qh = pack_h2(qr.x, qr.y), kh = pack_h2(kr.x, kr.y);
        const float2 qhf = unpack_h2(qh), khf = unpack_h2(kh);
        sts32(aq, qh);
        sts32(ak, kh);
        sts32(aql, pack_h2(qr.x - qhf.x, qr.y - qhf.y));
        sts32(akl, pack_h2(kr.x - khf.x, kr.y - khf.y));
    }
}

// A fragments (two k steps of 16) of the 16 x 32 tile at rows r0.. of a staged matrix (column offset col0)
__device__ __forceinline__ void load_a(uint32_t (&a)[2][4], uint32_t base, int pitch_h, int r0, int col0, int lane) {
    const uint32_t addr = base + (uint32_t)((r0 + (lane & 15)) * pitch_h + col0 + (lane >> 4) * 8) * 2u;
    ldsm4(a[0], addr);
    ldsm4(a[1], addr + 32u);
}

// acc[nt] (16 x 8 tiles over all Fp rows of M) = A(16 x 32) * M^T, M = staged [Fp][32] matrix (rows are the n index)
template <int NT>
__device__ __forceinline__ void gemm_nt(float (&acc)[NT][4], const uint32_t (&a)[2][4], uint32_t base, int pitch_h, int col0,
                                        int lane) {
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        uint32_t b[4];
        ldsm4(b, base + (uint32_t)((nt * 8 + (lane & 7)) * pitch_h + col0 + (lane >> 3) * 8) * 2u);
        acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
        mma(acc[nt], a[0], b[0], b[1]);
        mma(acc[nt], a[1], b[2], b[3]);
    }
}

// the same for logits from hi / lo pairs: acc = A_hi M_hi^T + A_lo M_hi^T + A_hi M_lo^T (small terms first)
template <int NT>
__device__ __forceinline__ void gemm_nt_split(float (&acc)[NT][4], const uint32_t (&a)[2][4], const uint32_t (&al)[2][4],
                                              uint32_t base, int pitch_h, int col0, int col0_lo, int lane) {
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const uint32_t row = base + (uint32_t)((nt * 8 + (lane & 7)) * pitch_h + (lane >> 3) * 8) * 2u;
        uint32_t b[4], bl[4];
        ldsm4(b, row + (uint32_t)col0 * 2u);
        ldsm4(bl, row + (uint32_t)col0_lo * 2u);
        acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
        mma(acc[nt], al[0], b[0], b[1]);
        mma(acc[nt], al[1], b[2], b[3]);
        mma(acc[nt], a[0], bl[0], bl[1]);
        mma(acc[nt], a[1], bl[2], bl[3]);
        mma(acc[nt], a[0], b[0], b[1]);
        mma(acc[nt], a[1], b[2], b[3]);
    }
}

// out[nd] (16 x 32) = P(16 x Fp, fp32 accumulator fragments) * M, M = staged [Fp][32] matrix (rows are the k index)
template <int NT>
__device__ __forceinline__ void gemm_pv(float (&out)[4][4], const float (&p)[NT][4], uint32_t base, int pitch_h, int col0,
                                        int lane) {
#pragma unroll
    for (int i = 0; i < 4; ++i) out[i][0] = out[i][1] = out[i][2] = out[i][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < NT / 2; ++kk) {
        uint32_t a[4];
        a[0] = pack_h2(p[2 * kk][0], p[2 * kk][1]);
        a[1] = pack_h2(p[2 * kk][2], p[2 * kk][3]);
        a[2] = pack_h2(p[2 * kk + 1][0], p[2 * kk + 1][1]);
        a[3] = pack_h2(p[2 * kk + 1][2], p[2 * kk + 1][3]);
        const uint32_t row = base + (uint32_t)((kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * pitch_h + col0 +
                                               (lane >> 4) * 8) * 2u;
#pragma unroll
        for (int np = 0; np < 2; ++np) {
            uint32_t b[4];
            ldsm4_t(b, row + np * 32u);
            mma(out[2 * np], a, b[0], b[1]);
            mma(out[2 * np + 1], a, b[2], b[3]);
        }
    }
}

// store a 16 x 32 accumulator tile as fp16 at rows r0.. of a staged matrix
__device__ __forceinline__ void store_tile(const float (&o)[4][4], uint32_t base, int pitch_h, int r0, int col0, int lane) {
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int nd = 0; nd < 4; ++nd) {
        const uint32_t a = base + (uint32_t)((r0 + g) * pitch_h + col0 + nd * 8 + 2 * t) * 2u;
        sts32(a, pack_h2(o[nd][0], o[nd][1]));
        sts32(a + (uint32_t)(8 * pitch_h) * 2u, pack_h2(o[nd][2], o[nd][3]));
    }
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <int NT>  // NT = Fp / 8
__global__ void __launch_bounds__(256)
tattn_long_fwd_kernel(const h16* __restrict__ qkv, const float* __restrict__ bias_diag, const float* __restrict__ cs,
                      const float* __restrict__ sn, h16* __restrict__ out, float* __restrict__ lse, long long npix, Geo g,
                      float scale) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t tile = smem_u32(smem);
    float* bd = reinterpret_cast<float*>(smem + (size_t)g.Fp * g.pq * 2);   // [HG][2*Fp] bias by diagonal
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int h0 = blockIdx.y * g.HG;
    const int ld = 3 * g.H * D;
    // bd[hh][delta + Fp - 1], delta = key - query; entries outside |delta| < F belong to padded rows only
    for (int i = threadIdx.x; i < g.HG * 2 * g.Fp; i += blockDim.x) {
        const int hh = i / (2 * g.Fp), delta = i - hh * 2 * g.Fp - (g.Fp - 1);
        bd[i] = (delta > -g.F && delta < g.F) ? bias_diag[(h0 + hh) * (2 * g.F - 1) + delta + g.F - 1] : 0.f;
    }
    const int gq = lane >> 2, t = lane & 3;
    for (long long pix = blockIdx.x; pix < npix; pix += gridDim.x) {
        const long long b = pix / g.HW, hw = pix - b * g.HW;
        const long long row0 = b * g.F * g.HW + hw;
        __syncthreads();  // the previous column's output rows have been stored
        stage_rows(tile, g.pq, qkv + h0 * D, row0, g.HW, ld, 3, g.H * D, g.HG, g.F, g.Fp);
        cp_wait_all();
        __syncthreads();
        rotate_qk(tile, g, w, lane, cs, sn, scale);
        __syncwarp();
        const float* bw = bd + w * 2 * g.Fp + (g.Fp - 1);
#pragma unroll 1
        for (int mt = 0; mt < NT / 2; ++mt) {
            uint32_t a[2][4], al[2][4];
            load_a(a, tile, g.pq, mt * 16, w * D, lane);
            load_a(al, tile, g.pq, mt * 16, 3 * g.HG * D + w * D, lane);
            float s[NT][4];
            gemm_nt_split<NT>(s, a, al, tile, g.pq, g.HG * D + w * D, 4 * g.HG * D + w * D, lane);
            const int i0 = mt * 16 + gq, i1 = i0 + 8;
            float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int j = nt * 8 + 2 * t;
                s[nt][0] = j < g.F ? s[nt][0] + bw[j - i0] : -INFINITY;
                s[nt][1] = j + 1 < g.F ? s[nt][1] + bw[j + 1 - i0] : -INFINITY;
                s[nt][2] = j < g.F ? s[nt][2] + bw[j - i1] : -INFINITY;
                s[nt][3] = j + 1 < g.F ? s[nt][3] + bw[j + 1 - i1] : -INFINITY;
                m0 = fmaxf(m0, fmaxf(s[nt][0], s[nt][1]));
                m1 = fmaxf(m1, fmaxf(s[nt][2], s[nt][3]));
            }
            m0 = quad_max(m0);
            m1 = quad_max(m1);
            float l0 = 0.f, l1 = 0.f;
            const float m0l = m0 * kLog2e, m1l = m1 * kLog2e;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                s[nt][0] = exp_sub(s[nt][0], m0l);
                s[nt][1] = exp_sub(s[nt][1], m0l);
                s[nt][2] = exp_sub(s[nt][2], m1l);
                s[nt][3] = exp_sub(s[nt][3], m1l);
                l0 += s[nt][0] + s[nt][1];
                l1 += s[nt][2] + s[nt][3];
            }
            l0 = quad_sum(l0);
            l1 = quad_sum(l1);
            const float r0 = 1.f / l0, r1 = 1.f / l1;   // applied to the 16 x 32 output tile, not to the 16 x F probabilities
            if (t == 0) {
                if (i0 < g.F) lse[(row0 + (long long)i0 * g.HW) * g.H + h0 + w] = m0 + __logf(l0);
                if (i1 < g.F) lse[(row0 + (long long)i1 * g.HW) * g.H + h0 + w] = m1 + __logf(l1);
            }
            float o[4][4];
            gemm_pv<NT>(o, s, tile, g.pq, 2 * g.HG * D + w * D, lane);
#pragma unroll
            for (int nd = 0; nd < 4; ++nd) {
                o[nd][0] *= r0;
                o[nd][1] *= r0;
                o[nd][2] *= r1;
                o[nd][3] *= r1;
            }
            store_tile(o, tile, g.pq, mt * 16, w * D, lane);   // over this tile's (consumed) q rows
        }
        __syncthreads();
        // out rows: HG*64 contiguous bytes per frame (one warp per row, lanes over 16-byte chunks)
        const int cpr = g.HG * 4;
        for (int r = w; r < g.F; r += (int)(blockDim.x >> 5)) {
            h16* orow = out + (row0 + (long long)r * g.HW) * (g.H * D) + h0 * D;
            for (int ch = lane; ch < cpr; ch += 32)
                *reinterpret_cast<uint4*>(orow + ch * 8) = *reinterpret_cast<const uint4*>(smem + (size_t)(r * g.pq + ch * 8) * 2);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(256)
tattn_long_bwd_kernel(const h16* __restrict__ qkv, const float* __restrict__ bias_diag, const float* __restrict__ cs,
                      const float* __restrict__ sn, const h16* __restrict__ out, const float* __restrict__ lse,
                      const h16* __restrict__ dout, h16* __restrict__ dqkv, float* __restrict__ dbias_diag, long long npix,
                      Geo g, float scale) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t tile = smem_u32(smem);
    const uint32_t t_do = tile + (uint32_t)g.Fp * g.pq * 2u;       // staged dout [Fp][HG*32]
    const uint32_t t_dq = t_do + (uint32_t)g.Fp * g.po * 2u;       // dq staging  [Fp][HG*32]
    uint8_t* fbase = smem + (size_t)g.Fp * g.pq * 2 + 2 * (size_t)g.Fp * g.po * 2;
    float* bd = reinterpret_cast<float*>(fbase);                   // [HG][2*Fp] bias by diagonal
    float* gd = bd + g.HG * 2 * g.Fp;                              // [HG][2*Fp] its gradient (whole kernel)
    float* s_lse = gd + g.HG * 2 * g.Fp;                           // [HG][Fp]
    float* s_dl = s_lse + g.HG * g.Fp;                             // [HG][Fp] delta_i = dO_i . O_i
    const int ps = g.Fp + 4;                                       // pitch of the per-warp dS scratch
    float* s_ds = s_dl + g.HG * g.Fp;                              // [HG][16][Fp + 4]
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int h0 = blockIdx.y * g.HG;
    const int ld = 3 * g.H * D, lo = g.H * D;
    for (int i = threadIdx.x; i < g.HG * 2 * g.Fp; i += blockDim.x) {
        const int hh = i / (2 * g.Fp), delta = i - hh * 2 * g.Fp - (g.Fp - 1);
        bd[i] = (delta > -g.F && delta < g.F) ? bias_diag[(h0 + hh) * (2 * g.F - 1) + delta + g.F - 1] : 0.f;
        gd[i] = 0.f;
    }
    const int gq = lane >> 2, t = lane & 3;
    const float* bw = bd + w * 2 * g.Fp + (g.Fp - 1);
    float* gw = gd + w * 2 * g.Fp + (g.Fp - 1);
    float* lw = s_lse + w * g.Fp;
    float* dw = s_dl + w * g.Fp;
    float* sw = s_ds + w * 16 * ps;
    for (long long pix = blockIdx.x; pix < npix; pix += gridDim.x) {
        const long long b = pix / g.HW, hw = pix - b * g.HW;
        const long long row0 = b * g.F * g.HW + hw;
        __syncthreads();  // the previous column's gradients have been stored
        stage_rows(tile, g.pq, qkv + h0 * D, row0, g.HW, ld, 3, g.H * D, g.HG, g.F, g.Fp);
        stage_rows(t_do, g.po, dout + h0 * D, row0, g.HW, lo, 1, 0, g.HG, g.F, g.Fp);
        cp_wait_all();
        __syncthreads();
        rotate_qk(tile, g, w, lane, cs, sn, scale);
        // delta_i and lse_i of this warp's head
        for (int r = lane; r < g.Fp; r += 32) {
            float dl = 0.f, ls = 0.f;
            if (r < g.F) {
                const long long row = row0 + (long long)r * g.HW;
                const uint4* op = reinterpret_cast<const uint4*>(out + row * lo + (h0 + w) * D);
                const uint4* dp = reinterpret_cast<const uint4*>(smem + (size_t)g.Fp * g.pq * 2 + (size_t)(r * g.po + w * D) * 2);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const uint4 a = __ldg(op + c), d4 = dp[c];
                    const float2 a0 = unpack_h2(a.x), a1 = unpack_h2(a.y), a2 = unpack_h2(a.z), a3 = unpack_h2(a.w);
                    const float2 d0 = unpack_h2(d4.x), d1 = unpack_h2(d4.y), d2 = unpack_h2(d4.z), d3 = unpack_h2(d4.w);
                    dl += a0.x * d0.x + a0.y * d0.y + a1.x * d1.x + a1.y * d1.y + a2.x * d2.x + a2.y * d2.y + a3.x * d3.x +
                          a3.y * d3.y;
                }
                ls = lse[row * g.H + h0 + w];
            }
            dw[r] = dl;
            lw[r] = ls;
        }
        __syncwarp();
        // ---- pass B: per query tile, dQ = dS K ----
#pragma unroll 1
        for (int mt = 0; mt < NT / 2; ++mt) {
            uint32_t a[2][4];
            float s[NT][4], dp[NT][4];
            {
                uint32_t al[2][4];
                load_a(a, tile, g.pq, mt * 16, w * D, lane);
                load_a(al, tile, g.pq, mt * 16, 3 * g.HG * D + w * D, lane);
                gemm_nt_split<NT>(s, a, al, tile, g.pq, g.HG * D + w * D, 4 * g.HG * D + w * D, lane);   // S = Q K^T
            }
            load_a(a, t_do, g.po, mt * 16, w * D, lane);
            gemm_nt<NT>(dp, a, tile, g.pq, 2 * g.HG * D + w * D, lane);            // dP = dO V^T
            const int i0 = mt * 16 + gq, i1 = i0 + 8;
            const float l0 = lw[i0] * kLog2e, l1 = lw[i1] * kLog2e, e0 = dw[i0], e1 = dw[i1];
            const bool v0 = i0 < g.F, v1 = i1 < g.F;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int j = nt * 8 + 2 * t;
                const bool c0 = j < g.F, c1 = j + 1 < g.F;
                const float p0 = (v0 && c0) ? exp_sub(s[nt][0] + bw[j - i0], l0) : 0.f;
                const float p1 = (v0 && c1) ? exp_sub(s[nt][1] + bw[j + 1 - i0], l0) : 0.f;
                const float p2 = (v1 && c0) ? exp_sub(s[nt][2] + bw[j - i1], l1) : 0.f;
                const float p3 = (v1 && c1) ? exp_sub(s[nt][3] + bw[j + 1 - i1], l1) : 0.f;
                s[nt][0] = p0 * (dp[nt][0] - e0);
                s[nt][1] = p1 * (dp[nt][1] - e0);
                s[nt][2] = p2 * (dp[nt][2] - e1);
                s[nt][3] = p3 * (dp[nt][3] - e1);
                // dS tile -> this warp's scratch (row-major fp32) for the per-diagonal bias gradient below
                *reinterpret_cast<float2*>(sw + gq * ps + nt * 8 + 2 * t) = make_float2(s[nt][0], s[nt][1]);
                *reinterpret_cast<float2*>(sw + (gq + 8) * ps + nt * 8 + 2 * t) = make_float2(s[nt][2], s[nt][3]);
            }
            // bias gradient by diagonal (key - query): each diagonal of the 16 x Fp tile belongs to ONE lane, which
            // sums its <= 16 entries (masked entries are exact zeros) and adds them to the warp's own table: no atomics
            __syncwarp();
            for (int d = lane; d < g.Fp + 15; d += 32) {
                float acc = 0.f;
#pragma unroll
                for (int v = 0; v < 16; ++v) {
                    const int c = v + d - 15;
                    if (c >= 0 && c < g.Fp) acc += sw[v * ps + c];
                }
                gw[d - 15 - mt * 16] += acc;
            }
            __syncwarp();
            float dq[4][4];
            gemm_pv<NT>(dq, s, tile, g.pq, g.HG * D + w * D, lane);                // dQ_rot = dS K
            // undo RoPE (transpose of the rotation) and the scale; pairs (2m, 2m+1) are adjacent fragment columns
#pragma unroll
            for (int nd = 0; nd < 4; ++nd) {
                const int m = nd * 4 + t;
                if (v0) {
                    const float c = __ldg(cs + i0 * 16 + m), sn_ = __ldg(sn + i0 * 16 + m);
                    const float g0 = dq[nd][0], g1 = dq[nd][1];
                    dq[nd][0] = (g0 * c + g1 * sn_) * scale;
                    dq[nd][1] = (g1 * c - g0 * sn_) * scale;
                }
                if (v1) {
                    const float c = __ldg(cs + i1 * 16 + m), sn_ = __ldg(sn + i1 * 16 + m);
                    const float g0 = dq[nd][2], g1 = dq[nd][3];
                    dq[nd][2] = (g0 * c + g1 * sn_) * scale;
                    dq[nd][3] = (g1 * c - g0 * sn_) * scale;
                }
            }
            store_tile(dq, t_dq, g.po, mt * 16, w * D, lane);
        }
        __syncwarp();
        // ---- pass A: per key tile, dV = P^T dO and dK = dS^T Q (transposed problem: rows are keys) ----
#pragma unroll 1
        for (int jt = 0; jt < NT / 2; ++jt) {
            uint32_t a[2][4];
            float st[NT][4], dpt[NT][4];
            {
                uint32_t al[2][4];
                load_a(a, tile, g.pq, jt * 16, g.HG * D + w * D, lane);
                load_a(al, tile, g.pq, jt * 16, 4 * g.HG * D + w * D, lane);
                gemm_nt_split<NT>(st, a, al, tile, g.pq, w * D, 3 * g.HG * D + w * D, lane);          // S^T = K Q^T
            }
            load_a(a, tile, g.pq, jt * 16, 2 * g.HG * D + w * D, lane);
            gemm_nt<NT>(dpt, a, t_do, g.po, w * D, lane);                          // dP^T = V dO^T
            const int j0 = jt * 16 + gq, j1 = j0 + 8;
            const bool v0 = j0 < g.F, v1 = j1 < g.F;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int i = nt * 8 + 2 * t;
                const bool c0 = i < g.F, c1 = i + 1 < g.F;
                const float la = lw[i] * kLog2e, lb = lw[i + 1] * kLog2e, ea = dw[i], eb = dw[i + 1];
                const float p0 = (v0 && c0) ? exp_sub(st[nt][0] + bw[j0 - i], la) : 0.f;
                const float p1 = (v0 && c1) ? exp_sub(st[nt][1] + bw[j0 - i - 1], lb) : 0.f;
                const float p2 = (v1 && c0) ? exp_sub(st[nt][2] + bw[j1 - i], la) : 0.f;
                const float p3 = (v1 && c1) ? exp_sub(st[nt][3] + bw[j1 - i - 1], lb) : 0.f;
                st[nt][0] = p0;
                st[nt][1] = p1;
                st[nt][2] = p2;
                st[nt][3] = p3;
                dpt[nt][0] = p0 * (dpt[nt][0] - ea);
                dpt[nt][1] = p1 * (dpt[nt][1] - eb);
                dpt[nt][2] = p2 * (dpt[nt][2] - ea);
                dpt[nt][3] = p3 * (dpt[nt][3] - eb);
            }
            float dv[4][4], dk[4][4];
            gemm_pv<NT>(dv, st, t_do, g.po, w * D, lane);                          // dV = P^T dO
            gemm_pv<NT>(dk, dpt, tile, g.pq, w * D, lane);                         // dK_rot = dS^T Q
#pragma unroll
            for (int nd = 0; nd < 4; ++nd) {
                const int m = nd * 4 + t;
                if (v0) {
                    const float c = __ldg(cs + j0 * 16 + m), sn_ = __ldg(sn + j0 * 16 + m);
                    const float g0 = dk[nd][0], g1 = dk[nd][1];
                    dk[nd][0] = g0 * c + g1 * sn_;
                    dk[nd][1] = g1 * c - g0 * sn_;
                }
                if (v1) {
                    const float c = __ldg(cs + j1 * 16 + m), sn_ = __ldg(sn + j1 * 16 + m);
                    const float g0 = dk[nd][2], g1 = dk[nd][3];
                    dk[nd][2] = g0 * c + g1 * sn_;
                    dk[nd][3] = g1 * c - g0 * sn_;
                }
            }
            __syncwarp();  // every lane has issued its ldmatrix reads of this key tile's k / v rows
            store_tile(dk, tile, g.pq, jt * 16, g.HG * D + w * D, lane);           // over this key tile's k rows
            store_tile(dv, tile, g.pq, jt * 16, 2 * g.HG * D + w * D, lane);       // ... and v rows
        }
        __syncthreads();
        // dq | dk | dv rows out: three runs of HG*64 bytes per frame (one warp per row)
        const int cpr = g.HG * 4;
        const uint8_t* sdq = smem + (size_t)g.Fp * g.pq * 2 + (size_t)g.Fp * g.po * 2;
        for (int r = w; r < g.F; r += (int)(blockDim.x >> 5)) {
            h16* grow = dqkv + (row0 + (long long)r * g.HW) * ld + h0 * D;
            for (int ch = lane; ch < cpr; ch += 32) {
                *reinterpret_cast<uint4*>(grow + ch * 8) = *reinterpret_cast<const uint4*>(sdq + (size_t)(r * g.po + ch * 8) * 2);
                *reinterpret_cast<uint4*>(grow + g.H * D + ch * 8) =
                    *reinterpret_cast<const uint4*>(smem + (size_t)(r * g.pq + g.HG * D + ch * 8) * 2);
                *reinterpret_cast<uint4*>(grow + 2 * g.H * D + ch * 8) =
                    *reinterpret_cast<const uint4*>(smem + (size_t)(r * g.pq + 2 * g.HG * D + ch * 8) * 2);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < g.HG * (2 * g.F - 1); i += blockDim.x) {
        const int hh = i / (2 * g.F - 1), dd = i - hh * (2 * g.F - 1);   // dd = delta + F - 1
        const float v = gd[hh * 2 * g.Fp + dd + (g.Fp - g.F)];
        if (v != 0.f) atomicAdd(dbias_diag + (h0 + hh) * (2 * g.F - 1) + dd, v);
    }
}

static size_t fwd_smem(const Geo& g) { return (size_t)g.Fp * g.pq * 2 + (size_t)g.HG * 2 * g.Fp * 4; }
static size_t bwd_smem(const Geo& g) {
    return (size_t)g.Fp * g.pq * 2 + 2 * (size_t)g.Fp * g.po * 2 + (size_t)g.HG * 2 * g.Fp * 4 * 2 + (size_t)g.HG * g.Fp * 4 * 2 +
           (size_t)g.HG * 16 * (g.Fp + 4) * 4;
}
static Geo make_geo(int F, int HW, int H, int HG) {
    Geo g;
    g.F = F;
    g.Fp = (F + 15) / 16 * 16;
    g.HW = HW;
    g.H = H;
    g.HG = HG;
    g.pq = 5 * HG * D + 8;
    g.po = HG * D + 8;
    return g;
}
// the largest head group (a divisor of H) whose staging fits two CTAs per SM, else one
static Geo pick_geo(int F, int HW, int H, bool bwd) {
    for (int pass = 0; pass < 2; ++pass) {
        const size_t cap = pass == 0 ? 112 * 1024 : 226 * 1024;
        for (int hg = H; hg >= 1; --hg) {
            if (H % hg) continue;
            Geo g = make_geo(F, HW, H, hg);
            if ((bwd ? bwd_smem(g) : fwd_smem(g)) <= cap) return g;
        }
    }
    return make_geo(F, HW, H, 0);
}

}  // namespace tl
}  // namespace cesm

using namespace cesm;

#define TL_DISPATCH(NTV, CALL)          \
    switch (NTV) {                      \
        case 2: { constexpr int NT = 2; CALL; } break;   \
        case 4: { constexpr int NT = 4; CALL; } break;   \
        case 6: { constexpr int NT = 6; CALL; } break;   \
        case 8: { constexpr int NT = 8; CALL; } break;   \
        case 12: { constexpr int NT = 12; CALL; } break; \
        case 16: { constexpr int NT = 16; CALL; } break; \
        default: CESM_REQUIRE(false, "long temporal attention supports F <= 128 in steps of 16 up to 64, then 96 / 128 (padded F = %d)", 8 * (NTV)); \
    }

extern "C" int cesm_tattn_long_max_frames(void) { return 128; }

extern "C" int cesm_tattn_long_fwd(const void* qkv, const float* bias_diag, const float* cs, const float* sn, void* out,
                                   float* lse, int B, int F, int HW, int H, int dim_head, float scale, void* stream) {
    CESM_REQUIRE(dim_head == tl::D, "temporal attention kernel needs dim_head == 32 (got %d)", dim_head);
    CESM_REQUIRE(H >= 1 && H <= 8 && F >= 1 && F <= 128, "long temporal attention: 1..8 heads, 1..128 frames (H=%d F=%d)", H, F);
    tl::Geo g = tl::pick_geo(F, HW, H, false);
    CESM_REQUIRE(g.HG > 0, "long temporal attention: F=%d does not fit in shared memory", F);
    const int nt = g.Fp / 8 <= 8 ? g.Fp / 8 : (g.Fp <= 96 ? 12 : 16);
    if (nt * 8 != g.Fp) {  // 80 / 112 frames: pad further to the next instantiated size
        g.Fp = nt * 8;
        CESM_REQUIRE(tl::fwd_smem(g) <= 226 * 1024, "long temporal attention: F=%d does not fit in shared memory", F);
    }
    const size_t sm = tl::fwd_smem(g);
    const long long npix = (long long)B * HW;
    dim3 grid((unsigned)(npix < 148 * 2 ? npix : 148 * 2), (unsigned)(H / g.HG));
    cudaStream_t st = as_stream(stream);
    TL_DISPATCH(nt, {
        static bool cfg = false;
        if (!cfg) {
            CESM_CHECK_CUDA(cudaFuncSetAttribute(tl::tattn_long_fwd_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
            cfg = true;
        }
        launch_pdl(tl::tattn_long_fwd_kernel<NT>, grid, 32 * g.HG, sm, st, (const h16*)qkv, bias_diag, cs, sn, (h16*)out, lse,
                   npix, g, scale);
    })
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_tattn_long_bwd(const void* qkv, const float* bias_diag, const float* cs, const float* sn, const void* out,
                                   const float* lse, const void* dout, void* dqkv, float* dbias_diag, int B, int F, int HW,
                                   int H, int dim_head, float scale, void* stream) {
    CESM_REQUIRE(dim_head == tl::D, "temporal attention kernel needs dim_head == 32 (got %d)", dim_head);
    CESM_REQUIRE(H >= 1 && H <= 8 && F >= 1 && F <= 128, "long temporal attention: 1..8 heads, 1..128 frames (H=%d F=%d)", H, F);
    tl::Geo g = tl::pick_geo(F, HW, H, true);
    CESM_REQUIRE(g.HG > 0, "long temporal attention backward: F=%d does not fit in shared memory", F);
    const int nt = g.Fp / 8 <= 8 ? g.Fp / 8 : (g.Fp <= 96 ? 12 : 16);
    if (nt * 8 != g.Fp) {
        g.Fp = nt * 8;
        CESM_REQUIRE(tl::bwd_smem(g) <= 226 * 1024, "long temporal attention backward: F=%d does not fit in shared memory", F);
    }
    const size_t sm = tl::bwd_smem(g);
    const long long npix = (long long)B * HW;
    cudaStream_t st = as_stream(stream);
    CESM_ZERO_SCRATCH(dbias_diag, sizeof(float) * H * (2 * F - 1), st);
    dim3 grid((unsigned)(npix < 148 * 2 ? npix : 148 * 2), (unsigned)(H / g.HG));
    TL_DISPATCH(nt, {
        static bool cfg = false;
        if (!cfg) {
            CESM_CHECK_CUDA(cudaFuncSetAttribute(tl::tattn_long_bwd_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
            cfg = true;
        }
        launch_pdl(tl::tattn_long_bwd_kernel<NT>, grid, 32 * g.HG, sm, st, (const h16*)qkv, bias_diag, cs, sn, (const h16*)out,
                   lse, (const h16*)dout, (h16*)dqkv, dbias_diag, npix, g, scale);
    })
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}
