// Bottleneck ("mid") spatial attention, use_mid_attn=True (video_net.py:713-719 + the Attention of :368-454 with no
// rotary embedding, no position bias and no mask): per image (b, f) and head, softmax((q * 32^-0.5) k^T) v over ALL
// n = h*w pixels of the frame, flash style on the tensor cores (mma.sync.m16n8k16, fp16 operands, fp32 accumulate).
//
// The sequence of one image is its n pixel rows, contiguous in the channels-last q|k|v tensor [NI*n][3*H*32], so a
// head's q / k / v tile is a run of 64-byte row slices.  A CTA owns 64 rows (4 warps x 16) of one (image, head):
//
//   forward      (per query tile): Q in registers; K / V tiles of 64 keys double-buffered in shared memory with
//                cp.async; S = Q K^T, online softmax in the accumulator registers (scale * log2 e folded into the
//                ex2), O += P V.  Writes O and lse = log sum_j exp(scale q.k_j) (natural log).
//   backward dQ  (per query tile): recomputes P from q, k and lse; delta_i = dO_i . O_i for its own rows (written to
//                a caller-provided fp32 buffer for the next kernel); dP = dO V^T, dS = P (dP - delta), dQ += dS K.
//   backward dKdV (per key tile, transposed so that the accumulators belong to the keys): S^T = K Q^T,
//                dP^T = V dO^T, dV += P^T dO, dK += dS^T Q over all query tiles.
// Each output row is produced by exactly one warp: no atomics, the backward is bitwise deterministic.
// Only P and dS are rounded to fp16 (as MMA operands); nothing is clamped, so a non-finite score reaches the output
// and, in training, the loss scaler's found-inf check.
//
// Tails: keys >= n are zero-filled in shared memory and their scores set to -inf (forward, dQ); queries >= n are
// zero-filled with lse = +inf, so their probabilities are exactly 0 (dKdV); rows >= n are never stored.
#include "api_common.h"
#include "common.cuh"

namespace cesm {
namespace ma {

static constexpr int D = 32;        // dim_head: the reference's Attention default, which the mid block always uses
static constexpr int BR = 64;       // rows (queries or keys) per CTA: 4 warps x 16
static constexpr int BC = 64;       // rows per streamed tile
static constexpr int PITCH = D + 8; // staged row pitch in halfs (80 bytes: ldmatrix rows hit distinct bank groups)
static constexpr int TILE_H = BC * PITCH;
static constexpr int NTH = 128;

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
// 16-byte async copy; `valid` = false zero-fills the destination without reading the source
__device__ __forceinline__ void cp16z(uint32_t dst, const void* src, bool valid) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ float quad_max(float v) {
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
    return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// Stage rows r0 .. r0+63 (< n) of one head's 32-column slice: `src` points at column 0 of the slice in image row 0,
// `ld` is the row length in halfs.  128 threads x 2 chunks of 16 bytes; rows >= n are zero-filled.
__device__ __forceinline__ void stage(uint32_t dst, const h16* __restrict__ src, long long ld, int r0, int n) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int c = threadIdx.x + k * NTH;   // 0..255
        const int r = c >> 2, ch = c & 3;
        const bool ok = r0 + r < n;
        cp16z(dst + (uint32_t)(r * PITCH + ch * 8) * 2u, ok ? src + (long long)(r0 + r) * ld + ch * 8 : src, ok);
    }
}

// A fragments (two k steps of 16) of the 16 x 32 tile at rows r0.. of a staged [.][PITCH] matrix
__device__ __forceinline__ void load_a(uint32_t (&a)[2][4], uint32_t base, int r0, int lane) {
    const uint32_t addr = base + (uint32_t)((r0 + (lane & 15)) * PITCH + (lane >> 4) * 8) * 2u;
    ldsm4(a[0], addr);
    ldsm4(a[1], addr + 32u);
}

// acc[nt] (16 x 64) = A(16 x 32) * M^T, M = staged [64][32] tile (its rows are the n index)
__device__ __forceinline__ void gemm_nt(float (&acc)[8][4], const uint32_t (&a)[2][4], uint32_t base, int lane) {
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        uint32_t b[4];
        ldsm4(b, base + (uint32_t)((nt * 8 + (lane & 7)) * PITCH + (lane >> 3) * 8) * 2u);
        acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
        mma(acc[nt], a[0], b[0], b[1]);
        mma(acc[nt], a[1], b[2], b[3]);
    }
}

// out[nd] (16 x 32) += P(16 x 64, fp32 accumulator fragments, rounded to fp16 here) * M, M = staged [64][32] tile
// (its rows are the k index)
__device__ __forceinline__ void gemm_pv_acc(float (&out)[4][4], const float (&p)[8][4], uint32_t base, int lane) {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        uint32_t a[4];
        a[0] = pack_h2(p[2 * kk][0], p[2 * kk][1]);
        a[1] = pack_h2(p[2 * kk][2], p[2 * kk][3]);
        a[2] = pack_h2(p[2 * kk + 1][0], p[2 * kk + 1][1]);
        a[3] = pack_h2(p[2 * kk + 1][2], p[2 * kk + 1][3]);
        const uint32_t row = base + (uint32_t)((kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * PITCH + (lane >> 4) * 8) * 2u;
#pragma unroll
        for (int np = 0; np < 2; ++np) {
            uint32_t b[4];
            ldsm4_t(b, row + np * 32u);
            mma(out[2 * np], a, b[0], b[1]);
            mma(out[2 * np + 1], a, b[2], b[3]);
        }
    }
}

// store a 16 x 32 accumulator tile (times `mul0` / `mul1` for its rows g / g+8) as fp16 rows of a global matrix;
// `dst` points at column 0 of the slice in this warp's first row, rows >= `valid` are skipped
__device__ __forceinline__ void store_rows(const float (&o)[4][4], h16* __restrict__ dst, long long ld, int valid,
                                           float mul0, float mul1, int lane) {
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int nd = 0; nd < 4; ++nd) {
        if (g < valid)
            *reinterpret_cast<uint32_t*>(dst + (long long)g * ld + nd * 8 + 2 * t) = pack_h2(o[nd][0] * mul0, o[nd][1] * mul0);
        if (g + 8 < valid)
            *reinterpret_cast<uint32_t*>(dst + (long long)(g + 8) * ld + nd * 8 + 2 * t) =
                pack_h2(o[nd][2] * mul1, o[nd][3] * mul1);
    }
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
// grid (ceil(n / 64), H, NI), 128 threads
__global__ void __launch_bounds__(NTH)
mattn_fwd_kernel(const h16* __restrict__ qkv, h16* __restrict__ out, float* __restrict__ lse, int n, int H, float sl2) {
    pdl_trigger();
    __shared__ __align__(128) h16 smem[TILE_H * 5];   // Q | K[2] | V[2]
    const uint32_t sQ = smem_u32(smem), sK = sQ + TILE_H * 2, sV = sK + 2 * TILE_H * 2;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, gq = lane >> 2, t = lane & 3;
    const int q0 = blockIdx.x * BR, h = blockIdx.y;
    const long long img = blockIdx.z;
    const int hid = H * D;
    const long long ld = 3LL * hid;
    const h16* base = qkv + img * n * ld + h * D;
    pdl_wait();
    stage(sQ, base, ld, q0, n);
    stage(sK, base + hid, ld, 0, n);
    stage(sV, base + 2 * hid, ld, 0, n);
    cp_commit();
    const int ntiles = (n + BC - 1) / BC;
    uint32_t qa[2][4];
    float o[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;   // running max (raw scores), per-thread partial sums
#pragma unroll 1
    for (int kt = 0; kt < ntiles; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < ntiles) {
            stage(sK + (buf ^ 1) * TILE_H * 2, base + hid, ld, (kt + 1) * BC, n);
            stage(sV + (buf ^ 1) * TILE_H * 2, base + 2 * hid, ld, (kt + 1) * BC, n);
            cp_commit();
            cp_wait<1>();
        } else {
            cp_wait<0>();
        }
        __syncthreads();
        if (kt == 0) load_a(qa, sQ, w * 16, lane);
        float s[8][4];
        gemm_nt(s, qa, sK + buf * TILE_H * 2, lane);
        if ((kt + 1) * BC > n) {   // tail tile: keys >= n do not exist
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const int j = kt * BC + nt * 8 + 2 * t;
                if (j >= n) s[nt][0] = s[nt][2] = -INFINITY;
                if (j + 1 >= n) s[nt][1] = s[nt][3] = -INFINITY;
            }
        }
        float mx0 = m0, mx1 = m1;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            mx0 = fmaxf(mx0, fmaxf(s[nt][0], s[nt][1]));
            mx1 = fmaxf(mx1, fmaxf(s[nt][2], s[nt][3]));
        }
        mx0 = quad_max(mx0);
        mx1 = quad_max(mx1);
        const float ml0 = mx0 * sl2, ml1 = mx1 * sl2;
        const float a0 = ex2_ftz(fmaf(m0, sl2, -ml0)), a1 = ex2_ftz(fmaf(m1, sl2, -ml1));   // 0 on the first tile
        m0 = mx0;
        m1 = mx1;
        l0 *= a0;
        l1 *= a1;
#pragma unroll
        for (int nd = 0; nd < 4; ++nd) {
            o[nd][0] *= a0;
            o[nd][1] *= a0;
            o[nd][2] *= a1;
            o[nd][3] *= a1;
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            s[nt][0] = ex2_ftz(fmaf(s[nt][0], sl2, -ml0));
            s[nt][1] = ex2_ftz(fmaf(s[nt][1], sl2, -ml0));
            s[nt][2] = ex2_ftz(fmaf(s[nt][2], sl2, -ml1));
            s[nt][3] = ex2_ftz(fmaf(s[nt][3], sl2, -ml1));
            l0 += s[nt][0] + s[nt][1];
            l1 += s[nt][2] + s[nt][3];
        }
        gemm_pv_acc(o, s, sV + buf * TILE_H * 2, lane);
        __syncthreads();   // every warp is done with this buffer before the next iteration refills it
    }
    l0 = quad_sum(l0);
    l1 = quad_sum(l1);
    const int r0 = q0 + w * 16;
    const int valid = n - r0;
    if (valid > 0) {
        const long long row = img * n + r0;
        store_rows(o, out + row * hid + h * D, hid, valid, 1.f / l0, 1.f / l1, lane);
        if (t == 0) {
            const float scale = sl2 * (1.f / kLog2e);
            if (gq < valid) lse[(row + gq) * H + h] = m0 * scale + __logf(l0);
            if (gq + 8 < valid) lse[(row + gq + 8) * H + h] = m1 * scale + __logf(l1);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// backward: dQ (+ delta)
// ------------------------------------------------------------------------------------------------
// grid (ceil(n / 64), H, NI), 128 threads.  delta: fp32 [NI*n][H] written here, read by mattn_bwd_dkdv_kernel.
__global__ void __launch_bounds__(NTH)
mattn_bwd_dq_kernel(const h16* __restrict__ qkv, const h16* __restrict__ out, const float* __restrict__ lse,
                    const h16* __restrict__ dout, h16* __restrict__ dqkv, float* __restrict__ delta, int n, int H, float sl2) {
    pdl_trigger();
    __shared__ __align__(128) h16 smem[TILE_H * 6];   // Q | dO | K[2] | V[2]
    const uint32_t sQ = smem_u32(smem), sO = sQ + TILE_H * 2, sK = sO + TILE_H * 2, sV = sK + 2 * TILE_H * 2;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, gq = lane >> 2, t = lane & 3;
    const int q0 = blockIdx.x * BR, h = blockIdx.y;
    const long long img = blockIdx.z;
    const int hid = H * D;
    const long long ld = 3LL * hid;
    const h16* base = qkv + img * n * ld + h * D;
    const h16* obase = out + img * n * hid + h * D;
    const h16* dobase = dout + img * n * hid + h * D;
    const int r0 = q0 + w * 16;
    pdl_wait();
    stage(sQ, base, ld, q0, n);
    stage(sO, dobase, hid, q0, n);
    stage(sK, base + hid, ld, 0, n);
    stage(sV, base + 2 * hid, ld, 0, n);
    cp_commit();
    // delta_i = dO_i . O_i of this warp's 16 rows: lane pair (2r, 2r+1) covers row r, 16 columns each
    float dl;
    {
        const int r = lane >> 1, c0 = (lane & 1) * 16;
        float acc = 0.f;
        if (r0 + r < n) {
            const uint4* op = reinterpret_cast<const uint4*>(obase + (long long)(r0 + r) * hid + c0);
            const uint4* dp = reinterpret_cast<const uint4*>(dobase + (long long)(r0 + r) * hid + c0);
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const uint4 a = __ldg(op + c), d4 = __ldg(dp + c);
                const uint32_t av[4] = {a.x, a.y, a.z, a.w}, dv[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 x = unpack_h2(av[k]), y = unpack_h2(dv[k]);
                    acc = fmaf(x.x, y.x, fmaf(x.y, y.y, acc));
                }
            }
        }
        dl = acc + __shfl_xor_sync(0xffffffffu, acc, 1);
        if ((lane & 1) == 0 && r0 + r < n) delta[(img * n + r0 + r) * H + h] = dl;
    }
    const float e0 = __shfl_sync(0xffffffffu, dl, 2 * gq), e1 = __shfl_sync(0xffffffffu, dl, 2 * (gq + 8));
    const float L0 = r0 + gq < n ? lse[(img * n + r0 + gq) * H + h] * kLog2e : 0.f;
    const float L1 = r0 + gq + 8 < n ? lse[(img * n + r0 + gq + 8) * H + h] * kLog2e : 0.f;
    const int ntiles = (n + BC - 1) / BC;
    uint32_t qa[2][4], da[2][4];
    float dq[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;
#pragma unroll 1
    for (int kt = 0; kt < ntiles; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < ntiles) {
            stage(sK + (buf ^ 1) * TILE_H * 2, base + hid, ld, (kt + 1) * BC, n);
            stage(sV + (buf ^ 1) * TILE_H * 2, base + 2 * hid, ld, (kt + 1) * BC, n);
            cp_commit();
            cp_wait<1>();
        } else {
            cp_wait<0>();
        }
        __syncthreads();
        if (kt == 0) {
            load_a(qa, sQ, w * 16, lane);
            load_a(da, sO, w * 16, lane);
        }
        float s[8][4], dp[8][4];
        gemm_nt(s, qa, sK + buf * TILE_H * 2, lane);    // S = Q K^T
        gemm_nt(dp, da, sV + buf * TILE_H * 2, lane);   // dP = dO V^T
        const bool tail = (kt + 1) * BC > n;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int j = kt * BC + nt * 8 + 2 * t;
            float p0 = ex2_ftz(fmaf(s[nt][0], sl2, -L0)), p1 = ex2_ftz(fmaf(s[nt][1], sl2, -L0));
            float p2 = ex2_ftz(fmaf(s[nt][2], sl2, -L1)), p3 = ex2_ftz(fmaf(s[nt][3], sl2, -L1));
            if (tail) {
                if (j >= n) p0 = p2 = 0.f;
                if (j + 1 >= n) p1 = p3 = 0.f;
            }
            s[nt][0] = p0 * (dp[nt][0] - e0);
            s[nt][1] = p1 * (dp[nt][1] - e0);
            s[nt][2] = p2 * (dp[nt][2] - e1);
            s[nt][3] = p3 * (dp[nt][3] - e1);
        }
        gemm_pv_acc(dq, s, sK + buf * TILE_H * 2, lane);   // dQ += dS K
        __syncthreads();
    }
    const int valid = n - r0;
    if (valid > 0) {
        const float scale = sl2 * (1.f / kLog2e);
        store_rows(dq, dqkv + (img * n + r0) * ld + h * D, ld, valid, scale, scale, lane);
    }
}

// ------------------------------------------------------------------------------------------------
// backward: dK, dV
// ------------------------------------------------------------------------------------------------
// grid (ceil(n / 64), H, NI), 128 threads; every warp owns 16 keys and streams all query tiles.  Two score-sized
// accumulator sets (S^T, dP^T) plus dK, dV: the (128, 3) bound gives 168 registers, without it ptxas caps at 128 and spills.
__global__ void __launch_bounds__(NTH, 3)
mattn_bwd_dkdv_kernel(const h16* __restrict__ qkv, const float* __restrict__ lse, const float* __restrict__ delta,
                      const h16* __restrict__ dout, h16* __restrict__ dqkv, int n, int H, float sl2) {
    pdl_trigger();
    __shared__ __align__(128) h16 smem[TILE_H * 6];   // K | V | Q[2] | dO[2]
    __shared__ float sL[2][BC], sD[2][BC];             // lse * log2 e (+inf past n) and delta of the staged queries
    const uint32_t sK = smem_u32(smem), sV = sK + TILE_H * 2, sQ = sV + TILE_H * 2, sO = sQ + 2 * TILE_H * 2;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, t = lane & 3;
    const int k0 = blockIdx.x * BR, h = blockIdx.y;
    const long long img = blockIdx.z;
    const int hid = H * D;
    const long long ld = 3LL * hid;
    const h16* base = qkv + img * n * ld + h * D;
    const h16* dobase = dout + img * n * hid + h * D;
    const float* lrow = lse + img * n * H + h;
    const float* drow = delta + img * n * H + h;
    pdl_wait();
    stage(sK, base + hid, ld, k0, n);
    stage(sV, base + 2 * hid, ld, k0, n);
    stage(sQ, base, ld, 0, n);
    stage(sO, dobase, hid, 0, n);
    cp_commit();
    if (threadIdx.x < BC) {
        const int i = threadIdx.x;
        sL[0][i] = i < n ? lrow[(long long)i * H] * kLog2e : INFINITY;
        sD[0][i] = i < n ? drow[(long long)i * H] : 0.f;
    }
    const int ntiles = (n + BC - 1) / BC;
    uint32_t ka[2][4], va[2][4];
    float dk[4][4], dv[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f;
        dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = 0.f;
    }
#pragma unroll 1
    for (int qt = 0; qt < ntiles; ++qt) {
        const int buf = qt & 1;
        if (qt + 1 < ntiles) {
            const int i0 = (qt + 1) * BC;
            stage(sQ + (buf ^ 1) * TILE_H * 2, base, ld, i0, n);
            stage(sO + (buf ^ 1) * TILE_H * 2, dobase, hid, i0, n);
            cp_commit();
            if (threadIdx.x < BC) {
                const int i = i0 + threadIdx.x;
                sL[buf ^ 1][threadIdx.x] = i < n ? lrow[(long long)i * H] * kLog2e : INFINITY;
                sD[buf ^ 1][threadIdx.x] = i < n ? drow[(long long)i * H] : 0.f;
            }
            cp_wait<1>();
        } else {
            cp_wait<0>();
        }
        __syncthreads();
        if (qt == 0) {
            load_a(ka, sK, w * 16, lane);
            load_a(va, sV, w * 16, lane);
        }
        float st[8][4], dpt[8][4];
        gemm_nt(st, ka, sQ + buf * TILE_H * 2, lane);    // S^T = K Q^T
        gemm_nt(dpt, va, sO + buf * TILE_H * 2, lane);   // dP^T = V dO^T
        const float* L = sL[buf];
        const float* E = sD[buf];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const int i = nt * 8 + 2 * t;   // query column within the tile
            const float la = L[i], lb = L[i + 1], ea = E[i], eb = E[i + 1];
            const float p0 = ex2_ftz(fmaf(st[nt][0], sl2, -la)), p1 = ex2_ftz(fmaf(st[nt][1], sl2, -lb));
            const float p2 = ex2_ftz(fmaf(st[nt][2], sl2, -la)), p3 = ex2_ftz(fmaf(st[nt][3], sl2, -lb));
            st[nt][0] = p0;
            st[nt][1] = p1;
            st[nt][2] = p2;
            st[nt][3] = p3;
            dpt[nt][0] = p0 * (dpt[nt][0] - ea);
            dpt[nt][1] = p1 * (dpt[nt][1] - eb);
            dpt[nt][2] = p2 * (dpt[nt][2] - ea);
            dpt[nt][3] = p3 * (dpt[nt][3] - eb);
        }
        gemm_pv_acc(dv, st, sO + buf * TILE_H * 2, lane);    // dV += P^T dO
        gemm_pv_acc(dk, dpt, sQ + buf * TILE_H * 2, lane);   // dK += dS^T Q
        __syncthreads();
    }
    const int r0 = k0 + w * 16;
    const int valid = n - r0;
    if (valid > 0) {
        const float scale = sl2 * (1.f / kLog2e);
        h16* g = dqkv + (img * n + r0) * ld + h * D;
        store_rows(dk, g + hid, ld, valid, scale, scale, lane);
        store_rows(dv, g + 2 * hid, ld, valid, 1.f, 1.f, lane);
    }
}

static int check_sizes(int NI, int n, int H, int dim_head) {
    CESM_REQUIRE(dim_head == D, "mid attention kernel needs dim_head == 32 (got %d)", dim_head);
    CESM_REQUIRE(NI >= 1 && NI <= 65535 && n >= 1 && H >= 1 && H <= 65535,
                 "mid attention: need 1 <= NI <= 65535, n >= 1, 1 <= H <= 65535 (NI=%d n=%d H=%d)", NI, n, H);
    return CESM_OK;
}
// fp16 tensors are read / written in 16-byte pieces, fp32 ones element-wise
static bool aligned(const void* p, uintptr_t a) { return p != nullptr && ((uintptr_t)p & (a - 1)) == 0; }

}  // namespace ma
}  // namespace cesm

using namespace cesm;

extern "C" int cesm_mattn_fwd(const void* qkv, void* out, float* lse, int NI, int n, int H, int dim_head, float scale,
                              void* stream) {
    if (int rc = ma::check_sizes(NI, n, H, dim_head)) return rc;
    CESM_REQUIRE(ma::aligned(qkv, 16) && ma::aligned(out, 16) && ma::aligned(lse, 4),
                 "mid attention: qkv / out must be 16-byte aligned, lse 4-byte aligned");
    dim3 grid((unsigned)ceil_div(n, ma::BR), (unsigned)H, (unsigned)NI);
    launch_pdl(ma::mattn_fwd_kernel, grid, ma::NTH, 0, as_stream(stream), (const h16*)qkv, (h16*)out, lse, n, H,
               scale * kLog2e);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_mattn_bwd(const void* qkv, const void* out, const float* lse, const void* dout, void* dqkv,
                              float* delta, int NI, int n, int H, int dim_head, float scale, void* stream) {
    if (int rc = ma::check_sizes(NI, n, H, dim_head)) return rc;
    CESM_REQUIRE(ma::aligned(qkv, 16) && ma::aligned(out, 16) && ma::aligned(dout, 16) && ma::aligned(dqkv, 16) &&
                     ma::aligned(lse, 4) && ma::aligned(delta, 4),
                 "mid attention: qkv / out / dout / dqkv must be 16-byte aligned, lse / delta 4-byte aligned");
    dim3 grid((unsigned)ceil_div(n, ma::BR), (unsigned)H, (unsigned)NI);
    cudaStream_t st = as_stream(stream);
    launch_pdl(ma::mattn_bwd_dq_kernel, grid, ma::NTH, 0, st, (const h16*)qkv, (const h16*)out, lse, (const h16*)dout,
               (h16*)dqkv, delta, n, H, scale * kLog2e);
    CESM_CHECK_LAUNCH();
    launch_pdl(ma::mattn_bwd_dkdv_kernel, grid, ma::NTH, 0, st, (const h16*)qkv, lse, (const float*)delta,
               (const h16*)dout, (h16*)dqkv, n, H, scale * kLog2e);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}
