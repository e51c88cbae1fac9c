// Spatial linear attention core (video_net.py:338-344) for sm_100a, fp16 in / fp32 accumulate.
//
// Per image (one frame of one sample) and head, with n pixels and d = e = 32:
//     qs = scale * softmax_d(q)         (over the 32 features of a pixel)
//     kh = softmax_n(k)                 (over the n pixels, per feature)
//     ctx[d][e] = sum_p kh[p][d] v[p][e]
//     out[p][e] = sum_d ctx[d][e] qs[p][d]
//
// The op moves ~1 KB per pixel and does ~4 kFLOP per pixel per head: it is HBM-bound as long as
// the two small contractions run on tensor cores, so they are warp-level mma.sync m16n8k16 tiles
// (one warp per head; operands are exponentiated / normalised in registers on their way from
// global memory to the fragments) and nothing but q, k, v, out ever touches HBM: the softmaxed
// copies the reference materialises are recomputed where needed, forward and backward.
//
//   forward : colmax(k) -> context (exp(k-max) & v -> unnormalised ctx, Z) -> finalize (ctx /= Z)
//             -> apply (softmax(q), ctx -> out)
//   backward: context (qs & dout -> dctx) -> delta = rowsum(ctx * dctx) -> bwd_apply (dq, dk, dv)
//
// Workspace `ws` (fp32, per image): [HD] encoded column max | [HD] Z | [H][32][32] ctx.
#include "api_common.h"
#include "common.cuh"

namespace cesm {

static constexpr int LD = 32;        // head dim
static constexpr int SPITCH = 40;    // fp16 elements per staged row (80 B: conflict-free ldmatrix)

__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr));
}
__device__ __forceinline__ void mma_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
        "{%0, %1, %2, %3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// order-preserving float <-> uint encoding, so that column maxima can use atomicMax on a zeroed buffer
__device__ __forceinline__ uint32_t enc_ordered(float f) {
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float dec_ordered(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
    float2 a = unpack_h2(u.x), b = unpack_h2(u.y), c = unpack_h2(u.z), d = unpack_h2(u.w);
    f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    uint4 u;
    u.x = pack_h2(f[0], f[1]); u.y = pack_h2(f[2], f[3]);
    u.z = pack_h2(f[4], f[5]); u.w = pack_h2(f[6], f[7]);
    return u;
}
__device__ __forceinline__ float quad_max(float v) {
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
    return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// cp.async (LDGSTS) ring: every global byte of these kernels goes global -> shared without passing
// through registers, several 16-pixel steps ahead of its use, so a warp keeps (stages-1) steps of
// loads in flight whatever its register budget.  Buffers are warp-private: only __syncwarp is needed.
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
static constexpr int kTileBytes = 16 * SPITCH * 2;  // one staged 16-pixel x 32-channel fp16 tile

struct LaWs {  // views into the per-image workspace
    uint32_t* kmax;
    float* z;
    float* ctx;
};
__device__ __forceinline__ LaWs la_ws(float* ws, int ni, int HD, int H) {
    float* base = ws + (size_t)ni * (2 * HD + (size_t)H * LD * LD);
    return {reinterpret_cast<uint32_t*>(base), base + HD, base + 2 * HD};
}

// ------------------------------------------------------------------------------------------------
// column max of k over the pixels of each image: thread = 8 channels (16 B), rows strided over the block
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
la_colmax_kernel(const h16* __restrict__ qkv, float* __restrict__ ws, int n, int H, int rows_per_block) {
    pdl_trigger();
    pdl_wait();
    const int HD = H * LD, cpr = HD / 8;
    const int ni = blockIdx.y;
    const int chunk = threadIdx.x % cpr, rl = threadIdx.x / cpr, nrl = blockDim.x / cpr;
    const int p0 = blockIdx.x * rows_per_block, p1 = min(n, p0 + rows_per_block);
    float m[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) m[i] = -INFINITY;
    if (rl < nrl) {
        const h16* base = qkv + ((size_t)ni * n) * (3 * HD) + HD + chunk * 8;
        for (int p = p0 + rl; p < p1; p += nrl) {
            float f[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(base + (size_t)p * 3 * HD)), f);
#pragma unroll
            for (int i = 0; i < 8; ++i) m[i] = fmaxf(m[i], f[i]);
        }
    }
    __shared__ float red[256][9];
#pragma unroll
    for (int i = 0; i < 8; ++i) red[threadIdx.x][i] = m[i];
    __syncthreads();
    if ((int)threadIdx.x < HD) {
        const int c = threadIdx.x, ch = c / 8, i = c % 8;
        float v = -INFINITY;
        for (int r = 0; r < nrl; ++r) v = fmaxf(v, red[r * cpr + ch][i]);
        if (v > -INFINITY) atomicMax(la_ws(ws, ni, HD, H).kmax + c, enc_ordered(v));
    }
}

// ------------------------------------------------------------------------------------------------
// context: acc[d][e] += sum_p A[p][d] * B[p][e] over a chunk of pixels; warp = head.
//   MODE 0 (forward) : A = exp(k - colmax) (also accumulates Z[d] = sum_p A[p][d]),  B = v
//   MODE 1 (backward): A = scale * softmax_d(q),                                     B = dout
// Each 16-pixel step is staged through a warp-private smem tile and read back with
// ldmatrix.trans, which yields the pixel-contracted (MN-major) fragments.
// ------------------------------------------------------------------------------------------------
static constexpr int CTX_STAGES = 3;
template <int MODE>
__global__ void __launch_bounds__(256)
la_context_kernel(const h16* __restrict__ qkv, const h16* __restrict__ dout,
                  float* __restrict__ ws, float* __restrict__ acc_out /* MODE 1: dctx [NI][H][32][32] */, int n, int H,
                  int chunk, float scale) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) uint8_t la_smem[];
    const int HD = H * LD, ld = 3 * HD;
    const int ni = blockIdx.y, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = lane >> 2, c = lane & 3;
    // per warp: [CTX_STAGES][2] raw tiles (A source, B) filled by cp.async (+ one transformed A tile in
    // MODE 1); operands go from there into fragments with ldmatrix.trans
    constexpr int kWarpTiles = 2 * CTX_STAGES + (MODE == 1 ? 1 : 0);
    uint8_t* wbase = la_smem + (size_t)w * kWarpTiles * kTileBytes;
    h16* sA = reinterpret_cast<h16*>(wbase + 2 * CTX_STAGES * kTileBytes);
    const uint32_t sA_addr = smem_u32(sA);
    const uint32_t ring_addr = smem_u32(wbase);
    const LaWs W = la_ws(ws, ni, HD, H);

    // MODE 0 works in mma-fragment layout: this lane's A registers hold channels d = 16 mt + r + 8 hh
    // (mt, hh in {0,1}) of pixel pairs, so it needs 4 column maxima and keeps 4 partial Z sums
    float cmf[2][2], zf[2][2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            cmf[mt][hh] = (MODE == 0) ? dec_ordered(W.kmax[w * LD + 16 * mt + r + 8 * hh]) * kLog2e : 0.f;
            zf[mt][hh] = 0.f;
        }
    float acc[2][4][4];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[a][b][k] = 0.f;

    const size_t img_row0 = (size_t)ni * n;
    const h16* a_base = qkv + img_row0 * ld + (MODE == 0 ? HD : 0) + w * LD + c * 8;
    const h16* b_base = (MODE == 0) ? qkv + img_row0 * ld + 2 * HD + w * LD + c * 8
                                              : dout + img_row0 * HD + w * LD + c * 8;
    const int b_ld = (MODE == 0) ? ld : HD;
    const int p0 = blockIdx.x * chunk, p1 = min(n, p0 + chunk);

    // ldmatrix lane addresses (fixed): A m-tile mt, B n-tile pair jp
    const int mi = lane >> 3, rr = lane & 7;
    uint32_t a_off[2], b_off[2];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) a_off[mt] = (((mi >> 1) * 8 + rr) * SPITCH + 16 * mt + (mi & 1) * 8) * 2;
#pragma unroll
    for (int jp = 0; jp < 2; ++jp) b_off[jp] = (((mi & 1) * 8 + rr) * SPITCH + 8 * (jp * 2 + (mi >> 1))) * 2;

    auto issue_loads = [&](int step) {  // rows beyond the chunk are clamped (finite data) and masked later
        const int pp = p0 + 16 * step;
        const uint32_t st = ring_addr + (step % CTX_STAGES) * 2 * kTileBytes;
        if (pp < p1) {
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                const int row = min(pp + r + 8 * h2, p1 - 1);
                const uint32_t off = ((r + 8 * h2) * SPITCH + c * 8) * 2;
                cp_async16(st + off, a_base + (size_t)row * ld);
                cp_async16(st + kTileBytes + off, b_base + (size_t)row * b_ld);
            }
        }
        cp_async_commit();
    };
    const int nsteps = (p1 - p0 + 15) / 16;
#pragma unroll
    for (int s0 = 0; s0 < CTX_STAGES - 1; ++s0) issue_loads(s0);
    for (int step = 0; step < nsteps; ++step) {
        const int p = p0 + 16 * step;
        issue_loads(step + CTX_STAGES - 1);      // refills the stage consumed in the previous iteration
        cp_async_wait<CTX_STAGES - 1>();         // this step's tiles have landed
        __syncwarp();
        const uint32_t st = ring_addr + (step % CTX_STAGES) * 2 * kTileBytes;
        const uint32_t sB_addr = st + kTileBytes;
        uint32_t af[2][4], bf[2][4];
        if (MODE == 0) {
            // exp(k - max) applied in fragment layout: raw k goes ring -> ldmatrix.trans -> registers, with no
            // second trip through shared memory.  af[mt][i]: channel 16 mt + r + 8 (i & 1), pixels
            // p + 2c + 8 (i >> 1) + {0, 1}
            ldmatrix_x4_trans(af[0], st + a_off[0]);
            ldmatrix_x4_trans(af[1], st + a_off[1]);
            const bool full = p + 16 <= p1;
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float2 x = unpack_h2(af[mt][i]);
                    float e0 = exp_sub(x.x, cmf[mt][i & 1]), e1 = exp_sub(x.y, cmf[mt][i & 1]);
                    if (!full) {
                        const int px = p + 2 * c + 8 * (i >> 1);
                        e0 = px < p1 ? e0 : 0.f;
                        e1 = px + 1 < p1 ? e1 : 0.f;
                    }
                    zf[mt][i & 1] += e0 + e1;
                    af[mt][i] = pack_h2(e0, e1);
                }
        } else {
            // scale * softmax_d(q): rows are normalised in the row layout (quad shuffles), staged through a
            // warp-private tile and read back transposed.  (Doing this in fragment layout like MODE 0 needs
            // 24 cross-quad shuffles per step and measured slower: 120 vs 88 us at 192x288.)
            uint4 ua[2];
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                const uint32_t off = ((r + 8 * h2) * SPITCH + c * 8) * 2;
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(ua[h2].x), "=r"(ua[h2].y), "=r"(ua[h2].z), "=r"(ua[h2].w)
                             : "r"(st + off));
            }
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                const bool valid = (p + r + 8 * h2) < p1;
                float f[8];
                unpack8(ua[h2], f);
                float m = f[0];
#pragma unroll
                for (int i = 1; i < 8; ++i) m = fmaxf(m, f[i]);
                m = quad_max(m) * kLog2e;
                float sum = 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    f[i] = exp_sub(f[i], m);
                    sum += f[i];
                }
                sum = quad_sum(sum);
                const float inv = valid ? scale / sum : 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] *= inv;
                *reinterpret_cast<uint4*>(sA + (r + 8 * h2) * SPITCH + c * 8) = pack8(f);
            }
            __syncwarp();
            ldmatrix_x4_trans(af[0], sA_addr + a_off[0]);
            ldmatrix_x4_trans(af[1], sA_addr + a_off[1]);
        }
        ldmatrix_x4_trans(bf[0], sB_addr + b_off[0]);
        ldmatrix_x4_trans(bf[1], sB_addr + b_off[1]);
        __syncwarp();
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int j = 0; j < 4; ++j) mma_16816(acc[mt][j], af[mt], bf[j >> 1][(j & 1) * 2], bf[j >> 1][(j & 1) * 2 + 1]);
    }

    // ---- reduce into global (fp32 atomics; a few dozen blocks per image) ----
    float* dst = (MODE == 0 ? W.ctx : acc_out + (size_t)ni * H * LD * LD) + (size_t)w * LD * LD;
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int d0 = 16 * mt + g, e0 = 8 * j + 2 * t;
            atomicAdd(dst + d0 * LD + e0, acc[mt][j][0]);
            atomicAdd(dst + d0 * LD + e0 + 1, acc[mt][j][1]);
            atomicAdd(dst + (d0 + 8) * LD + e0, acc[mt][j][2]);
            atomicAdd(dst + (d0 + 8) * LD + e0 + 1, acc[mt][j][3]);
        }
    if (MODE == 0) {
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const float z = quad_sum(zf[mt][hh]);  // the 4 lanes of a quad hold different pixels of channel d
                if (c == 0) atomicAdd(W.z + w * LD + 16 * mt + r + 8 * hh, z);
            }
    }
}

// ctx[d][e] /= Z[d]  (forward) -- one thread per element
__global__ void la_finalize_kernel(float* __restrict__ ws, int H, int NI) {
    pdl_trigger();
    pdl_wait();
    const int HD = H * LD;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int per = H * LD * LD;
    if (idx >= NI * per) return;
    const int ni = idx / per, x = idx % per;
    const LaWs W = la_ws(ws, ni, HD, H);
    W.ctx[x] = W.ctx[x] / W.z[x / LD];  // x / LD == h*32 + d
}

// delta[ni][h*32+d] = sum_e ctx[d][e] * dctx[d][e]
__global__ void la_delta_kernel(float* __restrict__ ws, const float* __restrict__ dctx, float* __restrict__ delta,
                                int H, int NI) {
    pdl_trigger();
    pdl_wait();
    const int HD = H * LD;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // ni*HD + h*32 + d
    if (idx >= NI * HD) return;
    const int ni = idx / HD, hd = idx % HD;
    const LaWs W = la_ws(ws, ni, HD, H);
    const float* dc = dctx + ((size_t)ni * HD + hd) * LD;
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < LD; ++e) s = fmaf(W.ctx[hd * LD + e], dc[e], s);
    delta[idx] = s;
}

// ------------------------------------------------------------------------------------------------
// The apply kernels keep everything in registers.  Lane (g = lane >> 2, t = lane & 3) owns the 8
// channels 8t..8t+7 (one 16-byte global access) of pixel rows g and g+8 of a 16-pixel step.  With the
// channel permutation  phi(8j + 2t + b) = 8t + 2j + b  (logical mma column -> physical channel) that
// row layout IS the mma.m16n8k16 C-fragment layout (n-tile j <-> 32-bit word j of the lane's uint4)
// and, k-step ks taking words 2ks and 2ks+1, also the A-fragment layout.  Only the small 32x32
// B operands (ctx, dctx) need the permutation, applied once per block when their fragments are read
// from global memory; the contraction index order is irrelevant to a sum.  So: 16-byte loads ->
// softmax / exp in registers -> mma -> 16-byte stores, no shared memory, no warp syncs.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int phi32(int L) { return ((L >> 1) & 3) * 8 + (L >> 3) * 2 + (L & 1); }

// B fragments of a 32x32 fp32 matrix M (row-major) for C = A * Bm, Bm[k][n] = TRANS ? M[n][k] : M[k][n],
// with both k and n taken through phi32
template <bool TRANS>
__device__ __forceinline__ void load_bfrag32(const float* __restrict__ M, int g, int t, uint32_t (&b)[2][4][2]) {
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int nn = phi32(8 * j + g);
#pragma unroll
            for (int hi = 0; hi < 2; ++hi) {
                const int k0 = phi32(16 * ks + 8 * hi + 2 * t), k1 = k0 + 1;  // phi keeps (even, odd) pairs adjacent
                b[ks][j][hi] = TRANS ? pack_h2(M[nn * LD + k0], M[nn * LD + k1])
                                     : pack_h2(M[k0 * LD + nn], M[k1 * LD + nn]);
            }
        }
}
// A fragments of a 16 x 32 tile whose rows g / g+8 this lane holds as packed fp16 (lo / hi)
__device__ __forceinline__ void rows_to_afrag(const uint4& lo, const uint4& hi, uint32_t (&a)[2][4]) {
    a[0][0] = lo.x; a[0][1] = hi.x; a[0][2] = lo.y; a[0][3] = hi.y;
    a[1][0] = lo.z; a[1][1] = hi.z; a[1][2] = lo.w; a[1][3] = hi.w;
}
// C (16x32 as 4 n-tiles) = A (16x32) * B; c[j][0..1] = row g, words j; c[j][2..3] = row g+8
__device__ __forceinline__ void frag_gemm(const uint32_t (&a)[2][4], const uint32_t (&b)[2][4][2], float (&c)[4][4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        c[j][0] = c[j][1] = c[j][2] = c[j][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) mma_16816(c[j], a[ks], b[ks][j][0], b[ks][j][1]);
    }
}
__device__ __forceinline__ void c_to_rows(const float (&c)[4][4], float (&o)[2][8]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        o[0][2 * j] = c[j][0]; o[0][2 * j + 1] = c[j][1];
        o[1][2 * j] = c[j][2]; o[1][2 * j + 1] = c[j][3];
    }
}
// softmax over the 32 channels of a row held by a quad (8 per lane)
__device__ __forceinline__ void row_softmax(float (&f)[8]) {
    float m = f[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) m = fmaxf(m, f[i]);
    m = quad_max(m) * kLog2e;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        f[i] = exp_sub(f[i], m);
        s += f[i];
    }
    const float inv = 1.f / quad_sum(s);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] *= inv;
}

// ------------------------------------------------------------------------------------------------
// apply (forward): out[p][e] = sum_d qs[p][d] ctx[d][e]; warp = head; APPLY_MT 16-pixel tiles per
// step, the next step's loads issued before this step's math
// ------------------------------------------------------------------------------------------------
static constexpr int APPLY_MT = 2;
static constexpr int RING_STAGES = 3;
__device__ __forceinline__ uint4 lds16(uint32_t addr) {
    uint4 u;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(addr));
    return u;
}
__global__ void __launch_bounds__(256, 3)
la_apply_kernel(const h16* __restrict__ qkv, float* __restrict__ ws, h16* __restrict__ out, int n,
                int H, int chunk, float scale) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) uint8_t la_smem[];
    const int HD = H * LD, ld = 3 * HD;
    const int ni = blockIdx.y, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = lane >> 2, c = lane & 3;
    const LaWs W = la_ws(ws, ni, HD, H);
    uint32_t bctx[2][4][2];
    load_bfrag32<false>(W.ctx + (size_t)w * LD * LD, r, c, bctx);
    const size_t row0 = (size_t)ni * n;
    const int p1 = min(n, (int)(blockIdx.x + 1) * chunk);
    const h16* qbase = qkv + row0 * ld + w * LD + c * 8;
    h16* obase = out + row0 * HD + w * LD + c * 8;
    // thread-private cp.async ring: [stage][vector][thread] x 16 B; the loads of step i+2 are in flight
    // while step i is computed, and a lane only reads back what it copied itself (no barriers)
    const uint32_t ring = smem_u32(la_smem) + threadIdx.x * 16u;
    constexpr uint32_t kVec = 256 * 16, kStage = APPLY_MT * 2 * kVec;
    auto issue_loads = [&](int pp, int stage) {
        if (pp < p1) {
#pragma unroll
            for (int mt = 0; mt < APPLY_MT; ++mt)
#pragma unroll
                for (int h2 = 0; h2 < 2; ++h2) {
                    const int row = min(pp + 16 * mt + r + 8 * h2, p1 - 1);
                    cp_async16(ring + stage * kStage + (mt * 2 + h2) * kVec, qbase + (size_t)row * ld);
                }
        }
        cp_async_commit();
    };
    const int pstart = blockIdx.x * chunk;
#pragma unroll
    for (int s0 = 0; s0 < RING_STAGES - 1; ++s0) issue_loads(pstart + s0 * 16 * APPLY_MT, s0);
    int stage = 0;
    for (int p = pstart; p < p1; p += 16 * APPLY_MT) {
        {
            int ns = stage + RING_STAGES - 1;
            if (ns >= RING_STAGES) ns -= RING_STAGES;
            issue_loads(p + (RING_STAGES - 1) * 16 * APPLY_MT, ns);
        }
        cp_async_wait<RING_STAGES - 1>();
        uint4 cq[APPLY_MT][2];
#pragma unroll
        for (int mt = 0; mt < APPLY_MT; ++mt)
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) cq[mt][h2] = lds16(ring + stage * kStage + (mt * 2 + h2) * kVec);
        if (++stage == RING_STAGES) stage = 0;
#pragma unroll
        for (int mt = 0; mt < APPLY_MT; ++mt) {
            uint4 pk[2];
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                float f[8];
                unpack8(cq[mt][h2], f);
                row_softmax(f);
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] *= scale;
                pk[h2] = pack8(f);
            }
            uint32_t a[2][4];
            rows_to_afrag(pk[0], pk[1], a);
            float cfr[4][4], o[2][8];
            frag_gemm(a, bctx, cfr);
            c_to_rows(cfr, o);
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                const int row = p + 16 * mt + r + 8 * h2;
                if (row < p1) *reinterpret_cast<uint4*>(obase + (size_t)row * HD) = pack8(o[h2]);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// backward apply: per pixel row
//   dqh = dout ctx^T ; dq = sm (scale dqh - sum_j sm_j scale dqh_j)
//   dkh = v dctx^T   ; dk = kh (dkh - delta) , kh = exp(k - max) / Z
//   dv  = kh dctx
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 2)
la_bwd_apply_kernel(const h16* __restrict__ qkv, const h16* __restrict__ dout,
                    float* __restrict__ ws, const float* __restrict__ dctx, const float* __restrict__ delta,
                    h16* __restrict__ dqkv, int n, int H, int chunk, float scale) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) uint8_t la_smem[];
    const int HD = H * LD, ld = 3 * HD;
    const int ni = blockIdx.y, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = lane >> 2, c = lane & 3;
    const LaWs W = la_ws(ws, ni, HD, H);
    const float* dcx = dctx + ((size_t)ni * H + w) * LD * LD;
    uint32_t b_ctxT[2][4][2], b_dctxT[2][4][2], b_dctx[2][4][2];
    load_bfrag32<true>(W.ctx + (size_t)w * LD * LD, r, c, b_ctxT);
    load_bfrag32<true>(dcx, r, c, b_dctxT);
    load_bfrag32<false>(dcx, r, c, b_dctx);
    // per-channel constants live in shared memory (read back as two float4 per use: registers are
    // what bounds this kernel's occupancy).  kh = exp(k - max) / Z = exp(k - (max + log Z))
    __shared__ __align__(16) float s_kml[8 * LD], s_del[8 * LD];
    {
        const int col = threadIdx.x;  // blockDim.x == HD
        s_kml[col] = (dec_ordered(W.kmax[col]) + __logf(W.z[col])) * kLog2e;  // pre-scaled for exp_sub
        s_del[col] = delta[(size_t)ni * HD + col];
    }
    __syncthreads();
    const float* kml = s_kml + w * LD + c * 8;
    const float* del = s_del + w * LD + c * 8;
    const size_t row0 = (size_t)ni * n;
    const int p1 = min(n, (int)(blockIdx.x + 1) * chunk);
    const h16* xbase = qkv + row0 * ld + w * LD + c * 8;
    const h16* dbase = dout + row0 * HD + w * LD + c * 8;
    h16* gbase = dqkv + row0 * ld + w * LD + c * 8;
    // thread-private cp.async ring (see la_apply_kernel): 8 x 16 B per lane and step, two steps ahead
    const uint32_t ring = smem_u32(la_smem) + threadIdx.x * 16u;
    constexpr uint32_t kVec = 256 * 16, kStage = 8 * kVec;
    auto issue_loads = [&](int pp, int stage) {
        if (pp < p1) {
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                const int row = min(pp + r + 8 * h2, p1 - 1);
                const h16* xg = xbase + (size_t)row * ld;
                const uint32_t st = ring + stage * kStage + h2 * 4 * kVec;
                cp_async16(st, dbase + (size_t)row * HD);
                cp_async16(st + kVec, xg);
                cp_async16(st + 2 * kVec, xg + HD);
                cp_async16(st + 3 * kVec, xg + 2 * HD);
            }
        }
        cp_async_commit();
    };
    const int pstart = blockIdx.x * chunk;
#pragma unroll
    for (int s0 = 0; s0 < RING_STAGES - 1; ++s0) issue_loads(pstart + s0 * 16, s0);
    int stage = 0;
    for (int p = pstart; p < p1; p += 16) {
        {
            int ns = stage + RING_STAGES - 1;
            if (ns >= RING_STAGES) ns -= RING_STAGES;
            issue_loads(p + (RING_STAGES - 1) * 16, ns);
        }
        cp_async_wait<RING_STAGES - 1>();
        float sm[2][8];
        uint4 ud[2], uv[2], uk[2];
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
            const uint32_t st = ring + stage * kStage + h2 * 4 * kVec;
            ud[h2] = lds16(st);
            unpack8(lds16(st + kVec), sm[h2]);
            uk[h2] = lds16(st + 2 * kVec);
            uv[h2] = lds16(st + 3 * kVec);
        }
        if (++stage == RING_STAGES) stage = 0;
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) row_softmax(sm[h2]);
        uint32_t a[2][4];
        float cfr[4][4], o[2][8];
        // ---- dq ----
        rows_to_afrag(ud[0], ud[1], a);
        frag_gemm(a, b_ctxT, cfr);  // dqh
        c_to_rows(cfr, o);
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
            float dot = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) dot = fmaf(sm[h2][i], o[h2][i], dot);
            dot = quad_sum(dot);
#pragma unroll
            for (int i = 0; i < 8; ++i) o[h2][i] = sm[h2][i] * scale * (o[h2][i] - dot);
            const int row = p + r + 8 * h2;
            if (row < p1) *reinterpret_cast<uint4*>(gbase + (size_t)row * ld) = pack8(o[h2]);
        }
        // ---- dk ----
        rows_to_afrag(uv[0], uv[1], a);
        frag_gemm(a, b_dctxT, cfr);  // dkh
        c_to_rows(cfr, o);
        uint4 ukh[2];
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
            float kh[8], km[8], dl[8];
            unpack8(uk[h2], kh);
            *reinterpret_cast<float4*>(km) = *reinterpret_cast<const float4*>(kml);
            *reinterpret_cast<float4*>(km + 4) = *reinterpret_cast<const float4*>(kml + 4);
            *reinterpret_cast<float4*>(dl) = *reinterpret_cast<const float4*>(del);
            *reinterpret_cast<float4*>(dl + 4) = *reinterpret_cast<const float4*>(del + 4);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                kh[i] = exp_sub(kh[i], km[i]);
                o[h2][i] = kh[i] * (o[h2][i] - dl[i]);
            }
            ukh[h2] = pack8(kh);
            const int row = p + r + 8 * h2;
            if (row < p1) *reinterpret_cast<uint4*>(gbase + (size_t)row * ld + HD) = pack8(o[h2]);
        }
        // ---- dv ----
        rows_to_afrag(ukh[0], ukh[1], a);
        frag_gemm(a, b_dctx, cfr);
        c_to_rows(cfr, o);
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
            const int row = p + r + 8 * h2;
            if (row < p1) *reinterpret_cast<uint4*>(gbase + (size_t)row * ld + 2 * HD) = pack8(o[h2]);
        }
    }
}

}  // namespace cesm

using namespace cesm;

static int la_chunk(int n, int NI) {
    // more blocks than SMs (>= ~4 per SM: 8 measured 6 % slower forward at 192x288, 2 measured 13 % slower)
    // so that the tail wave is a small fraction, while a block still amortises its per-head fragment
    // preloads and atomics over >= 128 pixels
    int chunk = 2048;
    while (chunk > 128 && (long long)NI * ((n + chunk - 1) / chunk) < 148 * 4) chunk >>= 1;
    return chunk;
}

static size_t la_context_smem(int H, int mode) {
    // per warp (= head): CTX_STAGES x {A source, B} cp.async tiles
    static bool cfg = false;
    if (!cfg) {
        cudaFuncSetAttribute(la_context_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * 2 * CTX_STAGES * kTileBytes);
        cudaFuncSetAttribute(la_context_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * (2 * CTX_STAGES + 1) * kTileBytes);
        cfg = true;
    }
    return (size_t)H * (2 * CTX_STAGES + (mode == 1 ? 1 : 0)) * kTileBytes;
}

extern "C" size_t cesm_linattn_ws_floats(int NI, int H) { return (size_t)NI * (2 * H * LD + (size_t)H * LD * LD); }

extern "C" int cesm_linattn_fwd(const void* qkv, float* ws, void* out, int NI, int n, int H, int dim_head, float scale,
                                void* stream) {
    CESM_REQUIRE(dim_head == LD, "linear attention kernel needs dim_head == 32 (got %d)", dim_head);
    CESM_REQUIRE(H >= 1 && H <= 8, "linear attention kernel supports 1..8 heads (got %d)", H);
    cudaStream_t st = as_stream(stream);
    const int HD = H * LD;
    CESM_ZERO_SCRATCH(ws, sizeof(float) * cesm_linattn_ws_floats(NI, H), st);
    const int chunk = la_chunk(n, NI);
    dim3 grid(ceil_div(n, chunk), NI);
    launch_pdl(la_colmax_kernel, grid, 256, 0, st, (const h16*)qkv, ws, n, H, chunk);
    CESM_CHECK_LAUNCH();
    const size_t sh = la_context_smem(H, 0);
    launch_pdl(la_context_kernel<0>, grid, 32 * H, sh, st, (const h16*)qkv, nullptr, ws, nullptr, n, H, chunk, scale);
    CESM_CHECK_LAUNCH();
    launch_pdl(la_finalize_kernel, ceil_div(NI * H * LD * LD, 256), 256, 0, st, ws, H, NI);
    CESM_CHECK_LAUNCH();
    const size_t sh_apply = (size_t)RING_STAGES * APPLY_MT * 2 * 256 * 16;  // 48 KB
    launch_pdl(la_apply_kernel, grid, 32 * H, sh_apply, st, (const h16*)qkv, ws, (h16*)out, n, H, chunk,
                                                    scale);
    CESM_CHECK_LAUNCH();
    (void)HD;
    return CESM_OK;
}

// scratch: fp32 [NI][H][32][32] (dctx) + [NI][H*32] (delta)
extern "C" int cesm_linattn_bwd(const void* qkv, float* ws, const void* dout, float* scratch, void* dqkv, int NI, int n,
                                int H, int dim_head, float scale, void* stream) {
    CESM_REQUIRE(dim_head == LD, "linear attention kernel needs dim_head == 32 (got %d)", dim_head);
    CESM_REQUIRE(H >= 1 && H <= 8, "linear attention kernel supports 1..8 heads (got %d)", H);
    cudaStream_t st = as_stream(stream);
    float* dctx = scratch;
    float* delta = scratch + (size_t)NI * H * LD * LD;
    CESM_ZERO_SCRATCH(dctx, sizeof(float) * NI * H * LD * LD, st);
    const int chunk = la_chunk(n, NI);
    dim3 grid(ceil_div(n, chunk), NI);
    const size_t sh = la_context_smem(H, 1);
    launch_pdl(la_context_kernel<1>, grid, 32 * H, sh, st, (const h16*)qkv, (const h16*)dout, ws, dctx, n, H,
                                                   chunk, scale);
    CESM_CHECK_LAUNCH();
    launch_pdl(la_delta_kernel, ceil_div(NI * H * LD, 128), 128, 0, st, ws, dctx, delta, H, NI);
    CESM_CHECK_LAUNCH();
    const size_t sh_bwd = (size_t)RING_STAGES * 8 * 256 * 16;  // 96 KB
    static bool bwd_cfg = false;
    if (!bwd_cfg) {
        CESM_CHECK_CUDA(cudaFuncSetAttribute(la_bwd_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh_bwd));
        bwd_cfg = true;
    }
    launch_pdl(la_bwd_apply_kernel, grid, 32 * H, sh_bwd, st, (const h16*)qkv, (const h16*)dout, ws, dctx, delta,
                                                 (h16*)dqkv, n, H, chunk, scale);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}
