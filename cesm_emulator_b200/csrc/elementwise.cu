// Small and bandwidth-bound kernels around the tensor-core path:
//   weight re-layout (fp32 parameter -> fp16 GEMM operand, and fp32 GEMM-layout gradient -> parameter)
//   7x7 input conv with fused concat / frame broadcast (video_net.py:808-815, model.py:110-121)
//   1x1x1 output conv fused with centre-frame selection (video_net.py:763, model.py:129-130)
//   time embedding + small fp32 linears (video_net.py:101-113, 651-656, 238-241)
//   DDPM q_sample / MSE / p_sample update (model.py:168-208), strided DDIM and DPM-Solver++(2M) updates
//   column sums (bias gradients)
#include "api_common.h"
#include "common.cuh"

namespace cesm {

struct TapOffsets {
    int32_t off[CESM_MAX_TAPS];
};

// dst[o][t][i] (fp16) = src[o*so + i*si + off[t]] (fp32)
__global__ void pack_weight_kernel(const float* __restrict__ src, h16* __restrict__ dst, int O, int T, int I,
                                   long long so, long long si, TapOffsets taps) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)O * T * I) return;
    const int i = idx % I;
    const int t = (idx / I) % T;
    const int o = idx / ((long long)I * T);
    dst[idx] = __float2half_rn(src[o * so + i * si + taps.off[t]]);
}
// dst[o*so + i*si + off[t]] (+)= src[o][t][i]
__global__ void unpack_wgrad_kernel(const float* __restrict__ src, float* __restrict__ dst, int O, int T, int I,
                                    long long so, long long si, TapOffsets taps, int accumulate) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)O * T * I) return;
    const int i = idx % I;
    const int t = (idx / I) % T;
    const int o = idx / ((long long)I * T);
    float* d = dst + o * so + i * si + taps.off[t];
    *d = accumulate ? (*d + src[idx]) : src[idx];
}

// out[c] = sum_rows x[row][c]; block handles a strip of rows, thread owns 8 channels
__global__ void __launch_bounds__(256)
colsum_kernel(const h16* __restrict__ x, float* __restrict__ out, long long M, int C) {
    pdl_trigger();
    pdl_wait();
    const int vec = C >> 3;
    const int slot = threadIdx.x % vec;
    const int rows_per_iter = 256 / vec;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    for (long long r = (long long)blockIdx.x * rows_per_iter + threadIdx.x / vec; r < M;
         r += (long long)gridDim.x * rows_per_iter) {
        uint4 u = *reinterpret_cast<const uint4*>(x + r * C + slot * 8);
        float2 a = unpack_h2(u.x), b = unpack_h2(u.y), c = unpack_h2(u.z), d = unpack_h2(u.w);
        acc[0] += a.x; acc[1] += a.y; acc[2] += b.x; acc[3] += b.y; acc[4] += c.x; acc[5] += c.y; acc[6] += d.x; acc[7] += d.y;
    }
    __shared__ float red[256][9];
#pragma unroll
    for (int i = 0; i < 8; ++i) red[threadIdx.x][i] = acc[i];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
        float s = 0.f;
        for (int t = c >> 3; t < 256; t += vec) s += red[t][c & 7];
        atomicAdd(&out[c], s);
    }
}

// ------------------------------------------------------------------------------------------------
// Input conv on the tensor cores: im2col of the two fp32 input planes into fp16 patch rows
//   [hi(x) 2*KS*KS | lo(x) 2*KS*KS | 1 | 1 | 0 ...]  (KPAD columns),  hi = fp16(x), lo = fp16(x - hi),
// so that the tcgen05 implicit GEMM (1 tap, K = KPAD) against [w | w | bias_hi | bias_lo | 0] reproduces the
// fp32-input convolution to ~2^-17 in the inputs (the weights are fp16 like every other layer's) and its
// weight-gradient kernel yields dW (sum of the hi and lo column blocks) and db (the ones column) from
// the same patch matrix.  A block stages a 16x16 pixel tile's halo once; a warp then writes one pixel's
// 2*KPAD bytes per trip, each lane a fixed 8-column chunk whose shared-memory offsets it computed once.
// keep (optional, [B]): batch element b reads its condition plane as zeros where keep[b] == 0 (classifier-free
// guidance's condition dropout), so the forward GEMM and the weight gradient, which both read these patches, see the
// null condition without a masked copy of it.
// ------------------------------------------------------------------------------------------------
template <int KS, int KPAD>
__global__ void __launch_bounds__(256)
input_patches_kernel(const float* __restrict__ in0, const float* __restrict__ in1, int f0, int f1,
                     const float* __restrict__ keep, h16* __restrict__ out, int F, int H, int W) {
    pdl_trigger();
    pdl_wait();
    constexpr int T = 16, PAD = KS / 2, PW = T + KS - 1, NT = 2 * KS * KS;
    static_assert(KPAD % 8 == 0 && KPAD >= 2 * NT + 2 && KPAD / 8 == 32, "one 8-column chunk per lane");
    __shared__ float sv[2][2][PW][PW];  // [hi | lo][plane][row][col], values already rounded to fp16
    const int img = blockIdx.z, b = img / F, f = img % F;
    const int h0 = blockIdx.y * T, w0 = blockIdx.x * T;
    const float* p0 = in0 + ((size_t)b * f0 + (f0 == 1 ? 0 : f)) * H * W;
    const float* p1 = in1 + ((size_t)b * f1 + (f1 == 1 ? 0 : f)) * H * W;
    const bool drop = keep && keep[b] == 0.f;
    for (int x = threadIdx.x; x < 2 * PW * PW; x += 256) {
        const int ci = x / (PW * PW), rr = (x / PW) % PW, cc = x % PW;
        const int hh = h0 + rr - PAD, ww = w0 + cc - PAD;
        float v = 0.f;
        if (hh >= 0 && hh < H && ww >= 0 && ww < W && !(ci && drop)) v = (ci ? p1 : p0)[(size_t)hh * W + ww];
        const float hi = __half2float(__float2half_rn(v));
        sv[0][ci][rr][cc] = hi;
        sv[1][ci][rr][cc] = __half2float(__float2half_rn(v - hi));
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int off[8];     // >= 0: offset into sv for pixel (0,0); -1: constant 1; -2: constant 0
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int k = lane * 8 + j;
        if (k < 2 * NT) {
            const int part = k / NT, rem = k % NT, ci = rem / (KS * KS), kh = (rem % (KS * KS)) / KS, kw = rem % KS;
            off[j] = ((part * 2 + ci) * PW + kh) * PW + kw;
        } else {
            off[j] = k < 2 * NT + 2 ? -1 : -2;
        }
    }
    __syncthreads();
    const float* s0 = &sv[0][0][0][0];
    for (int px = warp; px < T * T; px += 8) {
        const int ty = px / T, tx = px % T;
        const int h = h0 + ty, w = w0 + tx;
        if (h >= H || w >= W) continue;
        const int base = ty * PW + tx;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = off[j] >= 0 ? s0[off[j] + base] : (off[j] == -1 ? 1.f : 0.f);
        uint4 u;
        u.x = pack_h2(v[0], v[1]); u.y = pack_h2(v[2], v[3]);
        u.z = pack_h2(v[4], v[5]); u.w = pack_h2(v[6], v[7]);
        *reinterpret_cast<uint4*>(out + (((size_t)img * H + h) * W + w) * KPAD + lane * 8) = u;
    }
}
// fp16 GEMM operand [COUT][KPAD] = [w | w | fp16(bias) | fp16(bias - fp16(bias)) | 0]
__global__ void input_weight_pack_kernel(const float* __restrict__ w, const float* __restrict__ bias,
                                         h16* __restrict__ out, int cout, int nt, int kpad) {
    pdl_trigger();
    pdl_wait();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= cout * kpad) return;
    const int o = idx / kpad, k = idx % kpad;
    float v = 0.f;
    if (k < 2 * nt) v = w[o * nt + (k % nt)];
    else if (k == 2 * nt) v = bias[o];
    else if (k == 2 * nt + 1) v = bias[o] - __half2float(__float2half_rn(bias[o]));
    out[idx] = __float2half_rn(v);
}

// ------------------------------------------------------------------------------------------------
// 7x7 input conv, 2 input planes (noisy target, condition) -> COUT channels, fp16 NHWC output.
// Plane p of image (b, f) lives at in_p + (b*fp + (fp == 1 ? 0 : f)) * H*W  (frame broadcast).
// ------------------------------------------------------------------------------------------------
template <int KS, int COUT>
__global__ void __launch_bounds__(256)
input_conv_fwd_kernel(const float* __restrict__ in0, const float* __restrict__ in1, int f0, int f1,
                      const float* __restrict__ w /* [COUT][2][KS][KS] */, const float* __restrict__ bias,
                      h16* __restrict__ out, int F, int H, int W) {
    pdl_trigger();
    pdl_wait();
    constexpr int T = 16, PAD = KS / 2, PW = T + KS - 1;
    __shared__ float sw[2 * KS * KS][COUT];
    __shared__ float sin_[2][PW][PW + 1];
    const int img = blockIdx.z, b = img / F, f = img % F;
    const int h0 = blockIdx.y * T, w0 = blockIdx.x * T;
    for (int x = threadIdx.x; x < 2 * KS * KS * COUT; x += 256) {
        const int co = x % COUT, tap = x / COUT;
        sw[tap][co] = w[co * 2 * KS * KS + tap];
    }
    const float* p0 = in0 + ((size_t)b * f0 + (f0 == 1 ? 0 : f)) * H * W;
    const float* p1 = in1 + ((size_t)b * f1 + (f1 == 1 ? 0 : f)) * H * W;
    for (int x = threadIdx.x; x < 2 * PW * PW; x += 256) {
        const int ci = x / (PW * PW), rr = (x / PW) % PW, cc = x % PW;
        const int hh = h0 + rr - PAD, ww = w0 + cc - PAD;
        float v = 0.f;
        if (hh >= 0 && hh < H && ww >= 0 && ww < W) v = (ci ? p1 : p0)[(size_t)hh * W + ww];
        sin_[ci][rr][cc] = v;
    }
    __syncthreads();
    const int ty = threadIdx.x / T, tx = threadIdx.x % T;
    const int h = h0 + ty, ww = w0 + tx;
    float acc[COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) acc[c] = bias[c];
    for (int ci = 0; ci < 2; ++ci)
        for (int kh = 0; kh < KS; ++kh)
#pragma unroll
            for (int kw = 0; kw < KS; ++kw) {
                const float v = sin_[ci][ty + kh][tx + kw];
                const float4* wr = reinterpret_cast<const float4*>(sw[(ci * KS + kh) * KS + kw]);
#pragma unroll
                for (int c4 = 0; c4 < COUT / 4; ++c4) {
                    const float4 q = wr[c4];
                    acc[4 * c4 + 0] = fmaf(v, q.x, acc[4 * c4 + 0]);
                    acc[4 * c4 + 1] = fmaf(v, q.y, acc[4 * c4 + 1]);
                    acc[4 * c4 + 2] = fmaf(v, q.z, acc[4 * c4 + 2]);
                    acc[4 * c4 + 3] = fmaf(v, q.w, acc[4 * c4 + 3]);
                }
            }
    if (h < H && ww < W) {
        uint4* op = reinterpret_cast<uint4*>(out + (((size_t)img * H + h) * W + ww) * COUT);
#pragma unroll
        for (int j = 0; j < COUT / 8; ++j) {
            uint4 u;
            u.x = pack_h2(acc[8 * j + 0], acc[8 * j + 1]);
            u.y = pack_h2(acc[8 * j + 2], acc[8 * j + 3]);
            u.z = pack_h2(acc[8 * j + 4], acc[8 * j + 5]);
            u.w = pack_h2(acc[8 * j + 6], acc[8 * j + 7]);
            op[j] = u;
        }
    }
}

// dW[co][ci][kh][kw] += sum dy[img][h][w][co] * in_ci[img][h+kh-PAD][w+kw-PAD];  db[co] += sum dy
// Persistent blocks loop over 16x16 tiles; thread owns channel co = tid % COUT and every 4th tap.
template <int KS, int COUT>
__global__ void __launch_bounds__(256)
input_conv_wgrad_kernel(const float* __restrict__ in0, const float* __restrict__ in1, int f0, int f1,
                        const h16* __restrict__ dy, float* __restrict__ dw, float* __restrict__ db, int NI,
                        int F, int H, int W) {
    pdl_trigger();
    pdl_wait();
    // thread = 4 output channels x TPT taps: 4*TPT FMAs per (4 + TPT) shared-memory reads per pixel
    constexpr int T = 16, PAD = KS / 2, PW = T + KS - 1, NT = 2 * KS * KS, CG = COUT / 4, Q = 256 / CG;
    constexpr int TPT = (NT + Q - 1) / Q;  // taps per thread
    __shared__ float sin_[2][PW][PW + 1];
    __shared__ __align__(16) h16 sdy[T * T][COUT + 8];
    const int cg = threadIdx.x % CG, q = threadIdx.x / CG;
    float acc[TPT][4], accb[4] = {0.f, 0.f, 0.f, 0.f};
    int toff[TPT];  // offset of tap (ci, kh, kw) inside sin_ relative to [0][ty][tx]
#pragma unroll
    for (int i = 0; i < TPT; ++i) {
        acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
        const int tap = q + i * Q;
        const int ci = tap / (KS * KS), kh = (tap / KS) % KS, kw = tap % KS;
        toff[i] = tap < NT ? (ci * PW + kh) * (PW + 1) + kw : 0;
    }
    const float* sflat = &sin_[0][0][0];
    const int tiles_w = (W + T - 1) / T, tiles_h = (H + T - 1) / T;
    const int ntiles = tiles_w * tiles_h * NI;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int img = tile / (tiles_w * tiles_h), b = img / F, f = img % F;
        const int h0 = ((tile / tiles_w) % tiles_h) * T, w0 = (tile % tiles_w) * T;
        const float* p0 = in0 + ((size_t)b * f0 + (f0 == 1 ? 0 : f)) * H * W;
        const float* p1 = in1 + ((size_t)b * f1 + (f1 == 1 ? 0 : f)) * H * W;
        __syncthreads();
        for (int x = threadIdx.x; x < 2 * PW * PW; x += 256) {
            const int ci = x / (PW * PW), rr = (x / PW) % PW, cc = x % PW;
            const int hh = h0 + rr - PAD, ww = w0 + cc - PAD;
            float v = 0.f;
            if (hh >= 0 && hh < H && ww >= 0 && ww < W) v = (ci ? p1 : p0)[(size_t)hh * W + ww];
            sin_[ci][rr][cc] = v;
        }
        for (int x = threadIdx.x; x < T * T * (COUT / 8); x += 256) {
            const int px = x / (COUT / 8), v8 = x % (COUT / 8);
            const int h = h0 + px / T, ww = w0 + px % T;
            uint4 u = make_uint4(0, 0, 0, 0);
            if (h < H && ww < W) u = *reinterpret_cast<const uint4*>(dy + (((size_t)img * H + h) * W + ww) * COUT + v8 * 8);
            *reinterpret_cast<uint4*>(&sdy[px][v8 * 8]) = u;
        }
        __syncthreads();
#pragma unroll 2
        for (int px = 0; px < T * T; ++px) {
            const uint2 gu = *reinterpret_cast<const uint2*>(&sdy[px][cg * 4]);
            const float2 g01 = unpack_h2(gu.x), g23 = unpack_h2(gu.y);
            const int poff = (px / T) * (PW + 1) + (px % T);
            if (q == 0) {
                accb[0] += g01.x; accb[1] += g01.y; accb[2] += g23.x; accb[3] += g23.y;
            }
#pragma unroll
            for (int i = 0; i < TPT; ++i) {
                const float xv = sflat[poff + toff[i]];
                acc[i][0] = fmaf(g01.x, xv, acc[i][0]);
                acc[i][1] = fmaf(g01.y, xv, acc[i][1]);
                acc[i][2] = fmaf(g23.x, xv, acc[i][2]);
                acc[i][3] = fmaf(g23.y, xv, acc[i][3]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < TPT; ++i) {
        const int tap = q + i * Q;
        if (tap < NT) {
#pragma unroll
            for (int c = 0; c < 4; ++c) atomicAdd(&dw[(cg * 4 + c) * NT + tap], acc[i][c]);
        }
    }
    if (q == 0) {
#pragma unroll
        for (int c = 0; c < 4; ++c) atomicAdd(&db[cg * 4 + c], accb[c]);
    }
}

// d_in_p[b][fp][h][w] (+)= scale * sum_f sum_co sum_{kh,kw} dy[(b,f)][h-kh+PAD][w-kw+PAD][co] * W[co][p][kh][kw]:
// the transposed convolution of the input conv (zero padding), fp32 accumulation.  A block owns a 16x16 pixel tile
// of one batch element and walks its F frames: plane p is written after every frame when fp == F, and summed over
// the frames (the forward's broadcast) when fp == 1 < F.  Thread = one pixel.  Dynamic shared memory: the weights
// as float4 {W[co][0][t], W[co][1][t], W[co+1][0][t], W[co+1][1][t]} per (tap, channel pair), then the frame's dy
// halo tile as half2 words with a pixel stride of COUT/2 + 1 words and a row stride = 16 (mod 32) words, so the 32
// pixels (2 rows x 16) a warp reads per channel pair fall in 32 different banks.  keep (optional, [B]): where
// keep[b] == 0 the forward read a zero condition, so d_in1 of batch element b is 0 (written, or nothing added).
template <int KS, int COUT>
struct InputDgradSmem {
    static constexpr int T = 16, PAD = KS / 2, PW = T + KS - 1, CP = COUT / 2, PS = CP + 1;
    static constexpr int RS = PW * PS + ((16 - (PW * PS) % 32) + 32) % 32;
    static constexpr size_t W_BYTES = (size_t)KS * KS * CP * sizeof(float4);
    static constexpr size_t BYTES = W_BYTES + (size_t)PW * RS * sizeof(uint32_t);
};
template <int KS, int COUT, bool DX, bool DC>
__global__ void __launch_bounds__(256)
input_conv_dgrad_kernel(const h16* __restrict__ dy, const float* __restrict__ w /* [COUT][2][KS][KS] */,
                        float* __restrict__ dx, float* __restrict__ dc, const float* __restrict__ keep, int f0,
                        int f1, int F, int H, int W, float scale, int accumulate) {
    pdl_trigger();
    pdl_wait();
    using S = InputDgradSmem<KS, COUT>;
    constexpr int T = S::T, PAD = S::PAD, PW = S::PW, CP = S::CP, PS = S::PS, RS = S::RS, KK = KS * KS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float4* sw = reinterpret_cast<float4*>(smem_raw);                       // [KK][CP]
    uint32_t* sdy = reinterpret_cast<uint32_t*>(smem_raw + S::W_BYTES);     // [PW][RS], half2 words
    for (int x = threadIdx.x; x < KK * CP; x += 256) {
        const int tap = x / CP, cp = x % CP;
        const float* wa = w + (size_t)(2 * cp) * 2 * KK;
        const float* wb = wa + 2 * KK;
        sw[x] = make_float4(wa[tap], wa[KK + tap], wb[tap], wb[KK + tap]);
    }
    const int b = blockIdx.z, h0 = blockIdx.y * T, w0 = blockIdx.x * T;
    const int ty = threadIdx.x / T, tx = threadIdx.x % T;
    const int h = h0 + ty, ww = w0 + tx;
    const bool inside = h < H && ww < W;
    const bool drop = keep && keep[b] == 0.f;  // this batch element read a zero condition
    const size_t HW = (size_t)H * W, pix = (size_t)h * W + ww;
    const auto put = [&](float* p, float v) { *p = accumulate ? fmaf(scale, v, *p) : scale * v; };
    float a0 = 0.f, a1 = 0.f;
    for (int f = 0; f < F; ++f) {
        const size_t img = (size_t)b * F + f;
        __syncthreads();  // the previous frame's tile has been read by every thread
        for (int x = threadIdx.x; x < PW * PW * (COUT / 8); x += 256) {
            const int px = x / (COUT / 8), v8 = x % (COUT / 8);
            const int r = px / PW, c = px % PW;
            const int hh = h0 - PAD + r, wq = w0 - PAD + c;
            uint4 u = make_uint4(0, 0, 0, 0);
            if (hh >= 0 && hh < H && wq >= 0 && wq < W)
                u = *reinterpret_cast<const uint4*>(dy + ((img * H + hh) * W + wq) * COUT + v8 * 8);
            uint32_t* d = sdy + r * RS + c * PS + v8 * 4;
            d[0] = u.x; d[1] = u.y; d[2] = u.z; d[3] = u.w;
        }
        __syncthreads();
        // dy row of tap kh is h - kh + PAD, i.e. halo row ty - kh + 2*PAD (the halo starts at h0 - PAD)
        for (int kh = 0; kh < KS; ++kh) {
#pragma unroll
            for (int kw = 0; kw < KS; ++kw) {
                const uint32_t* dp = sdy + (ty - kh + 2 * PAD) * RS + (tx - kw + 2 * PAD) * PS;
                const float4* wp = sw + (kh * KS + kw) * CP;
#pragma unroll 8
                for (int cp = 0; cp < CP; ++cp) {
                    const float2 g = unpack_h2(dp[cp]);
                    const float4 q = wp[cp];
                    if (DX) { a0 = fmaf(g.x, q.x, a0); a0 = fmaf(g.y, q.z, a0); }
                    if (DC) { a1 = fmaf(g.x, q.y, a1); a1 = fmaf(g.y, q.w, a1); }
                }
            }
        }
        if (DX && f0 == F) {
            if (inside) put(dx + ((size_t)b * F + f) * HW + pix, a0);
            a0 = 0.f;
        }
        if (DC && f1 == F) {
            if (inside) put(dc + ((size_t)b * F + f) * HW + pix, drop ? 0.f : a1);
            a1 = 0.f;
        }
    }
    if (DX && f0 != F && inside) put(dx + (size_t)b * HW + pix, a0);
    if (DC && f1 != F && inside) put(dc + (size_t)b * HW + pix, drop ? 0.f : a1);
}

// eps[b][h][w] = bias + sum_c a[(b*F + mid)][h][w][c] * w[c]   ; 8 lanes per pixel (C == 64)
__global__ void __launch_bounds__(256)
out_conv_fwd_kernel(const h16* __restrict__ a, const float* __restrict__ w, const float* __restrict__ bias,
                    float* __restrict__ eps, int B, int F, int mid, long long HW) {
    pdl_trigger();
    pdl_wait();
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long pix = t >> 3;
    const int sub = t & 7;
    float s = 0.f;
    if (pix < (long long)B * HW) {
        const long long b = pix / HW, p = pix % HW;
        uint4 u = *reinterpret_cast<const uint4*>(a + (((size_t)b * F + mid) * HW + p) * 64 + sub * 8);
        float2 x0 = unpack_h2(u.x), x1 = unpack_h2(u.y), x2 = unpack_h2(u.z), x3 = unpack_h2(u.w);
        const float* ww = w + sub * 8;
        s = x0.x * ww[0] + x0.y * ww[1] + x1.x * ww[2] + x1.y * ww[3] + x2.x * ww[4] + x2.y * ww[5] + x3.x * ww[6] + x3.y * ww[7];
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (sub == 0 && pix < (long long)B * HW) eps[pix] = s + bias[0];
}
// da[(b,f)][p][c] = (f == mid) ? deps[b][p]*w[c] : 0 ; dw[c] += sum deps*a ; db += sum deps
__global__ void __launch_bounds__(256)
out_conv_bwd_kernel(const h16* __restrict__ a, const float* __restrict__ w, const float* __restrict__ deps,
                    h16* __restrict__ da, float* __restrict__ dw, float* __restrict__ db, int B, int F, int mid,
                    long long HW) {
    pdl_trigger();
    pdl_wait();
    const int sub = threadIdx.x & 7;
    float wv[8], acc[8], accb = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        wv[i] = w[sub * 8 + i];
        acc[i] = 0.f;
    }
    const long long total = (long long)B * F * HW;
    for (long long pix = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3; pix < total;
         pix += ((long long)gridDim.x * blockDim.x) >> 3) {
        const long long img = pix / HW, p = pix % HW;
        const int f = img % F;
        const long long b = img / F;
        uint4 o = make_uint4(0, 0, 0, 0);
        if (f == mid) {
            const float g = deps[b * HW + p];
            uint4 u = *reinterpret_cast<const uint4*>(a + pix * 64 + sub * 8);
            float2 x0 = unpack_h2(u.x), x1 = unpack_h2(u.y), x2 = unpack_h2(u.z), x3 = unpack_h2(u.w);
            acc[0] += g * x0.x; acc[1] += g * x0.y; acc[2] += g * x1.x; acc[3] += g * x1.y;
            acc[4] += g * x2.x; acc[5] += g * x2.y; acc[6] += g * x3.x; acc[7] += g * x3.y;
            if (sub == 0) accb += g;
            o.x = pack_h2(g * wv[0], g * wv[1]);
            o.y = pack_h2(g * wv[2], g * wv[3]);
            o.z = pack_h2(g * wv[4], g * wv[5]);
            o.w = pack_h2(g * wv[6], g * wv[7]);
        }
        *reinterpret_cast<uint4*>(da + pix * 64 + sub * 8) = o;
    }
    __shared__ float red[256][9];
#pragma unroll
    for (int i = 0; i < 8; ++i) red[threadIdx.x][i] = acc[i];
    red[threadIdx.x][8] = accb;
    __syncthreads();
    if (threadIdx.x < 64) {
        const int c = threadIdx.x;
        float s = 0.f;
        for (int t = c >> 3; t < 256; t += 8) s += red[t][c & 7];
        atomicAdd(&dw[c], s);
    } else if (threadIdx.x == 64) {
        float s = 0.f;
        for (int t = 0; t < 256; t += 8) s += red[t][8];
        atomicAdd(db, s);
    }
}

// ------------------------------------------------------------------------------------------------
// time embedding + small fp32 linears (batch <= a few hundred rows)
// ------------------------------------------------------------------------------------------------
__global__ void sinusoidal_kernel(const long long* __restrict__ t, float* __restrict__ out, int B, int dim) {
    pdl_trigger();
    pdl_wait();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * dim) return;
    const int b = idx / dim, i = idx % dim, half = dim / 2;
    const int k = i % half;
    const float freq = expf((float)k * -(logf(10000.f) / (float)(half - 1)));
    const float arg = (float)t[b] * freq;
    out[idx] = i < half ? sinf(arg) : cosf(arg);
}
// y[b][n] = sum_k act(x[b][k]) W[n][k] + bias[n]; warp per n
__global__ void __launch_bounds__(256)
small_linear_fwd_kernel(const float* __restrict__ x, const float* __restrict__ W, const float* __restrict__ bias,
                        float* __restrict__ y, int B, int K, int N, int act) {
    pdl_trigger();
    pdl_wait();
    const int n = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    for (int b = blockIdx.y; b < B; b += gridDim.y) {  // grid.y = B: one warp per (row, output)
        float s = 0.f;
        for (int k = lane; k < K; k += 32) {
            float v = x[(size_t)b * K + k];
            if (act) v = silu_precise(v);
            s = fmaf(v, W[(size_t)n * K + k], s);
        }
        s = warp_sum(s);
        if (lane == 0) y[(size_t)b * N + n] = s + (bias ? bias[n] : 0.f);
    }
}
// dW[n][k] = sum_b dy[b][n] act(x[b][k]) ; db[n] = sum_b dy[b][n]
__global__ void small_linear_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ dy,
                                          float* __restrict__ dW, float* __restrict__ db, int B, int K, int N, int act,
                                          int accumulate) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * K) return;
    const int k = idx % K, n = idx / K;
    float s = 0.f, sb = 0.f;
    for (int b = 0; b < B; ++b) {
        float v = x[(size_t)b * K + k];
        if (act) v = silu_precise(v);
        const float g = dy[(size_t)b * N + n];
        s = fmaf(g, v, s);
        sb += g;
    }
    dW[idx] = accumulate ? dW[idx] + s : s;
    if (k == 0 && db) db[n] = accumulate ? db[n] + sb : sb;
}
// dx[b][k] = act'(x[b][k]) * sum_n dy[b][n] W[n][k]
// block = (32 k-lanes x 8 n-groups); grid = (ceil(K/32), B): rows of W are read coalesced along k,
// the 8 warps split n and combine through shared memory.
__global__ void __launch_bounds__(256)
small_linear_dgrad_kernel(const float* __restrict__ x, const float* __restrict__ W, const float* __restrict__ dy,
                          float* __restrict__ dx, int B, int K, int N, int act) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int k = blockIdx.x * 32 + lane, b = blockIdx.y;
    float s = 0.f;
    if (k < K) {
#pragma unroll 4
        for (int n = w; n < N; n += 8) s = fmaf(__ldg(dy + (size_t)b * N + n), __ldg(W + (size_t)n * K + k), s);
    }
    __shared__ float red[8][33];
    red[w][lane] = s;
    __syncthreads();
    if (w == 0 && k < K) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += red[i][lane];
        if (act) t *= dsilu_precise(x[(size_t)b * K + k]);
        dx[(size_t)b * K + k] = t;
    }
}

// ------------------------------------------------------------------------------------------------
// All FiLM projections of the network at once (video_net.py:238-241, one per ResnetBlock): they share the
// input act(temb) and differ only in their weights, so the ~15 tiny linears of a pass -- and in the
// backward pass their weight gradients, and the sum of their data gradients -- are ONE launch each over a
// device table of layers instead of ~45 launches plus the autograd adds of d temb.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int film_find(const cesm_film_desc* __restrict__ L, int n_layers, int n, int& local) {
    int i = 0;
    while (i + 1 < n_layers && n >= L[i + 1].n0) ++i;
    local = n - L[i].n0;
    return i;
}
// y_i[b][j] = sum_k silu(x[b][k]) W_i[j][k] + bias_i[j]; warp per (global output, b)
__global__ void __launch_bounds__(256)
film_fwd_kernel(const float* __restrict__ x, const cesm_film_desc* __restrict__ L, float* __restrict__ Y, int n_layers,
                int n_total, int B, int K) {
    pdl_trigger();
    pdl_wait();
    const int n = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31, b = blockIdx.y;
    if (n >= n_total) return;
    int j;
    const cesm_film_desc d = L[film_find(L, n_layers, n, j)];
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s = fmaf(silu_precise(x[(size_t)b * K + k]), d.W[(size_t)j * K + k], s);
    s = warp_sum(s);
    if (lane == 0) Y[(size_t)B * d.n0 + (size_t)b * d.N + j] = s + d.bias[j];
}
// dW_i[j][k] += sum_b dy_i[b][j] silu(x[b][k]); db_i[j] += sum_b dy_i[b][j]   (thread per (global output, k))
__global__ void __launch_bounds__(256)
film_wgrad_kernel(const float* __restrict__ x, const cesm_film_desc* __restrict__ L, const float* __restrict__ DY,
                  int n_layers, int n_total, int B, int K, int accumulate) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n_total * K) return;
    const int k = idx % K, n = idx / K;
    int j;
    const cesm_film_desc d = L[film_find(L, n_layers, n, j)];
    float s = 0.f, sb = 0.f;
    for (int b = 0; b < B; ++b) {
        const float g = DY[(size_t)B * d.n0 + (size_t)b * d.N + j];
        s = fmaf(g, silu_precise(x[(size_t)b * K + k]), s);
        sb += g;
    }
    float* w = d.dW + (size_t)j * K + k;
    *w = accumulate ? *w + s : s;
    if (k == 0) d.db[j] = accumulate ? d.db[j] + sb : sb;
}
// dx[b][k] += silu'(x[b][k]) * sum_j dy_i[b][j] W_i[j][k] for layer i = blockIdx.z (dx zeroed by the caller);
// block = 32 k-lanes x 8 output groups
__global__ void __launch_bounds__(256)
film_dgrad_kernel(const float* __restrict__ x, const cesm_film_desc* __restrict__ L, const float* __restrict__ DY,
                  int n_layers, float* __restrict__ dx, int B, int K) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int k = blockIdx.x * 32 + lane, b = blockIdx.y, i = blockIdx.z;
    float s = 0.f;
    if (k < K) {
        const float* __restrict__ dy = DY + (size_t)B * L[i].n0 + (size_t)b * L[i].N;
        const float* __restrict__ W = L[i].W;
        const int N = L[i].N;
#pragma unroll 4
        for (int j = w; j < N; j += 8) s = fmaf(__ldg(dy + j), __ldg(W + (size_t)j * K + k), s);
    }
    __shared__ float red[8][33];
    red[w][lane] = s;
    __syncthreads();
    if (w == 0 && k < K) {
        float t = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) t += red[q][lane];
        atomicAdd(dx + (size_t)b * K + k, t * dsilu_precise(x[(size_t)b * K + k]));
    }
}

// ------------------------------------------------------------------------------------------------
// DDPM elementwise
// ------------------------------------------------------------------------------------------------
__global__ void q_sample_kernel(const float* __restrict__ x0, const float* __restrict__ noise,
                                const long long* __restrict__ t, const float* __restrict__ sqrt_ac,
                                const float* __restrict__ sqrt_1mac, float* __restrict__ xt, long long per, long long total) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long tb = t[idx / per];
    xt[idx] = sqrt_ac[tb] * x0[idx] + sqrt_1mac[tb] * noise[idx];
}
// dx0 = sqrt_ac[t] * g, dnoise = sqrt_1mac[t] * g (either may be null)
__global__ void q_sample_bwd_kernel(const float* __restrict__ g, const long long* __restrict__ t,
                                    const float* __restrict__ sqrt_ac, const float* __restrict__ sqrt_1mac,
                                    float* __restrict__ dx0, float* __restrict__ dnoise, long long per, long long total) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long tb = t[idx / per];
    const float gv = g[idx];
    if (dx0) dx0[idx] = sqrt_ac[tb] * gv;
    if (dnoise) dnoise[idx] = sqrt_1mac[tb] * gv;
}
// loss += sum (eps-noise)^2 / total ; diff = eps - noise
__global__ void __launch_bounds__(256)
mse_fwd_kernel(const float* __restrict__ eps, const float* __restrict__ noise, float* __restrict__ diff,
               float* __restrict__ loss, long long total) {
    pdl_trigger();
    pdl_wait();
    float s = 0.f;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const float d = eps[idx] - noise[idx];
        diff[idx] = d;
        s = fmaf(d, d, s);
    }
    __shared__ float red[8];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0.f;
        for (int i = 0; i < 8; ++i) tot += red[i];
        atomicAdd(loss, tot / (float)total);
    }
}
// Diffusion objective with a per-timestep target and weight.  Block (x, b) covers part of sample b, so t, the target
// row and the weight are uniform in a block.  target = c_n[t] * noise + c_x[t] * x0 from coef[T][2] rows (c_n, c_x);
// a null coef is the eps target (x0 not read).  A null weight is 1.  A t outside [0, T) yields NaN.
struct LossRow {
    float cn, cx, w;
    bool valid;
};
__device__ __forceinline__ LossRow loss_row(const long long* __restrict__ t, const float* __restrict__ coef,
                                            const float* __restrict__ weight, int T, int b) {
    const long long tb = t[b];
    LossRow r;
    r.valid = tb >= 0 && tb < T;
    r.cn = 1.f, r.cx = 0.f, r.w = 1.f;
    if (r.valid && coef) r.cn = coef[2 * tb], r.cx = coef[2 * tb + 1];
    if (r.valid && weight) r.w = weight[tb];
    return r;
}
// diff = pred - target;  loss += w[t] * sum diff^2 / total
__global__ void __launch_bounds__(256)
diffusion_loss_fwd_kernel(const float* __restrict__ pred, const float* __restrict__ x0, const float* __restrict__ noise,
                          const long long* __restrict__ t, const float* __restrict__ coef,
                          const float* __restrict__ weight, float* __restrict__ diff, float* __restrict__ loss, int T,
                          long long per, long long total) {
    pdl_trigger();
    pdl_wait();
    const int b = blockIdx.y;
    const LossRow r = loss_row(t, coef, weight, T, b);
    const float qnan = __int_as_float(0x7fc00000);
    const long long base = (long long)b * per;
    float s = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per; i += (long long)gridDim.x * blockDim.x) {
        const long long idx = base + i;
        float d = qnan;
        if (r.valid) d = pred[idx] - (coef ? fmaf(r.cn, noise[idx], r.cx * x0[idx]) : noise[idx]);
        diff[idx] = d;
        s = fmaf(d, d, s);
    }
    __shared__ float red[8];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0.f;
        for (int i = 0; i < 8; ++i) tot += red[i];
        atomicAdd(loss, r.valid ? tot * (r.w / (float)total) : qnan);
    }
}
// dpred = factor * g * w[t] * diff;  dnoise = -c_n[t] * dpred;  dx0 = -c_x[t] * dpred  (each output may be null)
__global__ void diffusion_loss_bwd_kernel(const float* __restrict__ diff, const long long* __restrict__ t,
                                          const float* __restrict__ coef, const float* __restrict__ weight,
                                          const float* __restrict__ gscale, float factor, float* __restrict__ dpred,
                                          float* __restrict__ dnoise, float* __restrict__ dx0, int T, long long per) {
    pdl_trigger();
    pdl_wait();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= per) return;
    const int b = blockIdx.y;
    const LossRow r = loss_row(t, coef, weight, T, b);
    const long long idx = (long long)b * per + i;
    const float p = r.valid ? diff[idx] * (factor * gscale[0] * r.w) : __int_as_float(0x7fc00000);
    if (dpred) dpred[idx] = p;
    if (dnoise) dnoise[idx] = -r.cn * p;
    if (dx0) dx0[idx] = -r.cx * p;
}
// out = in * factor * (*gscale)
__global__ void scale_by_device_scalar_kernel(const float* __restrict__ in, const float* __restrict__ gscale,
                                              float factor, float* __restrict__ out, long long total) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    out[idx] = in[idx] * factor * gscale[0];
}
// x_{t-1} = sqrt_recip_alpha[t] * (x_t - beta[t]/sqrt_1mac[t] * eps) + sqrt(post_var[t]) * z
// (post_var[0] == 0, so t == 0 adds no noise: identical to model.py:178-183).  Shared by the buffered-z and the
// seeded kernel so that both round the same way.
__device__ __forceinline__ float p_sample_update(float x, float e, float z, long long tb, const float* betas,
                                                 const float* sqrt_1mac, const float* sqrt_recip_a,
                                                 const float* post_var) {
    const float mean = sqrt_recip_a[tb] * (x - betas[tb] / sqrt_1mac[tb] * e);
    return mean + sqrtf(post_var[tb]) * z;
}
// Classifier-free guidance (Ho & Salimans) inside the update kernels: with kGuided the network output holds 2B rows,
// the B conditional predictions c, then the B null-condition predictions u of the same fields (u of element i at
// i + half, half = B * per), and the update uses c + w (c - u) = (1 + w) c - w u in the network's own output space.
// No combined tensor is written.  Without kGuided the kernels read eps[i] as before.
template <bool kGuided>
__device__ __forceinline__ float net_out(const float* eps, long long i, long long half, float w) {
    if (!kGuided) return eps[i];
    const float c = eps[i];
    return fmaf(w, c - eps[i + half], c);
}
template <bool kGuided>
__global__ void p_sample_kernel(const float* __restrict__ xt, const float* __restrict__ eps,
                                const float* __restrict__ z, const long long* __restrict__ t,
                                const float* __restrict__ betas, const float* __restrict__ sqrt_1mac,
                                const float* __restrict__ sqrt_recip_a, const float* __restrict__ post_var,
                                float* __restrict__ out, long long per, long long total, float w) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long tb = t[idx / per];
    out[idx] = p_sample_update(xt[idx], net_out<kGuided>(eps, idx, total, w), z[idx], tb, betas, sqrt_1mac,
                               sqrt_recip_a, post_var);
}
// Strided DDIM step (Song et al.): x_prev = A[t] * x_t + B[t] * eps + S[t] * z, with the three coefficients of each
// schedule timestep precomputed on the host in float64 (model.ddim_schedule) and stored as coef[T][3] fp32.
// `out` may alias `xt` (each thread reads its element before writing it), so no __restrict__ on either.
// z == nullptr drops the noise term (valid when every S is 0, i.e. eta = 0).  A timestep outside [0, T) writes
// NaN instead of reading outside the table.  t_out (optional, never aliasing t) receives next_t[t] per sample;
// an out-of-range t is passed through unchanged, so a chain that overruns its schedule keeps producing NaN.
// The noise term is fmaf(S, z, ddim_mean(...)) in this kernel and in the seeded one.
__device__ __forceinline__ float ddim_mean(const float* c, float x, float e) { return fmaf(c[0], x, c[1] * e); }
template <bool kGuided>
__global__ void ddim_step_kernel(const float* xt, const float* __restrict__ eps, const float* __restrict__ z,
                                 const long long* __restrict__ t, const float* __restrict__ coef,
                                 const long long* __restrict__ next_t, long long* __restrict__ t_out, float* out,
                                 int T, long long per, long long total, float w) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long b = idx / per;
    const long long tb = t[b];
    const bool valid = tb >= 0 && tb < T;
    if (t_out && idx == b * per) t_out[b] = valid ? next_t[tb] : tb;
    if (!valid) {
        out[idx] = __int_as_float(0x7fc00000);
        return;
    }
    const float* c = coef + 3 * tb;
    float v = ddim_mean(c, xt[idx], net_out<kGuided>(eps, idx, total, w));
    if (z) v = fmaf(c[2], z[idx], v);
    out[idx] = v;
}
// DPM-Solver++(2M) step (Lu et al.), data-prediction form, from the fp32 coef[T][5] rows (P, Q, R, K0, K1) that
// model.dpm_schedule computes on the host in float64:
//     x0 = P x + Q eps,   out = R x + K0 x0 + K1 hist,   hist <- x0
// hist is the previous step's x0 prediction.  Where K1 == 0 (the first-order first and last steps) hist is not read,
// so a stale or NaN history cannot reach the output and a new chain needs no reset.  `out` may alias `xt`; hist
// aliases nothing.  An out-of-range t writes NaN to out and hist and passes t through to t_out, as ddim_step does.
template <bool kGuided>
__global__ void dpm_step_kernel(const float* xt, const float* __restrict__ eps, float* __restrict__ hist,
                                const long long* __restrict__ t, const float* __restrict__ coef,
                                const long long* __restrict__ next_t, long long* __restrict__ t_out, float* out,
                                int T, long long per, long long total, float w) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long b = idx / per;
    const long long tb = t[b];
    const bool valid = tb >= 0 && tb < T;
    if (t_out && idx == b * per) t_out[b] = valid ? next_t[tb] : tb;
    if (!valid) {
        out[idx] = __int_as_float(0x7fc00000);
        hist[idx] = __int_as_float(0x7fc00000);
        return;
    }
    const float* c = coef + 5 * tb;
    const float x = xt[idx];
    const float x0 = fmaf(c[0], x, c[1] * net_out<kGuided>(eps, idx, total, w));
    float v = fmaf(c[2], x, c[3] * x0);
    const float k1 = c[4];
    if (k1 != 0.0f) v = fmaf(k1, hist[idx], v);
    hist[idx] = x0;
    out[idx] = v;
}

// ------------------------------------------------------------------------------------------------
// Counter-based noise of the seeded sampling chains.  Element e of field f in draw d is word e & 3 of
//     Philox4x32-10(counter = (e >> 2, d, f_lo, f_hi), key = (seed_lo, seed_hi))      (Salmon et al. 2011)
// turned into normals by Box-Muller on the word pairs (w0, w1) and (w2, w3): u = ((w >> 9) + 0.5) 2^-23 lies in
// (0, 1) and is exact in fp32 (24 significant bits; (w >> 8) + 0.5 would need 25 and round, up to 1.0 for the largest
// words), r = sqrt(-2 log u_a), normals (r cospi(2 u_b), r sinpi(2 u_b)).  A value depends on
// (seed, field, draw, e) only, never on the row, the batch, the device or the launch shape.  x_T is draw 0xFFFFFFFF
// and the step leaving timestep t draws with d = t.  logf and sincospif are the accurate ones (no fast math).
// One thread makes one quad of one field (grid.y = field row), so a quad never crosses a field.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, unsigned k0, unsigned k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
        const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}
__device__ __forceinline__ float philox_uniform(unsigned w) { return ((float)(w >> 9) + 0.5f) * 0x1p-23f; }
__device__ __forceinline__ void box_muller(unsigned wa, unsigned wb, float& n0, float& n1) {
    const float r = sqrtf(-2.0f * logf(philox_uniform(wa)));
    float s, c;
    sincospif(2.0f * philox_uniform(wb), &s, &c);
    n0 = r * c;
    n1 = r * s;
}
// The four normals of quad q (elements 4q .. 4q+3) of `field` in `draw`.
__device__ __forceinline__ void field_normal4(unsigned seed_lo, unsigned seed_hi, long long field, unsigned draw,
                                              long long q, float (&z)[4]) {
    const unsigned long long f = (unsigned long long)field;
    const uint4 w = philox4x32_10(make_uint4((unsigned)q, draw, (unsigned)f, (unsigned)(f >> 32)), seed_lo, seed_hi);
    box_muller(w.x, w.y, z[0], z[1]);
    box_muller(w.z, w.w, z[2], z[3]);
}
// n = valid elements of the quad (4 unless it is the tail of a field whose size is not a multiple of 4); kVec means
// per % 4 == 0 with 16-byte aligned rows, so the quad is one float4.
template <bool kVec>
__device__ __forceinline__ void load_quad(const float* p, int n, float (&v)[4]) {
    if (kVec) {
        const float4 a = *reinterpret_cast<const float4*>(p);
        v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w;
        return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = j < n ? p[j] : 0.0f;
}
template <bool kVec>
__device__ __forceinline__ void store_quad(float* p, int n, const float (&v)[4]) {
    if (kVec) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
        return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (j < n) p[j] = v[j];
}

template <bool kVec>
__global__ void __launch_bounds__(256)
field_normal_kernel(unsigned seed_lo, unsigned seed_hi, const long long* __restrict__ field_ids, unsigned draw,
                    float* __restrict__ out, long long per) {
    pdl_trigger();
    pdl_wait();
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (4 * q >= per) return;
    const int b = blockIdx.y;
    float z[4];
    field_normal4(seed_lo, seed_hi, field_ids[b], draw, q, z);
    store_quad<kVec>(out + (long long)b * per + 4 * q, (int)min(4LL, per - 4 * q), z);
}

// p_sample_kernel with z drawn in registers from (seed, field_ids[b], draw t[b]).  `out` may alias `xt` (a thread
// reads its quad before writing it).  A t outside [0, T) writes NaN instead of reading outside the schedule.
// The network output quad of the update: eps's, or with kGuided c + w (c - u) from both halves (net_out).
template <bool kVec, bool kGuided>
__device__ __forceinline__ void load_net_quad(const float* eps, long long off, long long half, float w, int n,
                                              float (&e)[4]) {
    load_quad<kVec>(eps + off, n, e);
    if (!kGuided) return;
    float u[4];
    load_quad<kVec>(eps + off + half, n, u);
#pragma unroll
    for (int j = 0; j < 4; ++j) e[j] = fmaf(w, e[j] - u[j], e[j]);
}

template <bool kVec, bool kGuided>
__global__ void __launch_bounds__(256)
p_sample_seeded_kernel(const float* xt, const float* __restrict__ eps, unsigned seed_lo, unsigned seed_hi,
                       const long long* __restrict__ field_ids, const long long* __restrict__ t,
                       const float* __restrict__ betas, const float* __restrict__ sqrt_1mac,
                       const float* __restrict__ sqrt_recip_a, const float* __restrict__ post_var, float* out, int T,
                       long long per, float w) {
    pdl_trigger();
    pdl_wait();
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (4 * q >= per) return;
    const int b = blockIdx.y;
    const int n = (int)min(4LL, per - 4 * q);
    const long long off = (long long)b * per + 4 * q;
    const long long tb = t[b];
    float v[4];
    if (tb < 0 || tb >= T) {
        const float nan = __int_as_float(0x7fc00000);
        v[0] = v[1] = v[2] = v[3] = nan;
        store_quad<kVec>(out + off, n, v);
        return;
    }
    float x[4], e[4], z[4];
    field_normal4(seed_lo, seed_hi, field_ids[b], (unsigned)tb, q, z);
    load_quad<kVec>(xt + off, n, x);
    load_net_quad<kVec, kGuided>(eps, off, (long long)gridDim.y * per, w, n, e);
#pragma unroll
    for (int j = 0; j < 4; ++j)
        v[j] = p_sample_update(x[j], e[j], z[j], tb, betas, sqrt_1mac, sqrt_recip_a, post_var);
    store_quad<kVec>(out + off, n, v);
}

// ddim_step_kernel with z drawn in registers from (seed, field_ids[b], draw t[b]); same t_out / NaN contract.
template <bool kVec, bool kGuided>
__global__ void __launch_bounds__(256)
ddim_step_seeded_kernel(const float* xt, const float* __restrict__ eps, unsigned seed_lo, unsigned seed_hi,
                        const long long* __restrict__ field_ids, const long long* __restrict__ t,
                        const float* __restrict__ coef, const long long* __restrict__ next_t,
                        long long* __restrict__ t_out, float* out, int T, long long per, float w) {
    pdl_trigger();
    pdl_wait();
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (4 * q >= per) return;
    const int b = blockIdx.y;
    const int n = (int)min(4LL, per - 4 * q);
    const long long off = (long long)b * per + 4 * q;
    const long long tb = t[b];
    const bool valid = tb >= 0 && tb < T;
    if (t_out && q == 0) t_out[b] = valid ? next_t[tb] : tb;
    float v[4];
    if (!valid) {
        const float nan = __int_as_float(0x7fc00000);
        v[0] = v[1] = v[2] = v[3] = nan;
        store_quad<kVec>(out + off, n, v);
        return;
    }
    float x[4], e[4], z[4];
    field_normal4(seed_lo, seed_hi, field_ids[b], (unsigned)tb, q, z);
    load_quad<kVec>(xt + off, n, x);
    load_net_quad<kVec, kGuided>(eps, off, (long long)gridDim.y * per, w, n, e);
    const float* c = coef + 3 * tb;
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = fmaf(c[2], z[j], ddim_mean(c, x[j], e[j]));
    store_quad<kVec>(out + off, n, v);
}

// Condition dropout of a training step: keep[b] = (u >= p) ? 1 : 0 with u the uniform of word 0 of
//     Philox4x32-10(counter = (g_lo, g_hi, s_lo, s_hi), key = (seed_lo, seed_hi)),   g = first + b, s = *step,
// then *step += 1.  The draw depends on (seed, step, global sample index g) only, so a global batch split over ranks
// (first = rank * B) drops the same samples as on one GPU.  One block; the counter is read by every thread before
// thread 0 advances it.
__global__ void __launch_bounds__(256)
cond_keep_kernel(unsigned seed_lo, unsigned seed_hi, long long* __restrict__ step, long long first, float p,
                 float* __restrict__ keep, int B) {
    pdl_trigger();
    pdl_wait();
    const unsigned long long s = (unsigned long long)*step;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const unsigned long long g = (unsigned long long)(first + b);
        const uint4 w = philox4x32_10(make_uint4((unsigned)g, (unsigned)(g >> 32), (unsigned)s, (unsigned)(s >> 32)),
                                      seed_lo, seed_hi);
        keep[b] = philox_uniform(w.x) >= p ? 1.0f : 0.0f;
    }
    __syncthreads();
    if (threadIdx.x == 0) *step = (long long)(s + 1);
}

// ------------------------------------------------------------------------------------------------
// On-device data path (dataset_single_member.py:168-196): the whole (T, M, H, W) condition and target
// arrays stay resident in HBM; one launch assembles a batch -- K-frame window gather with the
// time-reversal frame map folded in, target frame, common spatial crop.  Per-sample plan (host RNG, so
// the draw order is the reference's): plan[b] = {member, first frame, target frame, crop row, crop col,
// reverse flag}.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gather_windows_kernel(const float* __restrict__ cond, const float* __restrict__ tgt, const int* __restrict__ plan,
                      float* __restrict__ cond_out, float* __restrict__ x0_out, int M, int H, int W, int K, int h,
                      int w, long long total) {
    pdl_trigger();
    pdl_wait();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = idx % w;
    const int y = (idx / w) % h;
    const int k = (idx / ((long long)w * h)) % (K + 1);   // plane K is the target
    const int b = idx / ((long long)w * h * (K + 1));
    const int* pl = plan + b * 6;
    const int m = pl[0], t0 = pl[1], ta = pl[2], i0 = pl[3], j0 = pl[4], rev = pl[5];
    if (k == K) {
        x0_out[((size_t)b * h + y) * w + x] = tgt[(((size_t)ta * M + m) * H + i0 + y) * W + j0 + x];
        return;
    }
    // time reversal around the centre frame (dataset_single_member.py:178-186): the halves left and
    // right of the centre are flipped, the centre (anchor) frame stays
    const int mid = K / 2;
    int src = k;
    if (rev) src = k < mid ? mid - 1 - k : (k == mid ? mid : K + mid - k);
    cond_out[(((size_t)b * K + k) * h + y) * w + x] = cond[(((size_t)(t0 + src) * M + m) * H + i0 + y) * W + j0 + x];
}

}  // namespace cesm

using namespace cesm;

static inline int nblk(long long total, int threads) { return (int)((total + threads - 1) / threads); }

extern "C" int cesm_pack_weight(const float* src, void* dst, int O, int T, int I, long long so, long long si,
                                const int32_t* tap_off, void* stream) {
    CESM_REQUIRE(T >= 1 && T <= CESM_MAX_TAPS, "T=%d out of range", T);
    TapOffsets taps{};
    for (int t = 0; t < T; ++t) taps.off[t] = tap_off[t];
    const long long total = (long long)O * T * I;
    launch_pdl(pack_weight_kernel, nblk(total, 256), 256, 0, as_stream(stream), src, (h16*)dst, O, T, I, so, si, taps);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_unpack_wgrad(const float* src, float* dst, int O, int T, int I, long long so, long long si,
                                 const int32_t* tap_off, int accumulate, void* stream) {
    CESM_REQUIRE(T >= 1 && T <= CESM_MAX_TAPS, "T=%d out of range", T);
    TapOffsets taps{};
    for (int t = 0; t < T; ++t) taps.off[t] = tap_off[t];
    const long long total = (long long)O * T * I;
    launch_pdl(unpack_wgrad_kernel, nblk(total, 256), 256, 0, as_stream(stream), src, dst, O, T, I, so, si, taps, accumulate);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_colsum(const void* x, float* out, long long M, int C, int accumulate, void* stream) {
    CESM_REQUIRE(C % 8 == 0 && C <= 2048 && 2048 % C == 0, "colsum needs C dividing 2048 (C=%d)", C);
    cudaStream_t st = as_stream(stream);
    if (!accumulate) CESM_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * C, st));
    long long blocks = (M + 255) / 256;
    if (blocks > 148 * 4) blocks = 148 * 4;
    if (blocks < 1) blocks = 1;
    launch_pdl(colsum_kernel, (int)blocks, 256, 0, st, (const h16*)x, out, M, C);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_gather_windows(const float* cond, const float* tgt, const int* plan, float* cond_out, float* x0_out,
                                   int B, int T, int M, int H, int W, int K, int h, int w, void* stream) {
    CESM_REQUIRE(B > 0 && K >= 1 && h > 0 && w > 0 && h <= H && w <= W && T >= K, "bad window shape");
    const long long total = (long long)B * (K + 1) * h * w;
    launch_pdl(gather_windows_kernel, nblk(total, 256), 256, 0, as_stream(stream), cond, tgt, plan, cond_out, x0_out, M, H,
               W, K, h, w, total);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_input_patches_masked(const float* in0, const float* in1, int f0, int f1, const float* keep, void* out,
                                         int B, int F, int H, int W, int ks, int kpad, void* stream) {
    CESM_REQUIRE(ks == 7 && kpad == 256, "input patch kernel is specialised for 7x7, 256 columns (ks=%d kpad=%d)", ks, kpad);
    CESM_REQUIRE((f0 == 1 || f0 == F) && (f1 == 1 || f1 == F), "frame counts must be 1 or F");
    dim3 grid(ceil_div(W, 16), ceil_div(H, 16), B * F);
    launch_pdl(input_patches_kernel<7, 256>, grid, 256, 0, as_stream(stream), in0, in1, f0, f1, keep, (h16*)out, F, H,
               W);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_input_patches(const float* in0, const float* in1, int f0, int f1, void* out, int B, int F, int H,
                                  int W, int ks, int kpad, void* stream) {
    return cesm_input_patches_masked(in0, in1, f0, f1, nullptr, out, B, F, H, W, ks, kpad, stream);
}

extern "C" int cesm_input_weight_pack(const float* w, const float* bias, void* out, int cout, int ks, int kpad,
                                      void* stream) {
    CESM_REQUIRE(kpad >= 4 * ks * ks + 2, "kpad=%d too small for 2 planes x hi/lo x %dx%d + 2", kpad, ks, ks);
    launch_pdl(input_weight_pack_kernel, nblk((long long)cout * kpad, 256), 256, 0, as_stream(stream), 
        w, bias, (h16*)out, cout, 2 * ks * ks, kpad);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_input_conv_fwd(const float* in0, const float* in1, int f0, int f1, const float* w,
                                   const float* bias, void* out, int B, int F, int H, int W, int ks, int cout,
                                   void* stream) {
    CESM_REQUIRE(ks == 7 && cout == 64, "input conv kernel is specialised for 7x7, 64 channels (ks=%d cout=%d)", ks, cout);
    CESM_REQUIRE((f0 == 1 || f0 == F) && (f1 == 1 || f1 == F), "frame counts must be 1 or F");
    dim3 grid(ceil_div(W, 16), ceil_div(H, 16), B * F);
    launch_pdl(input_conv_fwd_kernel<7, 64>, grid, 256, 0, as_stream(stream), in0, in1, f0, f1, w, bias, (h16*)out, F, H, W);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_input_conv_wgrad(const float* in0, const float* in1, int f0, int f1, const void* dy, float* dw,
                                     float* db, int B, int F, int H, int W, int ks, int cout, void* stream) {
    CESM_REQUIRE(ks == 7 && cout == 64, "input conv kernel is specialised for 7x7, 64 channels (ks=%d cout=%d)", ks, cout);
    cudaStream_t st = as_stream(stream);
    CESM_CHECK_CUDA(cudaMemsetAsync(dw, 0, sizeof(float) * cout * 2 * ks * ks, st));
    CESM_CHECK_CUDA(cudaMemsetAsync(db, 0, sizeof(float) * cout, st));
    const int ntiles = ceil_div(W, 16) * ceil_div(H, 16) * B * F;
    const int grid = ntiles < 148 * 2 ? ntiles : 148 * 2;
    launch_pdl(input_conv_wgrad_kernel<7, 64>, grid, 256, 0, st, in0, in1, f0, f1, (const h16*)dy, dw, db, B * F, F, H, W);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

template <bool DX, bool DC>
static int launch_input_conv_dgrad(const void* dy, const float* w, float* dx, float* dc, const float* keep, int f0,
                                   int f1, int B, int F, int H, int W, float scale, int accumulate, cudaStream_t st) {
    auto kern = input_conv_dgrad_kernel<7, 64, DX, DC>;
    constexpr size_t smem = InputDgradSmem<7, 64>::BYTES;
    static bool attr_set = false;
    if (!attr_set) {
        CESM_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    dim3 grid(ceil_div(W, 16), ceil_div(H, 16), B);
    launch_pdl(kern, grid, 256, smem, st, (const h16*)dy, w, dx, dc, keep, f0, f1, F, H, W, scale, accumulate);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_input_conv_dgrad_masked(const void* dy, const float* w, float* d_in0, float* d_in1, const float* keep,
                                            int f0, int f1, int B, int F, int H, int W, int ks, int cout, float scale,
                                            int accumulate, void* stream) {
    CESM_REQUIRE(ks == 7 && cout == 64, "input conv kernel is specialised for 7x7, 64 channels (ks=%d cout=%d)", ks, cout);
    CESM_REQUIRE(B > 0 && B <= 65535 && F > 0 && H > 0 && W > 0, "bad input conv dgrad shape (B=%d F=%d H=%d W=%d)", B, F,
                 H, W);
    CESM_REQUIRE((f0 == 1 || f0 == F) && (f1 == 1 || f1 == F), "frame counts must be 1 or F");
    CESM_REQUIRE(dy && w && (d_in0 || d_in1), "input conv dgrad needs dy, w and at least one output");
    cudaStream_t st = as_stream(stream);
    if (d_in0 && d_in1)
        return launch_input_conv_dgrad<true, true>(dy, w, d_in0, d_in1, keep, f0, f1, B, F, H, W, scale, accumulate, st);
    if (d_in0)
        return launch_input_conv_dgrad<true, false>(dy, w, d_in0, d_in1, keep, f0, f1, B, F, H, W, scale, accumulate, st);
    return launch_input_conv_dgrad<false, true>(dy, w, d_in0, d_in1, keep, f0, f1, B, F, H, W, scale, accumulate, st);
}

extern "C" int cesm_input_conv_dgrad(const void* dy, const float* w, float* d_in0, float* d_in1, int f0, int f1, int B,
                                     int F, int H, int W, int ks, int cout, float scale, int accumulate, void* stream) {
    return cesm_input_conv_dgrad_masked(dy, w, d_in0, d_in1, nullptr, f0, f1, B, F, H, W, ks, cout, scale, accumulate,
                                        stream);
}

extern "C" int cesm_out_conv_fwd(const void* a, const float* w, const float* bias, float* eps, int B, int F, int mid,
                                 long long HW, int C, void* stream) {
    CESM_REQUIRE(C == 64, "output conv kernel needs 64 input channels (C=%d)", C);
    const long long threads = (long long)B * HW * 8;
    launch_pdl(out_conv_fwd_kernel, nblk(threads, 256), 256, 0, as_stream(stream), (const h16*)a, w, bias, eps, B, F, mid, HW);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_out_conv_bwd(const void* a, const float* w, const float* deps, void* da, float* dw, float* db,
                                 int B, int F, int mid, long long HW, int C, void* stream) {
    CESM_REQUIRE(C == 64, "output conv kernel needs 64 input channels (C=%d)", C);
    cudaStream_t st = as_stream(stream);
    CESM_CHECK_CUDA(cudaMemsetAsync(dw, 0, sizeof(float) * C, st));
    CESM_CHECK_CUDA(cudaMemsetAsync(db, 0, sizeof(float), st));
    long long blocks = ((long long)B * F * HW * 8 + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    launch_pdl(out_conv_bwd_kernel, (int)blocks, 256, 0, st, (const h16*)a, w, deps, (h16*)da, dw, db, B, F, mid, HW);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_sinusoidal(const long long* t, float* out, int B, int dim, void* stream) {
    CESM_REQUIRE(dim >= 4 && dim % 2 == 0, "dim=%d must be even and >= 4", dim);
    launch_pdl(sinusoidal_kernel, nblk((long long)B * dim, 128), 128, 0, as_stream(stream), t, out, B, dim);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_small_linear_fwd(const float* x, const float* W, const float* bias, float* y, int B, int K, int N,
                                     int act_silu_in, void* stream) {
    launch_pdl(small_linear_fwd_kernel, dim3(ceil_div(N, 8), B < 64 ? B : 64), 256, 0, as_stream(stream), x, W, bias, y, B, K, N,
                                                                                              act_silu_in);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_small_linear_bwd(const float* x, const float* W, const float* dy, float* dx, float* dW, float* db,
                                     int B, int K, int N, int act_silu_in, int accumulate, void* stream) {
    cudaStream_t st = as_stream(stream);
    launch_pdl(small_linear_wgrad_kernel, nblk((long long)N * K, 256), 256, 0, st, x, dy, dW, db, B, K, N, act_silu_in,
                                                                           accumulate);
    CESM_CHECK_LAUNCH();
    if (dx) {
        launch_pdl(small_linear_dgrad_kernel, dim3(ceil_div(K, 32), B), 256, 0, st, x, W, dy, dx, B, K, N, act_silu_in);
        CESM_CHECK_LAUNCH();
    }
    return CESM_OK;
}

extern "C" int cesm_film_fwd(const float* x, const cesm_film_desc* layers_device, float* y, int n_layers, int n_total,
                             int B, int K, void* stream) {
    CESM_REQUIRE(n_layers > 0 && n_total > 0 && B > 0 && K > 0, "bad FiLM table");
    launch_pdl(film_fwd_kernel, dim3(ceil_div(n_total, 8), B), 256, 0, as_stream(stream), x, layers_device, y, n_layers,
               n_total, B, K);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_film_bwd(const float* x, const cesm_film_desc* layers_device, const float* dy, int n_layers,
                             int n_total, float* dx, int B, int K, int accumulate, void* stream) {
    CESM_REQUIRE(n_layers > 0 && n_total > 0 && B > 0 && K > 0, "bad FiLM table");
    cudaStream_t st = as_stream(stream);
    launch_pdl(film_wgrad_kernel, nblk((long long)n_total * K, 256), 256, 0, st, x, layers_device, dy, n_layers, n_total, B,
               K, accumulate);
    CESM_CHECK_LAUNCH();
    if (dx) {
        CESM_ZERO_SCRATCH(dx, sizeof(float) * (size_t)B * K, st);
        launch_pdl(film_dgrad_kernel, dim3(ceil_div(K, 32), B, n_layers), 256, 0, st, x, layers_device, dy, n_layers, dx, B, K);
        CESM_CHECK_LAUNCH();
    }
    return CESM_OK;
}

extern "C" int cesm_q_sample(const float* x0, const float* noise, const long long* t, const float* sqrt_ac,
                             const float* sqrt_1mac, float* xt, int B, long long per_sample, void* stream) {
    const long long total = (long long)B * per_sample;
    launch_pdl(q_sample_kernel, nblk(total, 256), 256, 0, as_stream(stream), x0, noise, t, sqrt_ac, sqrt_1mac, xt, per_sample, total);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_q_sample_bwd(const float* g, const long long* t, const float* sqrt_ac, const float* sqrt_1mac,
                                 float* dx0, float* dnoise, int B, long long per_sample, void* stream) {
    CESM_REQUIRE(B > 0 && per_sample > 0, "bad q_sample backward sizes (B=%d per_sample=%lld)", B, per_sample);
    CESM_REQUIRE(g && t && sqrt_ac && sqrt_1mac && (dx0 || dnoise),
                 "q_sample backward needs g, t, both schedule tables and at least one output");
    const long long total = (long long)B * per_sample;
    launch_pdl(q_sample_bwd_kernel, nblk(total, 256), 256, 0, as_stream(stream), g, t, sqrt_ac, sqrt_1mac, dx0, dnoise,
               per_sample, total);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_mse_fwd(const float* eps, const float* noise, float* diff, float* loss, long long total,
                            void* stream) {
    cudaStream_t st = as_stream(stream);
    CESM_CHECK_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), st));
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 4) blocks = 148 * 4;
    launch_pdl(mse_fwd_kernel, (int)blocks, 256, 0, st, eps, noise, diff, loss, total);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_diffusion_loss_fwd(const float* pred, const float* x0, const float* noise, const long long* t,
                                       const float* tgt_coef, const float* weight, float* diff, float* loss, int B,
                                       long long per_sample, int T, void* stream) {
    CESM_REQUIRE(T > 0 && B > 0 && B <= 65535 && per_sample > 0, "bad diffusion loss sizes (T=%d B=%d per_sample=%lld)",
                 T, B, per_sample);
    CESM_REQUIRE(pred && noise && t && diff && loss && (x0 || !tgt_coef),
                 "diffusion loss needs pred, noise, t, diff, loss, and x0 with a target table");
    cudaStream_t st = as_stream(stream);
    CESM_CHECK_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), st));
    long long bx = (per_sample + 255) / 256;
    const long long cap = (148 * 4 + B - 1) / B;  // about as many blocks in all as cesm_mse_fwd
    if (bx > cap) bx = cap;
    launch_pdl(diffusion_loss_fwd_kernel, dim3((unsigned)bx, B), 256, 0, st, pred, x0, noise, t, tgt_coef, weight, diff,
               loss, T, per_sample, (long long)B * per_sample);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_diffusion_loss_bwd(const float* diff, const long long* t, const float* tgt_coef, const float* weight,
                                       const float* gscale, float factor, float* dpred, float* dnoise, float* dx0, int B,
                                       long long per_sample, int T, void* stream) {
    CESM_REQUIRE(T > 0 && B > 0 && B <= 65535 && per_sample > 0, "bad diffusion loss backward sizes (T=%d B=%d per_sample=%lld)",
                 T, B, per_sample);
    CESM_REQUIRE(diff && t && gscale && (dpred || dnoise || dx0),
                 "diffusion loss backward needs diff, t, gscale and at least one output");
    launch_pdl(diffusion_loss_bwd_kernel, dim3((unsigned)((per_sample + 255) / 256), B), 256, 0, as_stream(stream), diff, t,
               tgt_coef, weight, gscale, factor, dpred, dnoise, dx0, T, per_sample);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_scale_by_scalar(const float* in, const float* gscale, float factor, float* out, long long total,
                                    void* stream) {
    launch_pdl(scale_by_device_scalar_kernel, nblk(total, 256), 256, 0, as_stream(stream), in, gscale, factor, out, total);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_p_sample(const float* xt, const float* eps, const float* z, const long long* t, const float* betas,
                             const float* sqrt_1mac, const float* sqrt_recip_a, const float* post_var, float* out,
                             int B, long long per_sample, void* stream) {
    const long long total = (long long)B * per_sample;
    launch_pdl(p_sample_kernel<false>, nblk(total, 256), 256, 0, as_stream(stream), xt, eps, z, t, betas, sqrt_1mac,
               sqrt_recip_a, post_var, out, per_sample, total, 0.0f);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

// The guided entries take the 2B-row network output (conditional rows, then null-condition rows) and a finite w > 0.
#define CESM_REQUIRE_GUIDANCE(what)                                                                              \
    CESM_REQUIRE(isfinite(guidance) && guidance > 0.0f, what " needs a finite guidance weight > 0 (got %g)",      \
                 (double)guidance)

extern "C" int cesm_p_sample_guided(const float* xt, const float* eps, const float* z, const long long* t,
                                    const float* betas, const float* sqrt_1mac, const float* sqrt_recip_a,
                                    const float* post_var, float* out, int B, long long per_sample, float guidance,
                                    void* stream) {
    CESM_REQUIRE(B > 0 && per_sample > 0, "bad guided p_sample sizes (B=%d per_sample=%lld)", B, per_sample);
    CESM_REQUIRE(xt && eps && z && t && betas && sqrt_1mac && sqrt_recip_a && post_var && out,
                 "guided p_sample needs xt, eps, z, t, the four schedule tables and out");
    CESM_REQUIRE_GUIDANCE("guided p_sample");
    const long long total = (long long)B * per_sample;
    launch_pdl(p_sample_kernel<true>, nblk(total, 256), 256, 0, as_stream(stream), xt, eps, z, t, betas, sqrt_1mac,
               sqrt_recip_a, post_var, out, per_sample, total, guidance);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

template <bool kGuided>
static int launch_ddim_step(const float* xt, const float* eps, const float* z, const long long* t, const float* coef,
                            const long long* next_t, long long* t_out, float* out, int T, int B, long long per_sample,
                            float w, void* stream) {
    CESM_REQUIRE(T > 0 && B > 0 && per_sample > 0, "bad DDIM step sizes (T=%d B=%d per_sample=%lld)", T, B, per_sample);
    CESM_REQUIRE(xt && eps && t && coef && out, "DDIM step needs xt, eps, t, coef and out");
    CESM_REQUIRE(!t_out || next_t, "t_out needs the next_t table");
    CESM_REQUIRE(!t_out || (const void*)t_out != (const void*)t, "t_out must not alias t");
    const long long total = (long long)B * per_sample;
    launch_pdl(ddim_step_kernel<kGuided>, nblk(total, 256), 256, 0, as_stream(stream), xt, eps, z, t, coef, next_t, t_out,
               out, T, per_sample, total, w);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_ddim_step(const float* xt, const float* eps, const float* z, const long long* t, const float* coef,
                              const long long* next_t, long long* t_out, float* out, int T, int B, long long per_sample,
                              void* stream) {
    return launch_ddim_step<false>(xt, eps, z, t, coef, next_t, t_out, out, T, B, per_sample, 0.0f, stream);
}

extern "C" int cesm_ddim_step_guided(const float* xt, const float* eps, const float* z, const long long* t,
                                     const float* coef, const long long* next_t, long long* t_out, float* out, int T,
                                     int B, long long per_sample, float guidance, void* stream) {
    CESM_REQUIRE_GUIDANCE("guided DDIM step");
    return launch_ddim_step<true>(xt, eps, z, t, coef, next_t, t_out, out, T, B, per_sample, guidance, stream);
}

// True when the byte ranges [a, a + na) and [b, b + nb) share a byte (a null b shares none).
static bool ranges_overlap(const void* a, size_t na, const void* b, size_t nb) {
    const char *pa = (const char*)a, *pb = (const char*)b;
    return pb && pa < pb + nb && pb < pa + na;
}

template <bool kGuided>
static int launch_dpm_step(const float* xt, const float* eps, float* hist, const long long* t, const float* coef,
                           const long long* next_t, long long* t_out, float* out, int T, int B, long long per_sample,
                           float w, void* stream) {
    CESM_REQUIRE(T > 0 && B > 0 && per_sample > 0, "bad DPM step sizes (T=%d B=%d per_sample=%lld)", T, B, per_sample);
    CESM_REQUIRE(xt && eps && hist && t && coef && out, "DPM step needs xt, eps, hist, t, coef and out");
    CESM_REQUIRE(!t_out || next_t, "t_out needs the next_t table");
    CESM_REQUIRE(!t_out || (const void*)t_out != (const void*)t, "t_out must not alias t");
    const long long total = (long long)B * per_sample;
    const size_t field = (size_t)total * sizeof(float), tb = (size_t)B * sizeof(long long);
    CESM_REQUIRE(!ranges_overlap(hist, field, xt, field) && !ranges_overlap(hist, field, eps, (kGuided ? 2 : 1) * field) &&
                     !ranges_overlap(hist, field, out, field) && !ranges_overlap(hist, field, t, tb) &&
                     !ranges_overlap(hist, field, t_out, tb) &&
                     !ranges_overlap(hist, field, coef, (size_t)T * 5 * sizeof(float)) &&
                     !ranges_overlap(hist, field, next_t, (size_t)T * sizeof(long long)),
                 "hist must not overlap xt, eps, out, t, t_out, coef or next_t");
    launch_pdl(dpm_step_kernel<kGuided>, nblk(total, 256), 256, 0, as_stream(stream), xt, eps, hist, t, coef, next_t,
               t_out, out, T, per_sample, total, w);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_dpm_step(const float* xt, const float* eps, float* hist, const long long* t, const float* coef,
                             const long long* next_t, long long* t_out, float* out, int T, int B, long long per_sample,
                             void* stream) {
    return launch_dpm_step<false>(xt, eps, hist, t, coef, next_t, t_out, out, T, B, per_sample, 0.0f, stream);
}

extern "C" int cesm_dpm_step_guided(const float* xt, const float* eps, float* hist, const long long* t,
                                    const float* coef, const long long* next_t, long long* t_out, float* out, int T,
                                    int B, long long per_sample, float guidance, void* stream) {
    CESM_REQUIRE_GUIDANCE("guided DPM step");
    return launch_dpm_step<true>(xt, eps, hist, t, coef, next_t, t_out, out, T, B, per_sample, guidance, stream);
}

// Seeded sampling noise: one thread per quad of a field, grid.y = field row.  The element index inside a field is
// the Philox counter's first word after >> 2, so a field may hold up to 2^34 elements.
static bool quads_aligned(long long per, const void* a, const void* b = nullptr, const void* c = nullptr) {
    const auto al = [](const void* p) { return ((uintptr_t)p & 15) == 0; };
    return per % 4 == 0 && al(a) && al(b) && al(c);
}
static dim3 quad_grid(int B, long long per) { return dim3((unsigned)nblk((per + 3) / 4, 256), (unsigned)B); }
#define CESM_REQUIRE_SEEDED_SIZES(what)                                                                          \
    CESM_REQUIRE(B > 0 && B <= 65535 && per_sample > 0 && per_sample <= (1LL << 34),                             \
                 what " needs 0 < B <= 65535 and 0 < per_sample <= 2^34 (B=%d per_sample=%lld)", B, per_sample)

extern "C" int cesm_field_normal(unsigned seed_lo, unsigned seed_hi, const long long* field_ids, unsigned draw,
                                 float* out, int B, long long per_sample, void* stream) {
    CESM_REQUIRE_SEEDED_SIZES("field_normal");
    CESM_REQUIRE(field_ids && out, "field_normal needs field_ids and out");
    const dim3 grid = quad_grid(B, per_sample);
    if (quads_aligned(per_sample, out))
        launch_pdl(field_normal_kernel<true>, grid, 256, 0, as_stream(stream), seed_lo, seed_hi, field_ids, draw, out,
                   per_sample);
    else
        launch_pdl(field_normal_kernel<false>, grid, 256, 0, as_stream(stream), seed_lo, seed_hi, field_ids, draw, out,
                   per_sample);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

template <bool kGuided>
static int launch_p_sample_seeded(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                                  const long long* field_ids, const long long* t, const float* betas,
                                  const float* sqrt_1mac, const float* sqrt_recip_a, const float* post_var, float* out,
                                  int T, int B, long long per_sample, float w, void* stream) {
    CESM_REQUIRE_SEEDED_SIZES("seeded p_sample");
    CESM_REQUIRE(T > 0, "seeded p_sample needs T > 0 (T=%d)", T);
    CESM_REQUIRE(xt && eps && field_ids && t && betas && sqrt_1mac && sqrt_recip_a && post_var && out,
                 "seeded p_sample needs xt, eps, field_ids, t, the four schedule tables and out");
    const dim3 grid = quad_grid(B, per_sample);
    if (quads_aligned(per_sample, xt, eps, out))
        launch_pdl(p_sample_seeded_kernel<true, kGuided>, grid, 256, 0, as_stream(stream), xt, eps, seed_lo, seed_hi,
                   field_ids, t, betas, sqrt_1mac, sqrt_recip_a, post_var, out, T, per_sample, w);
    else
        launch_pdl(p_sample_seeded_kernel<false, kGuided>, grid, 256, 0, as_stream(stream), xt, eps, seed_lo, seed_hi,
                   field_ids, t, betas, sqrt_1mac, sqrt_recip_a, post_var, out, T, per_sample, w);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_p_sample_seeded(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                                    const long long* field_ids, const long long* t, const float* betas,
                                    const float* sqrt_1mac, const float* sqrt_recip_a, const float* post_var,
                                    float* out, int T, int B, long long per_sample, void* stream) {
    return launch_p_sample_seeded<false>(xt, eps, seed_lo, seed_hi, field_ids, t, betas, sqrt_1mac, sqrt_recip_a,
                                         post_var, out, T, B, per_sample, 0.0f, stream);
}

extern "C" int cesm_p_sample_seeded_guided(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                                           const long long* field_ids, const long long* t, const float* betas,
                                           const float* sqrt_1mac, const float* sqrt_recip_a, const float* post_var,
                                           float* out, int T, int B, long long per_sample, float guidance,
                                           void* stream) {
    CESM_REQUIRE_GUIDANCE("guided seeded p_sample");
    return launch_p_sample_seeded<true>(xt, eps, seed_lo, seed_hi, field_ids, t, betas, sqrt_1mac, sqrt_recip_a,
                                        post_var, out, T, B, per_sample, guidance, stream);
}

template <bool kGuided>
static int launch_ddim_step_seeded(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                                   const long long* field_ids, const long long* t, const float* coef,
                                   const long long* next_t, long long* t_out, float* out, int T, int B,
                                   long long per_sample, float w, void* stream) {
    CESM_REQUIRE_SEEDED_SIZES("seeded DDIM step");
    CESM_REQUIRE(T > 0, "seeded DDIM step needs T > 0 (T=%d)", T);
    CESM_REQUIRE(xt && eps && field_ids && t && coef && out, "seeded DDIM step needs xt, eps, field_ids, t, coef and out");
    CESM_REQUIRE(!t_out || next_t, "t_out needs the next_t table");
    CESM_REQUIRE(!t_out || ((const void*)t_out != (const void*)t && (const void*)t_out != (const void*)field_ids),
                 "t_out must not alias t or field_ids");
    const dim3 grid = quad_grid(B, per_sample);
    if (quads_aligned(per_sample, xt, eps, out))
        launch_pdl(ddim_step_seeded_kernel<true, kGuided>, grid, 256, 0, as_stream(stream), xt, eps, seed_lo, seed_hi,
                   field_ids, t, coef, next_t, t_out, out, T, per_sample, w);
    else
        launch_pdl(ddim_step_seeded_kernel<false, kGuided>, grid, 256, 0, as_stream(stream), xt, eps, seed_lo, seed_hi,
                   field_ids, t, coef, next_t, t_out, out, T, per_sample, w);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_ddim_step_seeded(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                                     const long long* field_ids, const long long* t, const float* coef,
                                     const long long* next_t, long long* t_out, float* out, int T, int B,
                                     long long per_sample, void* stream) {
    return launch_ddim_step_seeded<false>(xt, eps, seed_lo, seed_hi, field_ids, t, coef, next_t, t_out, out, T, B,
                                          per_sample, 0.0f, stream);
}

extern "C" int cesm_ddim_step_seeded_guided(const float* xt, const float* eps, unsigned seed_lo, unsigned seed_hi,
                                            const long long* field_ids, const long long* t, const float* coef,
                                            const long long* next_t, long long* t_out, float* out, int T, int B,
                                            long long per_sample, float guidance, void* stream) {
    CESM_REQUIRE_GUIDANCE("guided seeded DDIM step");
    return launch_ddim_step_seeded<true>(xt, eps, seed_lo, seed_hi, field_ids, t, coef, next_t, t_out, out, T, B,
                                         per_sample, guidance, stream);
}

extern "C" int cesm_cond_keep(unsigned seed_lo, unsigned seed_hi, long long* step, long long first, float p, float* keep,
                              int B, void* stream) {
    CESM_REQUIRE(B > 0 && first >= 0, "bad condition-dropout sizes (B=%d first=%lld)", B, first);
    CESM_REQUIRE(step && keep, "condition dropout needs the step counter and the keep buffer");
    CESM_REQUIRE(p >= 0.0f && p < 1.0f, "condition dropout probability must be in [0, 1) (got %g)", (double)p);
    launch_pdl(cond_keep_kernel, 1, 256, 0, as_stream(stream), seed_lo, seed_hi, step, first, p, keep, B);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}
