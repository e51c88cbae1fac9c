// Optimizer-step kernels (train.py:864-867, 1078-1083): everything between "gradients are final" and
// "the next forward can start" is four bandwidth-bound launches over flat fp32 buffers:
//
//   relayout_tiled<1>  packed fp32 weight-gradient scratch [O][T][I] -> += parameter-gradient layout
//   grad_sumsq         per-block partial sums of g^2 (deterministic order)
//   adamw_clip         loss-scale removal + inf check + global-norm clip + AdamW on (p, g, m, v), all parameters
//   scaler_update      GradScaler.update(): step count, loss-scale backoff / growth (one warp)
//   relayout_tiled<0>  fp32 parameters -> fp16 GEMM-operand copies [O][T][I]
//
// The two re-layouts are 3-D permutations (conv weight [co][ci][tap] <-> operand [o][tap][i] with
// (o, i) = (co, ci) or (ci, co)); they go through a shared-memory tile so that both the parameter
// side (runs of 32 x T' contiguous floats) and the packed side (32 contiguous elements) are coalesced.
#include "api_common.h"
#include "common.cuh"

namespace cesm {

static constexpr int kRelayoutThreads = 256;
static constexpr int kTile = 32;
static constexpr int kRelayoutSmem = kTile * (kTile * 9 + 1) * (int)sizeof(float);  // 32 rows x 9 taps; 16 rows x 16 taps

__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// MODE 0: dst (fp16 [O][T][I]) = src[o*so + i*si + tap_off[t]]                      (pack)
// MODE 1: dst[o*so + i*si + tap_off[t]] += src (fp32 [O][T][I]); src = 0             (un-pack)
// Requires min(so, si) = T' >= 1 (the parameter's own tap count), tap_off[t] in [0, T'), T' <= 16.
// A tile is (rows of the outer index) x (32 of the inner index) x (all T' taps): each row is one
// contiguous run of 32*T' floats on the parameter side, fetched with cp.async so that the whole tile
// is in flight at once; the packed side is written / read 32 contiguous elements at a time.
template <int MODE>
__global__ void __launch_bounds__(kRelayoutThreads)
relayout_tiled_kernel(const cesm_pack_desc* __restrict__ descs) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ float tile[];
    __shared__ int s_off[CESM_MAX_TAPS];
    const cesm_pack_desc& d = descs[blockIdx.y];
    const long long so = d.so, si = d.si;
    const int O = d.O, T = d.T, I = d.I;
    const bool inner_is_i = si < so;
    const long long s_in = inner_is_i ? si : so, s_out = inner_is_i ? so : si;
    const int n_in = inner_is_i ? I : O, n_out = inner_is_i ? O : I;
    const int Tp = (int)s_in;
    const int rows = Tp > 9 ? kTile / 2 : kTile;  // keeps the tile within kRelayoutSmem
    const int pitch = kTile * Tp + 1;
    const int tiles_in = (n_in + kTile - 1) / kTile, tiles_out = (n_out + rows - 1) / rows;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t covered = 0;
    for (int t = 0; t < T; ++t) {
        const int o = d.tap_off[t];
        covered |= 1u << o;
        if (threadIdx.x == 0) s_off[t] = o;
    }
    // parameter-layout side (fp32) and packed side
    float* __restrict__ par = MODE == 0 ? const_cast<float*>(d.src) : reinterpret_cast<float*>(d.dst);
    h16* __restrict__ pk16 = reinterpret_cast<h16*>(d.dst);       // MODE 0
    float* __restrict__ pk32 = const_cast<float*>(d.src);                            // MODE 1
    const uint32_t tile_addr = smem_u32(tile);
    for (int tl = blockIdx.x; tl < tiles_in * tiles_out; tl += gridDim.x) {
        const int in0 = (tl % tiles_in) * kTile, out0 = (tl / tiles_in) * rows;
        const int nin = min(kTile, n_in - in0), nout = min(rows, n_out - out0);
        const int run = nin * Tp;
        __syncthreads();  // previous tile fully consumed (and s_off visible)
        for (int r = warp; r < nout; r += kRelayoutThreads / 32) {
            const float* g = par + (long long)(out0 + r) * s_out + (long long)in0 * s_in;
            const uint32_t row_addr = tile_addr + (uint32_t)(r * pitch) * 4u;
            for (int pos = lane; pos < run; pos += 32) cp_async4(row_addr + pos * 4u, g + pos);
        }
        cp_async_wait_all();
        __syncthreads();
        // packed side: (o_l, t, i_l), i_l fastest; one warp-row per (o_l, t)
        const int n_il = inner_is_i ? nin : nout, n_ol = inner_is_i ? nout : nin;
        const int i_g = (inner_is_i ? in0 : out0) + lane;
        const bool act = lane < n_il;
#pragma unroll 4
        for (int rest = warp; rest < n_ol * T; rest += kRelayoutThreads / 32) {
            const int o_l = rest / T, t = rest - o_l * T;
            const int outer_l = inner_is_i ? o_l : lane, inner_l = inner_is_i ? lane : o_l;
            const int sp = outer_l * pitch + inner_l * Tp + s_off[t];
            const int o_g = (inner_is_i ? out0 : in0) + o_l;
            const long long q = ((long long)o_g * T + t) * I + i_g;
            if (act) {
                if (MODE == 0) {
                    pk16[q] = __float2half_rn(tile[sp]);
                } else {
                    tile[sp] += pk32[q];
                    pk32[q] = 0.f;
                }
            }
        }
        if (MODE == 1) {
            __syncthreads();
            for (int r = warp; r < nout; r += kRelayoutThreads / 32) {
                float* g = par + (long long)(out0 + r) * s_out + (long long)in0 * s_in;
                int tap = lane % Tp;  // pos % Tp, advanced incrementally (32 % Tp per trip)
                const int adv = 32 % Tp;
                for (int pos = lane; pos < run; pos += 32) {
                    if ((covered >> tap) & 1u) g[pos] = tile[r * pitch + pos];
                    tap += adv;
                    if (tap >= Tp) tap -= Tp;
                }
            }
        }
    }
}

// ---- global gradient norm: per-block partials in a fixed order (bit-reproducible run to run) ----
static constexpr int kOptThreads = 256;
__global__ void __launch_bounds__(kOptThreads)
grad_sumsq_kernel(const float* __restrict__ g, long long n, float* __restrict__ partials, float* __restrict__ state) {
    pdl_trigger();
    pdl_wait();
    float s = 0.f;
    const long long n4 = n >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    for (long long i = (long long)blockIdx.x * kOptThreads + threadIdx.x; i < n4; i += (long long)gridDim.x * kOptThreads) {
        const float4 v = g4[i];
        s = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, s))));
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const float v = g[(n4 << 2) + threadIdx.x];
        s = fmaf(v, v, s);
    }
    __shared__ float red[kOptThreads / 32];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < kOptThreads / 32; ++i) t += red[i];
        partials[blockIdx.x] = t;
    }
}

// Optimizer state vector (fp32, on the device so that a replayed CUDA graph sees every change):
//   [0] step count   [1] last gradient norm (unscaled, before clipping)   [2] loss scale S
//   [3] growth tracker   [4] found_inf of the last step   [5] number of skipped steps
//   [6] learning rate   [7] weight decay   [8] growth interval (0 = static scale)
// AdamW exactly as torch.optim.AdamW (decoupled decay, bias correction, eps outside the sqrt), with
// torch.amp.GradScaler's unscale / inf check / skip (train.py:862-867) and the global-norm clip coefficient
// min(1, max_norm / (|g| + 1e-6)) (torch.nn.utils.clip_grad_norm_, train.py:865) folded in: the gradients in
// `g` are S times the true ones; a non-finite sum of squares means some gradient overflowed fp16 -> the step
// is skipped (parameters and moments untouched) and scaler_update_kernel backs S off.
// kEma: also the exponential moving average `ema` of the updated parameters, in the same pass -- a copy e = p while
// the step count after this step is <= ema_start, else e += ema_w (p - e) with ema_w = 1 - decay.  A skipped step
// returns before it.  The EMA arguments come last so that the kEma = false instance keeps the parameter layout (and
// the code) of the kernel without them.  Left alone, ptxas gives the kEma = true instance 52 registers (4 blocks of
// 256 per SM); the minimum of 5 blocks holds it at the 48 registers and 5 blocks of the false instance, without
// spills.  0 leaves the false instance unconstrained, as it was.
template <bool kEma>
__global__ void __launch_bounds__(kOptThreads, kEma ? 5 : 0)
adamw_clip_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                  long long n, const float* __restrict__ partials, int n_partials, float* __restrict__ state,
                  float beta1, float beta2, float eps, float max_norm, float* __restrict__ ema, float ema_w,
                  long long ema_start) {
    pdl_trigger();
    pdl_wait();
    __shared__ float s_coef;
    __shared__ int s_skip;
    if (threadIdx.x < 32) {  // every block re-reduces the partials in the same order
        float t = 0.f;
        for (int i = threadIdx.x; i < n_partials; i += 32) t += partials[i];
        t = warp_sum(t);
        if (threadIdx.x == 0) {
            const float inv_scale = 1.f / state[2];
            const float norm = sqrtf(t) * inv_scale;
            s_skip = !isfinite(t);
            s_coef = (max_norm > 0.f ? fminf(1.f, max_norm / (norm + 1e-6f)) : 1.f) * inv_scale;
            if (blockIdx.x == 0) state[1] = norm;
        }
    }
    __syncthreads();
    if (s_skip) return;
    const float coef = s_coef;
    const float step = state[0] + 1.f;  // scaler_update_kernel commits the increment after this kernel
    const float lr = state[6], wd = state[7];
    const float bc1 = 1.f - powf(beta1, step), bc2 = 1.f - powf(beta2, step);
    const float step_size = lr / bc1, inv_bc2_sqrt = rsqrtf(bc2), decay = 1.f - lr * wd;
    const long long n4 = n >> 2;
    float4* p4 = reinterpret_cast<float4*>(p);
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    auto upd = [&](float& pp, float gg, float& mm, float& vv) {
        gg *= coef;
        pp *= decay;
        mm = fmaf(gg - mm, 1.f - beta1, mm);
        vv = fmaf(vv, beta2, (1.f - beta2) * gg * gg);
        pp -= step_size * mm / (sqrtf(vv) * inv_bc2_sqrt + eps);
    };
    const bool ema_copy = (long long)step <= ema_start;
    float4* e4 = reinterpret_cast<float4*>(ema);
    auto ema_upd = [&](float& ee, float pp) { ee = ema_copy ? pp : fmaf(ema_w, pp - ee, ee); };
    for (long long i = (long long)blockIdx.x * kOptThreads + threadIdx.x; i < n4; i += (long long)gridDim.x * kOptThreads) {
        float4 pp = p4[i], mm = m4[i], vv = v4[i];
        const float4 gg = g4[i];
        float4 ee;
        if constexpr (kEma) ee = e4[i];
        upd(pp.x, gg.x, mm.x, vv.x);
        upd(pp.y, gg.y, mm.y, vv.y);
        upd(pp.z, gg.z, mm.z, vv.z);
        upd(pp.w, gg.w, mm.w, vv.w);
        p4[i] = pp;
        m4[i] = mm;
        v4[i] = vv;
        if constexpr (kEma) {
            ema_upd(ee.x, pp.x);
            ema_upd(ee.y, pp.y);
            ema_upd(ee.z, pp.z);
            ema_upd(ee.w, pp.w);
            e4[i] = ee;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const long long i = (n4 << 2) + threadIdx.x;
        upd(p[i], g[i], m[i], v[i]);
        if constexpr (kEma) ema_upd(ema[i], p[i]);
    }
}

// torch.amp.GradScaler.update() (backoff 0.5 on overflow, growth 2 every `growth interval` clean steps) and the
// step-count commit, one warp after the AdamW kernel has finished reading the state.
__global__ void scaler_update_kernel(const float* __restrict__ partials, int n_partials, float* __restrict__ state) {
    pdl_trigger();
    pdl_wait();
    float t = 0.f;
    for (int i = threadIdx.x; i < n_partials; i += 32) t += partials[i];
    t = warp_sum(t);
    if (threadIdx.x == 0) {
        if (!isfinite(t)) {
            state[2] = fmaxf(state[2] * 0.5f, 1.f);
            state[3] = 0.f;
            state[4] = 1.f;
            state[5] += 1.f;
        } else {
            state[0] += 1.f;
            state[4] = 0.f;
            const float interval = state[8];
            if (interval > 0.f) {
                const float tr = state[3] + 1.f;
                if (tr >= interval) {
                    state[2] = fminf(state[2] * 2.f, 16777216.f);
                    state[3] = 0.f;
                } else {
                    state[3] = tr;
                }
            }
        }
    }
}

}  // namespace cesm

using namespace cesm;

static int relayout_launch(const cesm_pack_desc* descs_device, int n, int mode, cudaStream_t st) {
    constexpr int kSmem = kRelayoutSmem;
    static bool cfg = false;
    if (!cfg) {
        CESM_CHECK_CUDA(cudaFuncSetAttribute(relayout_tiled_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
        CESM_CHECK_CUDA(cudaFuncSetAttribute(relayout_tiled_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
        cfg = true;
    }
    dim3 grid(32, n);
    if (mode == 0)
        launch_pdl(relayout_tiled_kernel<0>, grid, kRelayoutThreads, kSmem, st, descs_device);
    else
        launch_pdl(relayout_tiled_kernel<1>, grid, kRelayoutThreads, kSmem, st, descs_device);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_pack_weights_batched(const cesm_pack_desc* descs_device, int n, void* stream) {
    if (n <= 0) return CESM_OK;
    return relayout_launch(descs_device, n, 0, as_stream(stream));
}

extern "C" int cesm_unpack_wgrads_batched(const cesm_pack_desc* descs_device, int n, void* stream) {
    if (n <= 0) return CESM_OK;
    return relayout_launch(descs_device, n, 1, as_stream(stream));
}

extern "C" int cesm_adamw_partials(void) { return 148 * 4; }

// grad_sumsq -> adamw_clip<kEma> -> scaler_update: the whole optimizer step, with or without the EMA.
template <bool kEma>
static int adamw_launch(float* p, const float* g, float* m, float* v, float* ema, long long n, float* partials,
                        float* state, float beta1, float beta2, float eps, float max_norm, float ema_w,
                        long long ema_start, void* stream) {
    CESM_REQUIRE(n > 0 && (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(m) & 15) == 0 && (reinterpret_cast<uintptr_t>(v) & 15) == 0,
                 "adamw_step needs n > 0 and 16-byte aligned flat buffers (n=%lld)", n);
    cudaStream_t st = as_stream(stream);
    const int nb = cesm_adamw_partials();
    launch_pdl(grad_sumsq_kernel, nb, kOptThreads, 0, st, g, n, partials, state);
    CESM_CHECK_LAUNCH();
    launch_pdl(adamw_clip_kernel<kEma>, nb * 2, kOptThreads, 0, st, p, g, m, v, n, partials, nb, state, beta1, beta2,
               eps, max_norm, ema, ema_w, ema_start);
    CESM_CHECK_LAUNCH();
    launch_pdl(scaler_update_kernel, 1, 32, 0, st, (const float*)partials, nb, state);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

extern "C" int cesm_adamw_step(float* p, const float* g, float* m, float* v, long long n, float* partials,
                               float* state, float beta1, float beta2, float eps, float max_norm, void* stream) {
    return adamw_launch<false>(p, g, m, v, nullptr, n, partials, state, beta1, beta2, eps, max_norm, 0.f, 0, stream);
}

extern "C" int cesm_adamw_ema_step(float* p, const float* g, float* m, float* v, float* ema, long long n,
                                   float* partials, float* state, float beta1, float beta2, float eps, float max_norm,
                                   double ema_decay, long long ema_start, void* stream) {
    CESM_REQUIRE(ema != nullptr && (reinterpret_cast<uintptr_t>(ema) & 15) == 0,
                 "adamw_ema_step needs a 16-byte aligned EMA buffer");
    CESM_REQUIRE(ema_decay >= 0.0 && ema_decay < 1.0, "adamw_ema_step needs 0 <= ema_decay < 1 (got %g)", ema_decay);
    CESM_REQUIRE(ema_start >= 0, "adamw_ema_step needs ema_start >= 0 (got %lld)", ema_start);
    // 1 - decay rounded once, as torch's lerp weight in AveragedModel(get_ema_multi_avg_fn(decay))
    return adamw_launch<true>(p, g, m, v, ema, n, partials, state, beta1, beta2, eps, max_norm,
                              (float)(1.0 - ema_decay), ema_start, stream);
}
