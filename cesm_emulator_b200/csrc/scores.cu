// Ensemble scores of a generated ensemble against a target ensemble, per (year, pixel) column, in one pass:
// fair CRPS, bias, the two standard deviations, the ensemble-mean squared error and the rank histogram.
//
// A block owns C adjacent pixels of one year.  It stages the n predicted and m target values of its C columns in
// shared memory with coalesced row loads (rows of C floats, a padded stride so that a warp walking one column hits
// distinct banks), then each warp scores whole columns: bitonic sort of the column's X (n padded to a power of two
// with +inf), prefix sums of the sorted values, and one binary search per target value for its rank r.
//   sum_{i<k} |x_i - x_k| = sum_k (2k - n + 1) x_(k)        (k from 0, sorted)
//   sum_i |x_i - y|       = y (2r - n) - 2 S_r + S_n           (S_r = sum of the r smallest)
// Every sum is taken after subtracting a per-column shift (the column's middle order statistic), so the scores do not
// lose accuracy with the offset of the data.  Reductions are shuffles in a fixed order and the histogram is integer
// counts, so results are bitwise reproducible.
#include "api_common.h"
#include "common.cuh"

namespace cesm {

constexpr int kScoreWarps = 8;
constexpr int kScoreMaxMembers = 1024;

struct ScoreSmem {
    int npad, st;
    size_t xs, ys, sw, hist, bad, total;  // offsets in 4-byte words
};

__host__ __device__ inline ScoreSmem score_smem(int n, int m, int C) {
    ScoreSmem s;
    s.npad = 2;
    while (s.npad < n) s.npad <<= 1;
    s.st = C + 1;
    s.xs = 0;
    s.ys = s.xs + (size_t)s.npad * s.st;
    s.sw = s.ys + (size_t)m * s.st;
    s.hist = s.sw + (size_t)kScoreWarps * (s.npad + 1);
    s.bad = s.hist + (size_t)(n + 1);
    s.total = s.bad + C;
    return s;
}

template <int C>
__global__ void __launch_bounds__(kScoreWarps * 32) ensemble_scores_kernel(
    const float* __restrict__ pred, const float* __restrict__ target, float* __restrict__ crps,
    float* __restrict__ bias, float* __restrict__ sd_pred, float* __restrict__ sd_target,
    float* __restrict__ mse_mean, unsigned long long* __restrict__ hist, int n, int m, long long HW) {
    extern __shared__ float smem[];
    const ScoreSmem L = score_smem(n, m, C);
    const int st = L.st, npad = L.npad;
    float* xs = smem + L.xs;
    float* ys = smem + L.ys;
    int* hist_s = reinterpret_cast<int*>(smem + L.hist);
    int* bad = reinterpret_cast<int*>(smem + L.bad);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int t = blockIdx.y;
    const long long p0 = (long long)blockIdx.x * C;
    const int ncols = (int)min((long long)C, HW - p0);

    for (int r = tid; r <= n; r += blockDim.x) hist_s[r] = 0;
    for (int c = tid; c < C; c += blockDim.x) bad[c] = 0;
    __syncthreads();

    // Stage X and Y: row i of C floats per load step; columns past HW read as 0 and are never scored.
    const float* px = pred + (long long)t * n * HW + p0;
    const float* py = target + (long long)t * m * HW + p0;
#pragma unroll 4
    for (int e = tid; e < npad * C; e += blockDim.x) {
        const int i = e / C, c = e % C;
        float v = INFINITY;  // sorts past every finite value
        if (i < n) {
            v = 0.0f;
            if (c < ncols) {
                v = __ldcs(px + (long long)i * HW + c);
                if (!isfinite(v)) atomicOr(bad + c, 1);
            }
        }
        xs[i * st + c] = v;
    }
#pragma unroll 4
    for (int e = tid; e < m * C; e += blockDim.x) {
        const int j = e / C, c = e % C;
        float v = 0.0f;
        if (c < ncols) {
            v = __ldcs(py + (long long)j * HW + c);
            if (!isfinite(v)) atomicOr(bad + c, 1);
        }
        ys[j * st + c] = v;
    }
    __syncthreads();

    float* sw = smem + L.sw + (size_t)warp * (npad + 1);  // this warp's prefix sums S_0..S_n
    const float fn = (float)n, fm = (float)m;
    for (int c = warp; c < ncols; c += kScoreWarps) {
        const long long o = (long long)t * HW + p0 + c;
        if (bad[c]) {
            if (lane == 0) crps[o] = bias[o] = sd_pred[o] = sd_target[o] = mse_mean[o] = NAN;
            continue;
        }
        float* col = xs + c;
        // bitonic sort of col[0], col[st], ..., col[(npad-1) st], ascending
        for (int k = 2; k <= npad; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int q = lane; q < (npad >> 1); q += 32) {
                    const int lo = ((q & ~(j - 1)) << 1) | (q & (j - 1));
                    const int hi = lo + j;
                    const float a = col[lo * st], b = col[hi * st];
                    if ((a > b) == ((lo & k) == 0)) {
                        col[lo * st] = b;
                        col[hi * st] = a;
                    }
                }
                __syncwarp();
            }
        }
        const float shift = col[(n >> 1) * st];
        // prefix sums of the shifted sorted values, and the pair sum sum_k (2k - n + 1) x'_(k)
        float carry = 0.0f, pair = 0.0f;
        if (lane == 0) sw[0] = 0.0f;
        for (int b0 = 0; b0 < n; b0 += 32) {
            const int k = b0 + lane;
            const float v = k < n ? col[k * st] - shift : 0.0f;
            float s = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float u = __shfl_up_sync(0xffffffffu, s, d);
                if (lane >= d) s += u;
            }
            if (k < n) sw[k + 1] = carry + s;
            carry += __shfl_sync(0xffffffffu, s, 31);
            pair += (float)(2 * k - n + 1) * v;
        }
        pair = warp_sum(pair);
        const float mx = carry / fn;  // mean of X - shift
        float vx = 0.0f;
        for (int k = lane; k < n; k += 32) {
            const float d = col[k * st] - shift - mx;
            vx += d * d;
        }
        vx = warp_sum(vx);
        __syncwarp();
        const float sn = sw[n];
        // targets: rank by binary search on the raw sorted values (ties are not below), then sum_i |x_i - y|
        float abs_xy = 0.0f, sy = 0.0f;
        for (int j = lane; j < m; j += 32) {
            const float y = ys[j * st + c];
            int lo = 0, hi = n;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (col[mid * st] < y) lo = mid + 1;
                else hi = mid;
            }
            const float yv = y - shift;
            abs_xy += yv * (float)(2 * lo - n) - 2.0f * sw[lo] + sn;
            sy += yv;
            atomicAdd(hist_s + lo, 1);
        }
        abs_xy = warp_sum(abs_xy);
        const float my = warp_sum(sy) / fm;
        float vy = 0.0f, se = 0.0f;
        for (int j = lane; j < m; j += 32) {
            const float yv = ys[j * st + c] - shift;
            vy += (yv - my) * (yv - my);
            se += (mx - yv) * (mx - yv);
        }
        vy = warp_sum(vy);
        se = warp_sum(se);
        if (lane == 0) {
            crps[o] = abs_xy / (fn * fm) - pair / (fn * (fn - 1.0f));
            bias[o] = mx - my;
            sd_pred[o] = sqrtf(vx / (fn - 1.0f));
            sd_target[o] = sqrtf(vy / (fm - 1.0f));
            mse_mean[o] = se / fm;
        }
        __syncwarp();  // sw is rewritten for the warp's next column
    }
    __syncthreads();
    for (int r = tid; r <= n; r += blockDim.x)
        if (hist_s[r]) atomicAdd(hist + (long long)t * (n + 1) + r, (unsigned long long)hist_s[r]);
}

template <int C>
static int launch_scores(const float* pred, const float* target, float* crps, float* bias, float* sd_pred,
                         float* sd_target, float* mse_mean, long long* hist, int T, int n, int m, long long HW,
                         size_t smem, cudaStream_t st) {
    CESM_CHECK_CUDA(cudaFuncSetAttribute(ensemble_scores_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
    const dim3 grid((unsigned)((HW + C - 1) / C), (unsigned)T);
    ensemble_scores_kernel<C><<<grid, kScoreWarps * 32, smem, st>>>(
        pred, target, crps, bias, sd_pred, sd_target, mse_mean, reinterpret_cast<unsigned long long*>(hist), n, m,
        HW);
    CESM_CHECK_LAUNCH();
    return CESM_OK;
}

}  // namespace cesm

using namespace cesm;

extern "C" int cesm_ensemble_scores(const float* pred, const float* target, float* crps, float* bias, float* sd_pred,
                                    float* sd_target, float* mse_mean, long long* hist, int T, int n, int m,
                                    long long HW, void* stream) {
    CESM_REQUIRE(n >= 2 && n <= kScoreMaxMembers && m >= 2 && m <= kScoreMaxMembers,
                 "ensemble scores need 2 <= n, m <= %d members (n=%d m=%d)", kScoreMaxMembers, n, m);
    CESM_REQUIRE(T >= 1 && T <= 65535 && HW >= 1 && (HW + 15) / 16 <= 0x7fffffffLL,
                 "bad ensemble score sizes (T=%d HW=%lld)", T, HW);
    CESM_REQUIRE(pred && target && crps && bias && sd_pred && sd_target && mse_mean && hist,
                 "ensemble scores need pred, target, the five maps and hist");
    const cudaStream_t st = as_stream(stream);
    CESM_CHECK_CUDA(cudaMemsetAsync(hist, 0, (size_t)T * (n + 1) * sizeof(long long), st));
    // 32 pixels per block (128-byte rows) whenever the tile fits in shared memory; 16 otherwise (n and m near 1024)
    const size_t s32 = score_smem(n, m, 32).total * 4, s16 = score_smem(n, m, 16).total * 4;
    if (s32 <= 227 * 1024)
        return launch_scores<32>(pred, target, crps, bias, sd_pred, sd_target, mse_mean, hist, T, n, m, HW, s32, st);
    return launch_scores<16>(pred, target, crps, bias, sd_pred, sd_target, mse_mean, hist, T, n, m, HW, s16, st);
}
