// C-ABI core: error reporting, TMA descriptor cache, and the cesm_igemm / cesm_wgrad entry points
// (tile-shape selection + tensor-map construction for igemm2.cu, wgrad.cu and wgrad3.cu).
#include <atomic>
#include <mutex>
#include <string>
#include <unordered_map>

#include "api_common.h"
#include "igemm.h"

namespace cesm {

static thread_local std::string g_last_error;
static std::atomic<long long> g_launches{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
static std::atomic<int> g_prezeroed{0};
bool scratch_prezeroed() { return g_prezeroed.load(std::memory_order_relaxed) != 0; }

int set_error(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

// ------------------------------------------------------------------------------------------------
// TMA descriptors
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn resolve_encode() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

struct MapKey {
    uint64_t v[14];
    bool operator==(const MapKey& o) const {
        for (int i = 0; i < 14; ++i)
            if (v[i] != o.v[i]) return false;
        return true;
    }
};
struct MapKeyHash {
    size_t operator()(const MapKey& k) const {
        uint64_t h = 1469598103934665603ull;
        for (int i = 0; i < 14; ++i) {
            h ^= k.v[i];
            h *= 1099511628211ull;
        }
        return static_cast<size_t>(h);
    }
};
static std::mutex g_map_mutex;  // autograd runs backward on its own threads
static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_map_cache;

int get_tensor_map_h16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                        const uint64_t* strides_bytes, const uint32_t* box) {
    CESM_REQUIRE(rank >= 2 && rank <= 4, "tensor map rank %d unsupported", rank);
    CESM_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15u) == 0, "tensor base %p not 16-byte aligned", base);
    MapKey key{};
    key.v[0] = reinterpret_cast<uint64_t>(base);
    key.v[1] = static_cast<uint64_t>(rank);
    for (int i = 0; i < rank; ++i) {
        key.v[2 + i] = dims[i];
        key.v[6 + i] = (i == 0) ? 0 : strides_bytes[i - 1];
        key.v[10 + i] = box[i];
    }
    {
        std::lock_guard<std::mutex> lk(g_map_mutex);
        auto it = g_map_cache.find(key);
        if (it != g_map_cache.end()) {
            *out = it->second;
            return CESM_OK;
        }
    }
    EncodeTiledFn enc = resolve_encode();
    if (!enc) return set_error(CESM_ERR_CUDA, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    cuuint64_t gdim[4], gstr[3];
    cuuint32_t bx[4], es[4];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bx[i] = box[i];
        es[i] = 1;
        if (i > 0) {
            gstr[i - 1] = strides_bytes[i - 1];
            CESM_REQUIRE(gstr[i - 1] % 16 == 0, "tensor map stride %llu not a multiple of 16 B",
                         (unsigned long long)gstr[i - 1]);
        }
        CESM_REQUIRE(bx[i] >= 1 && bx[i] <= 256, "tensor map box[%d]=%u out of range", i, bx[i]);
    }
    alignas(64) CUtensorMap m;
    CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank, const_cast<void*>(base), gdim, gstr, bx, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(CESM_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    {
        std::lock_guard<std::mutex> lk(g_map_mutex);
        if (g_map_cache.size() > 8192) g_map_cache.clear();
        g_map_cache.emplace(key, m);
    }
    *out = m;
    return CESM_OK;
}

// ------------------------------------------------------------------------------------------------
// tile-shape selection: split the 128 rows of an M tile over (w, h, n) to waste the fewest rows
// ------------------------------------------------------------------------------------------------
static void choose_tile(int n, int oh, int ow, int* bw, int* bh, int* bn) {
    long long best_tiles = -1;
    int b_w = 1, b_h = 1, b_n = 1;
    for (int w = 1; w <= 128 && w <= ow; ++w) {
        // only widths that are the full row, or powers of two, keep epilogue stores well formed
        if (!(w == ow || (w & (w - 1)) == 0)) continue;
        for (int h = 1; h * w <= 128 && h <= oh; ++h) {
            if (!(h == oh || (h & (h - 1)) == 0)) continue;
            int nn = 128 / (w * h);
            if (nn > n) nn = n;
            if (nn < 1) nn = 1;
            if (w != ow || h != oh) nn = 1;  // only batch whole images into one tile
            long long tiles = 1LL * ceil_div(ow, w) * ceil_div(oh, h) * ceil_div(n, nn);
            if (best_tiles < 0 || tiles < best_tiles || (tiles == best_tiles && w > b_w)) {
                best_tiles = tiles;
                b_w = w;
                b_h = h;
                b_n = nn;
            }
        }
    }
    *bw = b_w;
    *bh = b_h;
    *bn = b_n;
}

}  // namespace cesm

using namespace cesm;

extern "C" const char* cesm_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* cesm_version(void) { return "cesm_b200 0.1 sm_100a"; }
extern "C" void cesm_set_prezeroed_scratch(int on) { g_prezeroed.store(on ? 1 : 0, std::memory_order_relaxed); }
extern "C" long long cesm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// ------------------------------------------------------------------------------------------------
// second-generation persistent kernel: tile / shared-memory plan
// ------------------------------------------------------------------------------------------------
static int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0)
            n = v;
        else
            n = 148;
    }
    return n;
}

static bool is_3x3_unit_taps(const cesm_igemm_args* a) {
    if (a->num_taps != 9 || a->stride != 1) return false;
    bool seen[9] = {false};
    for (int t = 0; t < 9; ++t) {
        const int dh = a->tap_dh[t], dw = a->tap_dw[t];
        if (dh < -1 || dh > 1 || dw < -1 || dw > 1) return false;
        seen[(dh + 1) * 3 + dw + 1] = true;
    }
    for (bool b : seen)
        if (!b) return false;
    return true;
}

static int igemm2_run(const cesm_igemm_args* a, cudaStream_t st) {
    Igemm2Params p{};
    p.c0 = a->c0;
    p.c1 = a->c1;
    p.num_taps = a->num_taps;
    const int ctot = a->c0 + a->c1;
    p.num_kb = a->num_taps * (ctot / 64);
    p.n = a->n;
    p.oh = a->oh;
    p.ow = a->ow;
    p.cout = a->cout;
    int block_n = (a->cout % 256 == 0) ? 256 : (a->cout % 128 == 0 ? 128 : 64);

    // ---- HALO candidates: padded row width pw in {16, 32, 64, 128}, bw = pw - 2, bh = 128 / pw ----
    bool halo = false;
    if (is_3x3_unit_taps(a)) {
        double best = 0.0;
        int best_pw = 0;
        for (int pw = 16; pw <= 128; pw <<= 1) {
            const int bw = pw - 2, bh = 128 / pw;
            const double tiles = (double)ceil_div(a->ow, bw) * ceil_div(a->oh, bh);
            const double useful = ((double)a->ow * a->oh) / (tiles * 128.0);
            // prefer taller tiles (less halo re-fetch) when the useful fraction is close
            const double score = useful * (1.0 - 0.08 * 2.0 / (bh + 2));
            if (score > best) {
                best = score;
                best_pw = pw;
            }
        }
        if (best_pw && best >= 0.55) {
            halo = true;
            p.bw = best_pw - 2;
            p.bh = 128 / best_pw;
            p.bn = 1;
        }
    }
    if (!halo) choose_tile(a->n, a->oh, a->ow, &p.bw, &p.bh, &p.bn);
    p.tiles_w = ceil_div(a->ow, p.bw);
    p.tiles_h = ceil_div(a->oh, p.bh);
    p.m_tiles = p.tiles_w * p.tiles_h * ceil_div(a->n, p.bn);

    // ---- column-tile width of the tensor-bound (halo) shapes: MMA efficiency against wave quantisation ----
    // A 128 x N x 16 MMA is bound by the shared-memory operand feed (4 KB of A + N/32 KB of B per MMA): measured
    // ~75 / 90 / 165 clocks at N = 64 / 128 / 256 (tools/bench_igemm.py).  With few row tiles (48x72 x 6 frames = 216
    // tiles on 148 SMs) a narrower N fills the last wave: 3 waves of N=128 tiles beat 2 waves of N=256 tiles.
    // CTA pairs (cta_group::2, igemm2.cu): two row tiles per cluster share the weight rows, so a CTA reads
    // N*16 B instead of N*32 B of B per MMA (measured ~62 / 84 / 135 clocks).
    const bool pair = halo && p.m_tiles >= 2 && sm_count() >= 2;
    if (halo) {
        static const double clk1[3] = {75.0, 90.0, 165.0}, clk2[3] = {62.0, 84.0, 135.0};
        const double* clk = pair ? clk2 : clk1;
        const int units = pair ? sm_count() / 2 : sm_count();
        const long long m_units = pair ? (p.m_tiles + 1) / 2 : p.m_tiles;
        double best = 1e30;
        for (int n = 256, i = 2; n >= 64; n >>= 1, --i) {
            if (a->cout % n) continue;
            const long long tiles = m_units * (a->cout / n);
            const double t = (double)((tiles + units - 1) / units) * clk[i];
            if (t < best - 1e-9) {   // ties keep the wider tile
                best = t;
                block_n = n;
            }
        }
    }
    p.n_tiles = a->cout / block_n;

    // ---- GroupNorm statistics: every tile must lie within one sample ----
    p.gn_sums = a->gn_sums;
    if (a->gn_sums) {
        CESM_REQUIRE(a->gn_groups > 0 && a->gn_frames > 0 && a->cout % a->gn_groups == 0 && a->n % a->gn_frames == 0,
                     "bad GroupNorm statistics arguments (groups=%d frames=%d)", a->gn_groups, a->gn_frames);
        p.gn_groups = a->gn_groups;
        p.gn_cpg = a->cout / a->gn_groups;
        p.gn_frames = a->gn_frames;
        CESM_REQUIRE(a->gn_groups <= 32, "fused GroupNorm statistics support at most 32 groups (got %d)", a->gn_groups);
        CESM_REQUIRE(p.gn_cpg % 8 == 0 && (p.gn_cpg >= 64 ? p.gn_cpg % 64 == 0 : 64 % p.gn_cpg == 0),
                     "fused GroupNorm statistics need 8 | cout/groups and cout/groups | 64 or 64 | cout/groups (got %d)",
                     p.gn_cpg);
        if (p.bn > 1 && a->gn_frames % p.bn != 0) {  // re-tile with one image per tile
            p.bn = 1;
            p.m_tiles = p.tiles_w * p.tiles_h * a->n;
        }
        CESM_ZERO_SCRATCH(a->gn_sums, sizeof(float) * 2 * (a->n / a->gn_frames) * a->gn_groups, st);
    }

    // ---- shared-memory plan ----
    const int pw = halo ? p.bw + 2 : p.bw;
    if (halo) {
        const int rows_box = pw * (p.bh + 2), rows_need = 2 * pw + 2 + 128;
        const int rows = rows_box > rows_need ? rows_box : rows_need;
        p.a_stage_bytes = (uint32_t)((rows * 128 + 1023) / 1024 * 1024);
        p.a_box_bytes = (uint32_t)rows_box * 128u;
    } else {
        p.a_stage_bytes = 16384;
        p.a_box_bytes = 128u * p.bw * p.bh * p.bn;
    }
    const long long budget = (long long)kIgemm2MaxSmem - 1024 /*align*/ - 1024 /*barriers*/ - 2 * 16384 /*out staging*/;
    const long long b_total = (long long)a->cout * p.num_kb * 128 / (pair ? 2 : 1);   // per CTA
    const long long b_blk = (long long)block_n * 128 / (pair ? 2 : 1);
    const int a_min = 2;
    if (b_total + a_min * (long long)p.a_stage_bytes <= budget) {
        p.b_resident = 1;
        p.b_stages = 1;
        long long as = (budget - b_total) / p.a_stage_bytes;
        const int a_cap = halo ? 4 : 8;
        p.a_stages = (int)(as > a_cap ? a_cap : as);
    } else {
        p.b_resident = 0;
        p.a_stages = halo ? 2 : 4;
        long long bs = (budget - (long long)p.a_stages * p.a_stage_bytes) / b_blk;
        if (bs > 16) bs = 16;
        if (bs < 2) {  // very wide tiles: trade activation stages for weight stages
            p.a_stages = 2;
            bs = (budget - (long long)p.a_stages * p.a_stage_bytes) / b_blk;
        }
        CESM_REQUIRE(bs >= 2, "igemm2: no shared-memory plan for cout=%d K=%d", a->cout, p.num_kb * 64);
        p.b_stages = (int)bs;
    }
    const long long b_bytes = p.b_resident ? b_total : (long long)p.b_stages * b_blk;
    const size_t smem = 1024 + (size_t)p.a_stages * p.a_stage_bytes + (size_t)b_bytes + 2 * 16384 + 1024;
    CESM_REQUIRE(smem <= kIgemm2MaxSmem, "igemm2: shared-memory plan of %zu B exceeds the limit", smem);

    p.out_h = a->out_h;
    p.out_w = a->out_w;
    p.o_sh = a->o_sh;
    p.o_sw = a->o_sw;
    p.o_h0 = a->o_h0;
    p.o_w0 = a->o_w0;
    p.bias = a->bias;
    p.residual = a->residual;
    p.ldr = a->ldr;
    if (a->ln_colsum) {
        CESM_REQUIRE(a->cout == 64 && a->c0 == 64 && a->c1 == 0 && a->num_taps == 1 && a->stride == 1 && !a->gn_sums &&
                         a->residual == a->a0 && a->ldr == 64,
                     "the LayerNorm fold needs a 64 -> 64 one-tap projection whose residual is its own input");
        p.ln_colsum = a->ln_colsum;
        p.ln_eps = a->ln_eps;
    }

    // ---- tensor maps ----
    Igemm2Maps maps;
    int n_amaps = 0;
    const uint32_t abox[4] = {64u, (uint32_t)(halo ? pw : p.bw), (uint32_t)(halo ? p.bh + 2 : p.bh), (uint32_t)p.bn};
    if (a->stride == 1) {
        const void* src[2] = {a->a0, a->a1};
        const int cs[2] = {a->c0, a->c1};
        for (int s = 0; s < 2; ++s) {
            if (!src[s]) continue;
            const uint64_t dims[4] = {(uint64_t)cs[s], (uint64_t)a->w, (uint64_t)a->h, (uint64_t)a->n};
            const uint64_t str[3] = {(uint64_t)cs[s] * 2, (uint64_t)a->w * cs[s] * 2, (uint64_t)a->h * a->w * cs[s] * 2};
            int rc = get_tensor_map_h16(&maps.a[s], src[s], 4, dims, str, abox);
            if (rc) return rc;
            n_amaps = s + 1;
        }
        for (int t = 0; t < a->num_taps; ++t) {
            p.tap_map[t] = 0;
            p.tap_dh[t] = a->tap_dh[t];
            p.tap_dw[t] = a->tap_dw[t];
        }
    } else {
        const int c = a->c0;
        for (int ph = 0; ph < 2; ++ph)
            for (int pw2 = 0; pw2 < 2; ++pw2) {
                const char* base = static_cast<const char*>(a->a0) + (size_t)(ph * a->w + pw2) * c * 2;
                const uint64_t dims[4] = {(uint64_t)c, (uint64_t)a->w / 2, (uint64_t)a->h / 2, (uint64_t)a->n};
                const uint64_t str[3] = {(uint64_t)c * 4, (uint64_t)a->w * c * 4, (uint64_t)a->h * a->w * c * 2};
                int rc = get_tensor_map_h16(&maps.a[ph * 2 + pw2], base, 4, dims, str, abox);
                if (rc) return rc;
            }
        n_amaps = 4;
        for (int t = 0; t < a->num_taps; ++t) {
            const int ph = a->tap_dh[t] & 1, pw2 = a->tap_dw[t] & 1;
            p.tap_map[t] = ph * 2 + pw2;
            p.tap_dh[t] = (a->tap_dh[t] - ph) / 2;
            p.tap_dw[t] = (a->tap_dw[t] - pw2) / 2;
        }
    }
    for (int i = n_amaps; i < 4; ++i) maps.a[i] = maps.a[0];
    {
        const int ktot = p.num_kb * 64;
        const uint64_t dims[2] = {(uint64_t)ktot, (uint64_t)a->cout};
        const uint64_t str[1] = {(uint64_t)ktot * 2};
        const uint32_t bbox[2] = {64u, (uint32_t)(pair ? block_n / 2 : block_n)};
        int rc = get_tensor_map_h16(&maps.b, a->wt, 2, dims, str, bbox);
        if (rc) return rc;
    }
    {
        // output as a (possibly strided) [cout, ow, oh, n] tensor: pixel (n, oh, ow) lives at row
        // (n*out_h + oh*o_sh + o_h0)*out_w + ow*o_sw + o_w0 of a [*, ldo] matrix
        const char* base = static_cast<const char*>(a->out) + ((size_t)a->o_h0 * a->out_w + a->o_w0) * a->ldo * 2;
        const uint64_t dims[4] = {(uint64_t)a->cout, (uint64_t)a->ow, (uint64_t)a->oh, (uint64_t)a->n};
        const uint64_t str[3] = {(uint64_t)a->o_sw * a->ldo * 2, (uint64_t)a->o_sh * a->out_w * a->ldo * 2,
                                 (uint64_t)a->out_h * a->out_w * a->ldo * 2};
        // warp-private epilogue: each warp's 32 accumulator rows are one box
        if (halo)
            p.epi_warp = (pw == 32);
        else
            p.epi_warp = (p.bw % 32 == 0);
        uint32_t obox[4] = {64u, (uint32_t)p.bw, (uint32_t)(halo ? 1 : p.bh), (uint32_t)(halo ? 1 : p.bn)};
        if (p.epi_warp && !halo) {
            obox[1] = 32u;
            obox[2] = 1u;
            obox[3] = 1u;
        }
        int rc = get_tensor_map_h16(&maps.out, base, 4, dims, str, obox);
        if (rc) return rc;
    }
    // 64->768 projection at 192x288: 131.5 us n-major, 106.6 us m-major (the output rows are completed in one
    // go instead of in three passes over the 510 MB tensor; tools/bench_igemm.py)
    p.m_major = p.b_resident && p.n_tiles > 1 ? 1 : 0;
    int grid;
    if (pair) {
        const int units = ((p.m_tiles + 1) / 2) * p.n_tiles, clusters = sm_count() / 2;
        grid = 2 * (units < clusters ? units : clusters);
    } else {
        const int total_tiles = p.m_tiles * p.n_tiles;
        grid = total_tiles < sm_count() ? total_tiles : sm_count();
    }
    note_launch();
    CESM_CHECK_CUDA(igemm2_launch(maps, p, block_n, halo, pair, grid, smem, st));
    return CESM_OK;
}

extern "C" int cesm_igemm(const cesm_igemm_args* a, void* stream) {
    CESM_REQUIRE(a != nullptr, "args is NULL");
    CESM_REQUIRE(a->c0 > 0 && a->c0 % 64 == 0 && a->c1 >= 0 && a->c1 % 64 == 0,
                 "channel counts must be multiples of 64 (c0=%d c1=%d)", a->c0, a->c1);
    CESM_REQUIRE(a->cout > 0 && a->cout % 64 == 0, "cout=%d must be a multiple of 64", a->cout);
    CESM_REQUIRE(a->num_taps >= 1 && a->num_taps <= CESM_MAX_TAPS, "num_taps=%d out of range", a->num_taps);
    CESM_REQUIRE(a->stride == 1 || a->stride == 2, "stride=%d unsupported", a->stride);
    CESM_REQUIRE(a->stride == 1 || (a->c1 == 0 && a->h % 2 == 0 && a->w % 2 == 0),
                 "stride 2 needs a single source with even h, w");
    CESM_REQUIRE(a->n > 0 && a->h > 0 && a->w > 0 && a->oh > 0 && a->ow > 0, "empty geometry");
    CESM_REQUIRE((a->c1 == 0) == (a->a1 == nullptr), "a1 / c1 mismatch");
    CESM_REQUIRE(a->ldo % 8 == 0 && (a->residual == nullptr || a->ldr % 8 == 0), "row pitches must be multiples of 8");
    return igemm2_run(a, as_stream(stream));
}

// 64-pixel K tile for the weight gradient: powers of two with bw*bh*bn == 64, fewest tiles
static void choose_tile64(int n, int oh, int ow, int* bw, int* bh, int* bn) {
    long long best = -1;
    for (int w = 1; w <= 64; w <<= 1)
        for (int h = 1; h * w <= 64; h <<= 1) {
            const int nn = 64 / (w * h);
            const long long tiles = 1LL * ceil_div(ow, w) * ceil_div(oh, h) * ceil_div(n, nn);
            if (best < 0 || tiles < best || (tiles == best && w > *bw)) {
                best = tiles;
                *bw = w;
                *bh = h;
                *bn = nn;
            }
        }
}

// 3x3 stride-1 weight gradients with <= 128 output channels go to wgrad3.cu (one halo fetch serves all nine taps).
// Its accumulators are 64 columns wide, so at 256+ output channels the wider MMAs of wgrad.cu win again
// (tools/bench_wgrad.py on B200: 64->64 38.8 -> 32.2 us, 128->64 66.6 -> 53.4, 128->128 43.1 -> 33.9, 256->256 33.5 -> 36.1).
// Returns true when it handled the call (*rc = status).
static bool wgrad3_try(const cesm_wgrad_args* a, cudaStream_t st, int* rc) {
    if (a->stride != 1 || a->num_taps != 9 || a->cout > 128) return false;
    if (a->oh != a->h || a->ow != a->w || a->y_h != a->oh || a->y_w != a->ow || a->y_sh != 1 || a->y_sw != 1 ||
        a->y_h0 != 0 || a->y_w0 != 0)
        return false;
    bool seen[9] = {};
    for (int t = 0; t < 9; ++t) {
        const int dh = a->tap_dh[t], dw = a->tap_dw[t];
        if (dh < -1 || dh > 1 || dw < -1 || dw > 1 || seen[(dh + 1) * 3 + dw + 1]) return false;
        seen[(dh + 1) * 3 + dw + 1] = true;
    }
    auto run = [&]() -> int {
        Wgrad3Params p{};
        p.c0 = a->c0;
        p.c1 = a->c1;
        p.n = a->n;
        p.cout = a->cout;
        // pixel tile: 32 x 4 or 16 x 8, whichever wastes fewer out-of-range pixels
        const long long waste32 = (long long)ceil_div(a->ow, 32) * 32 * ceil_div(a->oh, 4) * 4;
        const long long waste16 = (long long)ceil_div(a->ow, 16) * 16 * ceil_div(a->oh, 8) * 8;
        p.bw = waste16 < waste32 ? 16 : 32;
        p.bh = 128 / p.bw;
        p.tiles_w = ceil_div(a->ow, p.bw);
        p.tiles_h = ceil_div(a->oh, p.bh);
        const int pw = p.bw + 2;
        p.halo_box_bytes = (uint32_t)(pw * (p.bh + 2) * 128);
        p.halo_stage_bytes = (p.halo_box_bytes + 256u + 1023u) / 1024u * 1024u;   // + the ghost tap's extra rows
        const int ctot = a->c0 + a->c1;
        long long so, si;
        int tap_off_in[9];
        if (a->dw_so != 0) {
            so = a->dw_so;
            si = a->dw_si;
            for (int t = 0; t < 9; ++t) tap_off_in[t] = a->dw_tap_off[t];
        } else {
            so = 9LL * ctot;
            si = 1;
            for (int t = 0; t < 9; ++t) tap_off_in[t] = t * ctot;
            CESM_CHECK_CUDA(cudaMemsetAsync(a->dw, 0, sizeof(float) * (size_t)a->cout * 9 * ctot, st));
        }
        p.so = so;
        p.si = si;
        p.dw = a->dw;
        // taps in ascending halo-row order (pairs are stacked through a positive leading-byte offset)
        for (int k = 0; k < 9; ++k) {
            const int dh = k / 3 - 1, dw = k % 3 - 1;
            for (int t = 0; t < 9; ++t)
                if (a->tap_dh[t] == dh && a->tap_dw[t] == dw) {
                    p.tap_row[k] = (1 + dh) * pw + (1 + dw);
                    p.tap_off[k] = tap_off_in[t];
                }
        }
        p.tap_row[9] = p.tap_row[8] + 1;
        p.tap_off[9] = p.tap_off[8];
        Wgrad3Maps maps;
        const uint32_t xbox[4] = {64u, (uint32_t)pw, (uint32_t)(p.bh + 2), 1u};
        const void* src[2] = {a->x0, a->x1};
        const int cs[2] = {a->c0, a->c1};
        for (int s = 0; s < 2; ++s) {
            if (!src[s]) {
                maps.x[s] = maps.x[0];
                continue;
            }
            const uint64_t dims[4] = {(uint64_t)cs[s], (uint64_t)a->w, (uint64_t)a->h, (uint64_t)a->n};
            const uint64_t str[3] = {(uint64_t)cs[s] * 2, (uint64_t)a->w * cs[s] * 2, (uint64_t)a->h * a->w * cs[s] * 2};
            int e = get_tensor_map_h16(&maps.x[s], src[s], 4, dims, str, xbox);
            if (e) return e;
        }
        {
            const int co = a->cout;
            const uint32_t ybox[4] = {64u, (uint32_t)p.bw, (uint32_t)p.bh, 1u};
            const uint64_t dims[4] = {(uint64_t)co, (uint64_t)a->ow, (uint64_t)a->oh, (uint64_t)a->n};
            const uint64_t str[3] = {(uint64_t)co * 2, (uint64_t)a->ow * co * 2, (uint64_t)a->oh * a->ow * co * 2};
            int e = get_tensor_map_h16(&maps.y, a->dy, 4, dims, str, ybox);
            if (e) return e;
        }
        const int cblk = ctot / 64;
        const int groups = cblk * (a->cout / 64);
        const int tiles = p.tiles_w * p.tiles_h * a->n;
        int ksplit = sm_count() / groups;   // one CTA per SM (512 TMEM columns, 4 x 42 KB ring)
        if (ksplit > tiles) ksplit = tiles;
        if (ksplit < 1) ksplit = 1;
        note_launch();
        CESM_CHECK_CUDA(wgrad3_launch(maps, p, cblk, ksplit, st));
        return CESM_OK;
    };
    *rc = run();
    return true;
}

extern "C" int cesm_wgrad(const cesm_wgrad_args* a, void* stream) {
    CESM_REQUIRE(a != nullptr, "args is NULL");
    CESM_REQUIRE(a->c0 > 0 && a->c0 % 64 == 0 && a->c1 >= 0 && a->c1 % 64 == 0,
                 "channel counts must be multiples of 64 (c0=%d c1=%d)", a->c0, a->c1);
    CESM_REQUIRE(a->cout > 0 && a->cout % 64 == 0, "cout=%d must be a multiple of 64", a->cout);
    CESM_REQUIRE(a->num_taps >= 1 && a->num_taps <= CESM_MAX_TAPS, "num_taps=%d out of range", a->num_taps);
    CESM_REQUIRE(a->stride == 1 || a->stride == 2, "stride=%d unsupported", a->stride);
    CESM_REQUIRE(a->stride == 1 || (a->c1 == 0 && a->h % 2 == 0 && a->w % 2 == 0),
                 "stride 2 needs a single source with even h, w");
    CESM_REQUIRE((a->c1 == 0) == (a->x1 == nullptr), "x1 / c1 mismatch");
    cudaStream_t st = as_stream(stream);

    {
        int rc = 0;
        if (wgrad3_try(a, st, &rc)) return rc;
    }

    WgradParams p{};
    p.c0 = a->c0;
    p.c1 = a->c1;
    p.num_taps = a->num_taps;
    p.n = a->n;
    p.oh = a->oh;
    p.ow = a->ow;
    choose_tile64(a->n, a->oh, a->ow, &p.bw, &p.bh, &p.bn);
    p.box_bytes = 64u * 2u * 64u;
    p.cout = a->cout;
    p.dw = a->dw;
    const uint32_t box[4] = {64u, (uint32_t)p.bw, (uint32_t)p.bh, (uint32_t)p.bn};

    CUtensorMap xmaps[4];
    int n_xmaps = 0;
    if (a->stride == 1) {
        const void* src[2] = {a->x0, a->x1};
        const int cs[2] = {a->c0, a->c1};
        for (int s = 0; s < 2; ++s) {
            if (!src[s]) continue;
            const uint64_t dims[4] = {(uint64_t)cs[s], (uint64_t)a->w, (uint64_t)a->h, (uint64_t)a->n};
            const uint64_t str[3] = {(uint64_t)cs[s] * 2, (uint64_t)a->w * cs[s] * 2, (uint64_t)a->h * a->w * cs[s] * 2};
            int rc = get_tensor_map_h16(&xmaps[s], src[s], 4, dims, str, box);
            if (rc) return rc;
            n_xmaps = s + 1;
        }
        for (int t = 0; t < a->num_taps; ++t) {
            p.tap_map[t] = 0;
            p.tap_dh[t] = a->tap_dh[t];
            p.tap_dw[t] = a->tap_dw[t];
        }
    } else {
        const int c = a->c0;
        for (int ph = 0; ph < 2; ++ph)
            for (int pw = 0; pw < 2; ++pw) {
                const char* base = static_cast<const char*>(a->x0) + (size_t)(ph * a->w + pw) * c * 2;
                const uint64_t dims[4] = {(uint64_t)c, (uint64_t)a->w / 2, (uint64_t)a->h / 2, (uint64_t)a->n};
                const uint64_t str[3] = {(uint64_t)c * 4, (uint64_t)a->w * c * 4, (uint64_t)a->h * a->w * c * 2};
                int rc = get_tensor_map_h16(&xmaps[ph * 2 + pw], base, 4, dims, str, box);
                if (rc) return rc;
            }
        n_xmaps = 4;
        for (int t = 0; t < a->num_taps; ++t) {
            const int ph = a->tap_dh[t] & 1, pw = a->tap_dw[t] & 1;
            p.tap_map[t] = ph * 2 + pw;
            p.tap_dh[t] = (a->tap_dh[t] - ph) / 2;
            p.tap_dw[t] = (a->tap_dw[t] - pw) / 2;
        }
    }
    CUtensorMap ymap;
    {
        const int co = a->cout;
        const char* base = static_cast<const char*>(a->dy) + ((size_t)a->y_h0 * a->y_w + a->y_w0) * co * 2;
        const uint64_t dims[4] = {(uint64_t)co, (uint64_t)a->ow, (uint64_t)a->oh, (uint64_t)a->n};
        const uint64_t str[3] = {(uint64_t)a->y_sw * co * 2, (uint64_t)a->y_sh * a->y_w * co * 2,
                                 (uint64_t)a->y_h * a->y_w * co * 2};
        int rc = get_tensor_map_h16(&ymap, base, 4, dims, str, box);
        if (rc) return rc;
    }
    const int ctot = a->c0 + a->c1;
    if (a->dw_so != 0) {  // accumulate straight into the caller's layout
        p.so = a->dw_so;
        p.si = a->dw_si;
        for (int t = 0; t < a->num_taps; ++t) p.tap_off[t] = a->dw_tap_off[t];
    } else {
        p.so = (long long)a->num_taps * ctot;
        p.si = 1;
        for (int t = 0; t < a->num_taps; ++t) p.tap_off[t] = t * ctot;
        CESM_CHECK_CUDA(cudaMemsetAsync(a->dw, 0, sizeof(float) * (size_t)a->cout * a->num_taps * ctot, st));
    }
    const int block_n = (a->cout % 256 == 0) ? 256 : (a->cout % 128 == 0 ? 128 : 64);
    const int units = a->num_taps * (ctot / 64);
    // CTA pairs where a launch has at least two 128-row blocks and is fed through L2 (multi-tap)
    const int m_tiles = (units + 1) / 2;
    const bool pair = block_n >= 128 && m_tiles >= 2 && a->num_taps > 1;
    const int base_ctas = (pair ? (m_tiles + 1) / 2 * 2 : m_tiles) * (a->cout / block_n);
    const int tiles = ceil_div(a->ow, p.bw) * ceil_div(a->oh, p.bh) * ceil_div(a->n, p.bn);
    // split-K so that the grid is ONE resident wave (two CTAs per SM; rounding up would leave a second
    // wave of a few CTAs that costs as much as the first)
    int ksplit = (148 * 2) / base_ctas;
    if (ksplit > tiles) ksplit = tiles;
    if (ksplit < 1) ksplit = 1;
    note_launch();
    CESM_CHECK_CUDA(wgrad_launch(xmaps, n_xmaps, ymap, p, block_n, ksplit, pair, st));
    return CESM_OK;
}
