// Shared device-side helpers for the sm_100a kernels: PTX wrappers for mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / TMEM load) and small math utilities.
// Everything here is hand-written inline PTX for sm_100a; there is no other backend.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace cesm {

// 16-bit storage / tensor-core operand type of every activation, gradient and packed weight: IEEE fp16
// (the reference's own autocast dtype, train.py:853), fp32 accumulation everywhere.  bf16's 8-bit
// mantissa cannot meet the 1e-2 per-tensor parity bar (weight rounding alone puts 15 % of the gradient
// tensors above it: tests/noise_model.py, profiles/r02_noise_budget.txt); fp16 has 11 bits at the same
// tensor-core rate and HBM traffic.  Gradients are kept in range by loss scaling (engine / GradScaler,
// train.py:862-867), exactly as in the reference.
typedef __half h16;

// ---------------------------------------------------------------------------------------------
// misc
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() {
    uint32_t l;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
    return l;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// exp(x) as ONE FFMA + ONE MUFU: ex2.approx.ftz(x * log2(e) - shift_l2e).  `__expf` adds a denormal-range
// fix-up (compare, two scalings, predicate shuffling: ~6 more instructions per element) that the
// softmax-style users here do not need: results that small flush to zero either way after fp16 rounding.
static constexpr float kLog2e = 1.4426950408889634f;
__device__ __forceinline__ float ex2_ftz(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// exp(x - m) with m pre-multiplied: m_l2e = m * log2(e)
__device__ __forceinline__ float exp_sub(float x, float m_l2e) { return ex2_ftz(fmaf(x, kLog2e, -m_l2e)); }

// Packed fp32 pairs (Blackwell FFMA2 / FMUL2 / FADD2: two fp32 lanes per issue slot).  The norm kernels
// are issue-limited before they are HBM-limited, and fp16x2 unpacks to exactly such pairs.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\t"
        "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "mul.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "add.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
// tanh / sigmoid: ONE MUFU op, tanh.approx.f32 (~2^-11 relative error).  Measured on B200 against the two-MUFU
// form (1 - e) / (1 + e), e = 2^(-2 h log2 e) through ex2.approx + rcp.approx (~2^-22;
// profiles/r02_ablation_sigmoid.txt, 3 input seeds at the config/baseline training shape): forward error 1.0-1.2e-3
// and worst gradient tensor 2.1-2.9e-3 with EITHER form -- the approximation error is the size of one fp16 rounding of
// the value it feeds -- while the two-MUFU form costs 0.16 ms per training step (the GroupNorm kernels are MUFU /
// issue limited).
__device__ __forceinline__ float tanh_f(float h) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return t;
}
__device__ __forceinline__ float2 tanh2(float2 h) { return make_float2(tanh_f(h.x), tanh_f(h.y)); }

// sigmoid(x) = 0.5 * tanh(x / 2) + 0.5 (see tanh_f for the measured effect of the one-MUFU form)
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(0.5f, tanh_f(0.5f * x), 0.5f); }
__device__ __forceinline__ float silu_f(float x) { return x * sigmoid_fast(x); }
// d/dx silu(x) = s + x*s*(1-s)
__device__ __forceinline__ float dsilu_f(float x) {
    const float s = sigmoid_fast(x);
    return s * (1.f + x * (1.f - s));
}
// The same derivative from h = x/2 with two fewer ops: t = tanh(h), s = (1+t)/2, s(1-s) = (1-t^2)/4, so
//   silu'(x) = 0.5 * (1 + R),  R = t + h (1 - t^2)          (callers fold the 0.5 * (1 + .) into their own FMAs)
__device__ __forceinline__ float dsilu_R_from_half(float h) {
    const float t = tanh_f(h);
    return fmaf(h, fmaf(-t, t, 1.f), t);
}
// full-precision variants for the fp32 paths (time-embedding MLP)
__device__ __forceinline__ float silu_precise(float x) { return __fdividef(x, 1.f + __expf(-x)); }
__device__ __forceinline__ float dsilu_precise(float x) {
    const float s = __fdividef(1.f, 1.f + __expf(-x));
    return s * (1.f + x * (1.f - s));
}

// fp32 pair -> packed fp16x2 (round to nearest even; |x| > 65504 becomes inf, which is what the loss
// scaler's overflow check looks for) and back
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_h2(uint32_t u) {
    return __half22float2(*reinterpret_cast<const __half2*>(&u));
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch.  Every kernel triggers at its top (so the NEXT kernel's CTAs may be
// scheduled, run their prologue and park as soon as this kernel's CTAs have all started), and every
// kernel launched through launch_pdl() waits here before it touches global memory: griddepcontrol.wait
// returns only when the preceding kernel has completed and flushed.  Both are no-ops for launches
// without the attribute.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
#ifdef CESM_MBAR_TEST_WAIT
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#else
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#endif
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}
// Bounded wait: a protocol bug must never hang the GPU (a hung box is a lost lease), so after
// ~2 s of spinning the kernel reports where it stuck and traps.
static __device__ __noinline__ void mbar_timeout_trap(uint32_t bar, uint32_t parity, int site) {
    printf("[cesm_b200] mbarrier wait timed out: block (%d,%d,%d) thread %d site %d bar 0x%x parity %u\n",
           blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, site, bar, parity);
    __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int site = 0) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) mbar_timeout_trap(bar, parity, site);
    }
}

// ---------------------------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t smem_dst, const void* map, uint32_t bar, int c0,
                                            int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2),
          "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const void* map, uint32_t bar, int c0,
                                            int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// ---------------------------------------------------------------------------------------------
// CTA pairs (cta_group::2): two CTAs of a cluster on one TPC issue ONE MMA of M = 256; each provides its own 128
// rows of A and HALF of the B rows from its own shared memory, so the operand bytes a CTA reads per MMA drop from
// 4 KB + N*32 B to 4 KB + N*16 B.  Only the even CTA (the leader) issues MMAs and owns the "full" barriers; TMA
// loads of both CTAs report to the leader's barrier (address with the peer bit cleared), commits are multicast.
// ---------------------------------------------------------------------------------------------
static constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // shared::cluster address of the pair's even CTA
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {   // every thread of both CTAs
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t smem_dst, const void* map, uint32_t bar, int c0, int c1,
                                                 int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2),
          "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t smem_dst, const void* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
// arrive on the LEADER's copy of a barrier (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_dst, uint32_t ncols) {   // one warp of EACH CTA
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B with M = 256, issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the barrier at this shared-memory offset in BOTH CTAs once all MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    asm volatile(
        "{\n\t.reg .b16 m;\n\t"
        "mov.b16 m, 3;\n\t"
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}" ::"r"(bar)
        : "memory");
}

// One lane of a fully converged warp (warp-uniform control flow lets the compiler keep MMA operands in
// uniform registers instead of emitting a per-thread "waterfall" loop around every tcgen05.mma).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
// D[tmem] (+)= A[smem] * B[smem], fp16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier when all previously issued MMAs of this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
                 : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets TMEM lane (base_lane + i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
          "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
          "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor (sm_100 "version 1").  Field layout:
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 | [32,46) stride byte offset >> 4
//   [46,48) version = 1 | [49,52) base offset | [61,64) layout type (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                         uint32_t sbo_bytes, uint32_t base_offset = 0) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(base_offset & 7u) << 49;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// Instruction descriptor for kind::f16 with fp16 A/B and fp32 accumulate.
//   [4,6) c_format (1 = f32) | [7,10) a_format (0 = f16, 1 = bf16) | [10,13) b_format (0 = f16, 1 = bf16)
//   [15] a_major (0 = K, 1 = MN) | [16] b_major | [17,23) N >> 3 | [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16(uint32_t M, uint32_t N, uint32_t a_mn_major,
                                                       uint32_t b_mn_major) {
    return (1u << 4) | (0u << 7) | (0u << 10) | (a_mn_major << 15) | (b_mn_major << 16) |
           ((N >> 3) << 17) | ((M >> 4) << 24);
}

}  // namespace cesm
