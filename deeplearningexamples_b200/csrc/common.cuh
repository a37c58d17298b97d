// Shared device helpers for the sm_100a kernels: mbarrier, TMA, tcgen05/TMEM PTX wrappers,
// counter-based RNG for dropout, bf16 packing, tanh-GELU.  Written for
// -gencode arch=compute_100a,code=sm_100a only.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#define DLE_OK 0
#define DLE_ERR_INVALID (-22)   /* EINVAL-style: bad shape / alignment / null pointer  */
#define DLE_ERR_CUDA (-5)       /* launch / driver failure (cudaGetLastError != success) */
#define DLE_ERR_NOSYS (-38)     /* feature not compiled in                              */

#define DLE_CHECK_ARG(cond) do { if (!(cond)) return DLE_ERR_INVALID; } while (0)
#define DLE_LAUNCH_CHECK() do { if (cudaGetLastError() != cudaSuccess) return DLE_ERR_CUDA; } while (0)

namespace dle {

typedef __nv_bfloat16 bf16;
typedef __nv_bfloat162 bf162;

// ---------------------------------------------------------------------------------------------
// generic
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
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
// Column sums of a 32x32 tile held one ROW per lane (v[c] = element (lane, c)): recursive halving, 31 shuffles + 31 adds.
// On return lane l holds the sum over the 32 rows of COLUMN l.
__device__ __forceinline__ float warp_column_sums32(float (&v)[32], int lane) {
#pragma unroll
    for (int half = 16; half >= 1; half >>= 1) {
        const bool hi = (lane & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float send = hi ? v[i] : v[i + half];
            const float keep = hi ? v[i + half] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
    return v[0];
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    bf162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t u) {
    bf162 t = *reinterpret_cast<bf162*>(&u);
    return __bfloat1622float2(t);
}

// ---------------------------------------------------------------------------------------------
// packed fp32x2 arithmetic (Blackwell FFMA2 / FADD2 / FMUL2: one issue slot for two lanes of work) and byte permute
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long pack_f32x2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack_f32x2(unsigned long long v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void ffma2(float& d0, float& d1, float a0, float a1, float b0, float b1, float c0, float c1) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(pack_f32x2(a0, a1)), "l"(pack_f32x2(b0, b1)), "l"(pack_f32x2(c0, c1)));
    unpack_f32x2(d, d0, d1);
}
__device__ __forceinline__ void fmul2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pack_f32x2(a0, a1)), "l"(pack_f32x2(b0, b1)));
    unpack_f32x2(d, d0, d1);
}
__device__ __forceinline__ void fadd2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pack_f32x2(a0, a1)), "l"(pack_f32x2(b0, b1)));
    unpack_f32x2(d, d0, d1);
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

// ---------------------------------------------------------------------------------------------
// math: tanh-GELU (reference modeling.py:121-122, approximate=True == tanh form)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float gelu_tanh(float x) {
    const float c = 0.7978845608028654f;
    float t = tanh_fast(c * (x + 0.044715f * x * x * x));
    return 0.5f * x * (1.0f + t);
}
// two lanes at a time on the packed-fp32 pipe (FMUL2 / FFMA2): 0.5 x (1 + tanh(c x (1 + 0.044715 x^2)))
__device__ __forceinline__ void gelu_tanh2(float x0, float x1, float& y0, float& y1) {
    const float c0 = 0.7978845608028654f, c1 = 0.7978845608028654f * 0.044715f;
    float s0, s1, a0, a1, h0, h1;
    fmul2(s0, s1, x0, x1, x0, x1);
    ffma2(s0, s1, s0, s1, c1, c1, c0, c0);
    fmul2(a0, a1, x0, x1, s0, s1);
    const float t0 = tanh_fast(a0), t1 = tanh_fast(a1);
    fmul2(h0, h1, x0, x1, 0.5f, 0.5f);
    ffma2(y0, y1, h0, h1, t0, t1, h0, h1);
}
// d/dx of the above for two lanes: 0.5 (1 + t) + 0.5 x (1 - t^2) c (1 + 3 * 0.044715 x^2),  t = tanh(c x (1 + 0.044715 x^2))
__device__ __forceinline__ void gelu_tanh_grad2(float x0, float x1, float& y0, float& y1) {
    const float c0 = 0.7978845608028654f, c1 = 0.7978845608028654f * 0.044715f, c3 = 3.0f * 0.7978845608028654f * 0.044715f;
    float s0, s1, i0, i1, a0, a1, d0, d1, q0, q1, h0, h1, r0, r1, g0, g1;
    fmul2(s0, s1, x0, x1, x0, x1);
    ffma2(i0, i1, s0, s1, c1, c1, c0, c0);
    fmul2(a0, a1, x0, x1, i0, i1);
    const float t0 = tanh_fast(a0), t1 = tanh_fast(a1);
    ffma2(d0, d1, -t0, -t1, t0, t1, 1.0f, 1.0f);            // 1 - t^2
    ffma2(q0, q1, s0, s1, c3, c3, c0, c0);                  // c (1 + 3 * 0.044715 x^2)
    fmul2(h0, h1, x0, x1, 0.5f, 0.5f);
    fmul2(r0, r1, h0, h1, d0, d1);
    ffma2(g0, g1, t0, t1, 0.5f, 0.5f, 0.5f, 0.5f);          // 0.5 (1 + t)
    ffma2(y0, y1, r0, r1, q0, q1, g0, g1);
}
__device__ __forceinline__ float gelu_tanh_grad(float x) {
    const float c = 0.7978845608028654f;
    float x2 = x * x;
    float t = tanh_fast(c * (x + 0.044715f * x * x2));
    return 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * c * (1.0f + 3.0f * 0.044715f * x2);
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-7: counter-based RNG, so forward and backward regenerate identical dropout masks
// from (seed, stream, element-group index) with no mask tensor in HBM.
// One call -> four 32-bit words -> (LCG expansion) -> keep decisions for 32 consecutive elements.
// ---------------------------------------------------------------------------------------------
template <int ROUNDS>
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0; key.y += W1;
    }
    return ctr;
}
// 32 keep-bits for the 32 consecutive elements of group `group32` (element index >> 5): ONE Philox4x32-7 call gives four
// independent 32-bit words; each word seeds a 32-bit LCG (x <- x*747796405 + 2891336453, PCG's multiplier/increment) that is
// stepped 7 times, and the top 16 bits of each state are compared with the 16-bit threshold.  The keyed, Crush-resistant
// generator decorrelates groups; inside a group the LCG's high bits are more than adequate for Bernoulli(p) decisions.
// Cost ~1.75 (Philox, amortised) + 3 instructions per element instead of ~10.
template <int ROUNDS = 7>
__device__ __forceinline__ uint32_t dropout_keep32(uint64_t seed, uint32_t stream, uint64_t group32, uint32_t thresh16) {
    const uint4 r = philox4x32<ROUNDS>(make_uint4((uint32_t)group32, (uint32_t)(group32 >> 32), stream, 0x5eed32u),
                                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t t = thresh16 << 16;
    uint32_t x[4] = {r.x, r.y, r.z, r.w};
    uint32_t m = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        uint32_t s = x[w];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            m |= (s >= t ? 1u : 0u) << (w * 8 + k);
            s = s * 747796405u + 2891336453u;
        }
    }
    return m;
}
// The same decisions for ONE byte of the group: bits [8*w, 8*w+8) of dropout_keep32(...), i.e. the keep bits of the 8 consecutive
// elements starting at (group32 << 5) + 8*w.  For kernels whose threads own 8 elements (LayerNorm, embedding): the Philox block is
// still needed in full, but only one of its four words is expanded (8 LCG steps instead of 32).
template <int ROUNDS = 7>
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t seed, uint32_t stream, uint64_t group32, int w, uint32_t thresh16) {
    const uint4 r = philox4x32<ROUNDS>(make_uint4((uint32_t)group32, (uint32_t)(group32 >> 32), stream, 0x5eed32u),
                                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t t = thresh16 << 16;
    uint32_t s = (w == 0) ? r.x : (w == 1) ? r.y : (w == 2) ? r.z : r.w;
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        m |= (s >= t ? 1u : 0u) << k;
        s = s * 747796405u + 2891336453u;
    }
    return m;
}
__host__ __device__ __forceinline__ uint32_t dropout_thresh16(float p) {
    float t = p * 65536.0f + 0.5f;
    return t <= 0.f ? 0u : (t >= 65535.f ? 65535u : (uint32_t)t);
}

// ---------------------------------------------------------------------------------------------
// dropout seeds under CUDA graphs: the host seed of a call site is frozen into a captured graph, so every dropout kernel also
// takes an optional DEVICE counter (`seed_dev`, bumped once per training step by dle_advance_u64); the effective seed is
// seed + *seed_dev * golden-ratio constant.  Forward and backward of one step read the same counter value.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long effective_seed(unsigned long long seed, const unsigned long long* seed_dev) {
    return seed_dev ? seed + __ldg(seed_dev) * 0x9E3779B97F4A7C15ull : seed;
}

// ---------------------------------------------------------------------------------------------
// Attention-probability dropout (forward and backward of the fused attention kernels): keep decisions for the 32 consecutive
// elements of group `group32`, delivered as 16 AND-masks for packed bf16x2 pairs (mask[i] covers elements 2i | 2i+1: 0xFFFF per kept
// half) -- P~ = P & mask costs one LOP3 per pair instead of a bit extract + select per element.
//   one Philox4x32-7 call -> four keyed words r_w; each is spread over four pair-words by an odd multiplier (bijective) and an
//   xor-shift (x ^ x>>16: both halfwords of the result are uniform and jointly independent); a halfword keeps its element iff its low
//   15 bits are >= t15 = round(p * 32768): (h & 0x7FFF) + (0x8000 - t15) sets bit 15 exactly then, and PRMT with sign replication
//   turns bits 15 / 31 into 0xFFFF / 0xFFFF0000.  p is therefore quantised to 1/32768; `dropout_thresh15` and the 1/(1-p) scale must
//   use the same quantised value (attn_drop_params).
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t dropout_thresh15(float p) {
    float t = p * 32768.0f + 0.5f;
    return t <= 0.f ? 0u : (t >= 32767.f ? 32767u : (uint32_t)t);
}
template <int ROUNDS = 7>
__device__ __forceinline__ void attn_dropout_masks16(unsigned long long seed, uint32_t stream, unsigned long long group32, uint32_t k2,
                                                     uint32_t (&mask)[16]) {
    const uint4 r = philox4x32<ROUNDS>(make_uint4((uint32_t)group32, (uint32_t)(group32 >> 32), stream, 0xa77d20u),
                                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t x[4] = {r.x, r.y, r.z, r.w};
    const uint32_t C[4] = {0x9E3779B1u, 0x85EBCA77u, 0xC2B2AE3Du, 0x27D4EB2Fu};
#pragma unroll
    for (int w = 0; w < 4; ++w) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t m = x[w] * C[k];
            const uint32_t y = ((m ^ (m >> 16)) & 0x7FFF7FFFu) + k2;
            mask[w * 4 + k] = prmt(y, 0u, 0xBB99u);
        }
    }
}
__host__ __device__ __forceinline__ uint32_t attn_dropout_k2(uint32_t thresh15) { return (0x8000u - thresh15) * 0x00010001u; }

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Wait for the phase with the given parity.  try_wait is given a suspend-time hint so that the hardware parks the waiting
// thread until the phase flips instead of returning after the (short) default limit: ncu showed ~30 % of all executed warp
// instructions of the attention kernels were TRYWAIT/BRA/YIELD iterations of single-lane producer / MMA-issuer waits, competing
// for issue slots with the softmax warps of the same SM sub-partition.
// Watchdog: a wait that has not completed after 4 s of wall clock (kernels here last milliseconds) is a protocol bug; trap so the
// launch fails with an error instead of hanging the GPU.
// Suspend-time hint of mbarrier.try_wait: 0 = none (the hardware's default time limit per attempt), else nanoseconds.  Round 1 used
// 10 ms to park single-lane waiters; since the producer / MMA warps wait warp-wide (see gemm_sm100.cu) the un-hinted form measures
// 0.6 % faster on the whole step and 3 % on attention backward (profiles/README.md, same-box A/B), so it is the default; gemm_sm100.cu
// defines the macro before including this header because the hinted form is the faster one for its long waits.
#ifndef DLE_MBAR_HINT_NS
#define DLE_MBAR_HINT_NS 0
#endif
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t addr, uint32_t parity) {
    uint32_t ok;
#if DLE_MBAR_HINT_NS
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n" : "=r"(ok) : "r"(addr), "r"(parity), "r"((uint32_t)DLE_MBAR_HINT_NS) : "memory");
#else
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n" : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
#endif
    return ok;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    if (mbar_try_wait(addr, parity)) return;
    const unsigned long long t0 = global_timer_ns();
    while (!mbar_try_wait(addr, parity)) {
        if (global_timer_ns() - t0 > 4000000000ull) __trap();
    }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// arrive on an mbarrier given by its shared::cluster address (mapa_shared), e.g. one in the peer CTA of a pair
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

// ---------------------------------------------------------------------------------------------
// clusters
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// every thread of every CTA of the cluster: arrive (release) + wait (acquire)
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the variable at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
// generic-proxy smem writes -> visible to the async proxy (TMA / tcgen05 operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor), 2D tiles, completion on an mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// CTA-pair form (tcgen05 cta_group::2): the data lands in THIS CTA's shared memory, the completed bytes are counted on the mbarrier at
// `bar_cluster` (a shared::cluster address, which may lie in the peer CTA)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N> __device__ __forceinline__ void tma_store_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// tcgen05.commit: arrive on `bar` once all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; bf16 in, fp32 accumulate
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// CTA-pair (cta_group::2) forms.  All tcgen05 instructions of one kernel must use the same cta_group.  alloc / relinquish / dealloc
// are executed collectively by one warp of EACH CTA of the pair and give both CTAs the same TMEM address.  The MMA is issued by the
// even CTA only: A (M = 256) is its 128 rows in each CTA's shared memory, B is N/2 rows in each, at the same offsets, and each CTA's
// TMEM receives its own 128 rows of D.
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrive on the mbarrier at this offset in BOTH CTAs of the pair once all previously issued MMAs have completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)0x3) : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32 (cute::UMMA::InstrDescriptor bit layout:
// c_format [4,6)=1 (F32), a_format [7,10)=1 (BF16), b_format [10,13)=1, a_major bit 15, b_major bit 16
// (0 = K-major, 1 = MN-major), n_dim [17,23) = N>>3, m_dim [24,29) = M>>4).
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, bool a_mn, bool b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type [61,64) (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) |
           ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (one row per thread)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
          "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
          "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// cp.async (LDGSTS): 16 bytes global -> shared without staging registers; groups are committed / waited per thread
__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
    uint4 r;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
    return r;
}

// 16-byte global store / load helpers
__device__ __forceinline__ void st_global_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_global_nc_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void red_add_v4_f32(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

}  // namespace dle

// ---------------------------------------------------------------------------------------------
// host: TMA descriptor encode through the driver entry point (no -lcuda link dependency)
// ---------------------------------------------------------------------------------------------
namespace dle {
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();
// bf16 row-major matrix [rows, cols] with leading dimension ld (elements); box = {box_cols, box_rows};
// 128B swizzle (box_cols * 2 bytes must be <= 128).
int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_cols, uint32_t box_rows);
}  // namespace dle
