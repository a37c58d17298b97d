// Dense bf16 GEMM for sm_100a: tcgen05.mma on CTA pairs (cta_group::2, M = 256) with fp32 accumulators in TMEM,
// operands staged by TMA into 128B-swizzled shared memory, persistent warp-specialised CTAs launched in clusters of 2
// (1 TMA producer warp, 1 MMA issuer warp, 8 or 16 epilogue warps per CTA), double-buffered accumulators so the
// epilogue of tile i overlaps the main loop of tile i+1.
//
//   D[M,N] = A[M,K] * B[N,K]^T     (K = reduction)
//
// A work unit is a 256 x BN output tile (and a K range, under split-K) shared by the two CTAs of a cluster: the even CTA
// owns rows 0-127 of the tile, the odd CTA rows 128-255.  Each CTA loads its own 128 rows of A and HALF of B (BN/2 rows),
// so per flop an SM moves a third less operand data out of L2 and reads a third less shared memory for the MMA than a
// 128 x BN tile per SM; one 256 x BN x 16 MMA issued by the even CTA serves both SMs, and each SM's TMEM receives its
// own 128 rows of D.
//
// Either operand may be "K-major" (row-major [rows, K], the reduction dim contiguous) or
// "MN-major" (row-major [K, rows], the M/N dim contiguous) so forward (x W^T), dgrad (dy W) and
// wgrad (dy^T x) all read the tensors where they lie -- no transposed copies in HBM.
//
// This replaces the cuBLAS calls behind the reference's F.linear sites
// (PyTorch/LanguageModeling/BERT/modeling.py:160,345-347,395,431,553) and fuses the reference's
// separate pointwise passes (bias, tanh-GELU :121-122, dropout+residual :396-397/:432-433) into
// the epilogue.
// mbarrier waits of THIS kernel carry a suspend-time hint (the hardware parks the waiting warp instead of re-polling): the epilogue warps
// wait ~2000 clk per tile for an accumulator, the producer waits on nearly every k-block for a free stage.  Same-box A/B on the whole step,
// hint here only vs nowhere: GEMM launches 1211 -> 1224 TFLOP/s, 856.6 -> 859.3 seq/s (profiles/r02_gemm_mbar_hint_ab.log); the attention
// kernels measure faster un-hinted (common.cuh) and keep the default.
#ifndef DLE_MBAR_HINT_NS
#define DLE_MBAR_HINT_NS 0x989680
#endif
#include "common.cuh"
#include "../../include/dle_b200.h"

namespace dle {

constexpr int BM = 128;      // rows of a tile per CTA; a pair tile has 2 * BM
constexpr int BK = 64;        // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
// Epilogue warps (template parameter EW): 8 (two per TMEM lane quarter, each draining half the columns) or 16 (four per quarter, a
// quarter of the columns each, <= 104 registers per thread).  With one 128 x BN tile per SM (a 48 KB stage at BN = 256) the 16-warp
// instance had to drop to 3 stages and only paid for the gelu'(u)-times-dgrad epilogue (profiles/r02_gemm_microbench_run7_*.log); a
// CTA's share of a pair stage is 32 KB, so 16 warps now cost one stage of six, not one of four.  Which epilogues take 16 warps:
// DLE_GEMM_EW16_EPILOGUES (bit mask over DLE_EPI_*; a compile-time switch so that variants can be built and measured side by side).
// Warp roles: epilogue warps 0..EW-1, then TMA, MMA, TMEM alloc (+ a spare with 8).  The single-issuer warps carry the HIGHEST
// warp ids: the SM sub-partition arbiter favours higher warp ids, and a starved MMA issuer idles the tensor pipe.
template <int BN, int EW> struct GemmCfg {
    static_assert(EW == 8 || EW == 16, "epilogue warps: 8 or 16");
    static constexpr int EPI_WARPS = EW;
    static constexpr int EPI_PARTS = EW / 4;                        // column parts per tile (one per warp of a quarter)
    static constexpr int THREADS = (EW == 8) ? 384 : 608;
    static constexpr int WARP_TMA = EW, WARP_MMA = EW + 1, WARP_ALLOC = EW + 2;
    static constexpr int A_BYTES = BM * BK * 2;                     // this CTA's 128 rows of A
    static constexpr int B_BYTES = (BN / 2) * BK * 2;               // this CTA's half of B
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;           // per CTA; a pair stage is twice this
    static constexpr int STAGES = (BN == 256) ? (EW == 8 ? 6 : 5) : (EW == 8 ? 8 : 6);
    static constexpr int TMEM_COLS = 2 * BN;            // double-buffered accumulator (128 lanes x BN columns each, in each CTA)
    // epilogue: per warp a 2 KB output staging tile + a 2 KB cp.async landing tile for the residual / pre-activation operand,
    // plus 3 x 2 x 256 B of bias staging (triple-buffered per tile, one slice per column half)
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_WARPS * 2048 + EPI_WARPS * 2048 + 1536 + 1024 /*align slack*/ + 256 /*barriers*/;
    static_assert(SMEM_BYTES <= 232448, "shared memory budget");
    static_assert((2 * STAGES + 4) * 8 + 4 <= 256, "barrier area");
};

#ifndef DLE_GEMM_EW16_EPILOGUES
#define DLE_GEMM_EW16_EPILOGUES (1u << DLE_EPI_DGELU)
#endif

struct GemmKernelParams {
    int M, N, K;
    int m_tiles, n_tiles, splits, kb_total;   // m_tiles: 256-row pair tiles
    int epilogue;
    const bf16* bias;      // [N] or null
    const bf16* aux;       // [M, ld_aux] residual / pre-activation, or null
    void* out;             // bf16 [M, ldo] (or fp32 for DLE_EPI_ATOMIC_F32 / DLE_EPI_F32)
    bf16* out2;            // second output (pre-activation for DLE_EPI_BIAS_GELU)
    long long ldo, ld_aux, ldo2;
    float drop_scale;      // 1/(1-p)
    uint32_t drop_thresh;  // 16-bit threshold, 0 = dropout off
    uint32_t drop_stream;
    unsigned long long seed;
    const unsigned long long* seed_dev;
    float alpha;
    float* colsum_out;     // [N] fp32 or null: += column sums of the (bf16-rounded) output, e.g. the bias gradient of the layer below
};

// ----------------------------------------------------------------------------------------------
// epilogue.  A TMEM load hands every thread 32 consecutive columns of ITS OWN row, so a direct 16-byte global
// access per thread would touch 32 different 128-byte lines per warp instruction (measured: the bias+GELU epilogue
// with two outputs ran at 53 % of peak, dropout+residual at 49 %).  Each epilogue warp therefore owns two 32 x 64 B
// tiles in shared memory, 16-byte units XOR-swizzled by (row >> 1) & 3 so that both access patterns are conflict-free:
//   out tile:  lane writes its row (4 x STS.128) -> __syncwarp -> lanes re-read as (row = it*8 + lane/4, unit = lane%4)
//              -> each ST.GLOBAL.128 covers 8 rows x 64 contiguous bytes
//   aux tile:  the residual / pre-activation operand of the NEXT chunk lands here by cp.async (row-contiguous, no registers)
//              while the current chunk is computed and stored; ncu showed 27 % of the dropout+residual epilogue's samples
//              waiting on that load when it was issued in line.
// The bias slice of the tile is staged once per tile (before the accumulator wait) instead of re-read from global per
// chunk (8.5 % of the bias+GELU epilogue's samples).  fp32 outputs (split-K atomics, logits) keep the direct path.
// ----------------------------------------------------------------------------------------------
constexpr int EPI_TILE_BYTES = 32 * 64;                 // per epilogue warp, out and aux each
constexpr int EPI_BIAS_BYTES = 3 * 512;                 // [tile % 3][column part][BN / EPI_PARTS bf16], BN <= 256

__device__ __forceinline__ uint32_t epi_off(int row, int unit) { return (uint32_t)(row * 64 + ((unit ^ ((row >> 1) & 3)) << 4)); }

__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
    uint4 r;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void cp_async_16(uint32_t smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// EPL (1, 2 or 4) consecutive bias values of one lane: global -> registers -> the staged slice
template <int EPL> __device__ __forceinline__ uint2 bias_load(const bf16* src) {
    uint2 r = make_uint2(0u, 0u);
    if constexpr (EPL == 4) r = *reinterpret_cast<const uint2*>(src);
    else if constexpr (EPL == 2) r.x = *reinterpret_cast<const uint32_t*>(src);
    else r.x = *reinterpret_cast<const unsigned short*>(src);
    return r;
}
template <int EPL> __device__ __forceinline__ void bias_stage(uint32_t slice, int lane, uint2 b) {
    if constexpr (EPL == 4) asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(slice + lane * 8), "r"(b.x), "r"(b.y) : "memory");
    else if constexpr (EPL == 2) asm volatile("st.shared.b32 [%0], %1;" ::"r"(slice + lane * 4), "r"(b.x) : "memory");
    else asm volatile("st.shared.u16 [%0], %1;" ::"r"(slice + lane * 2), "h"((unsigned short)b.x) : "memory");
}

// start the copy of rows [row_base, +32) x cols [col0, +32) of the bf16 aux matrix into this warp's aux tile
__device__ __forceinline__ void aux_prefetch(const GemmKernelParams& p, long long row_base, int col0, uint32_t aux_tile, int lane) {
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int rr = it * 8 + (lane >> 2), cc = lane & 3;
        const long long grow = row_base + rr; const int gcol = col0 + cc * 8;
        if (grow < p.M && gcol < p.N) cp_async_16(aux_tile + epi_off(rr, cc), p.aux + grow * p.ld_aux + gcol);
    }
}
// this lane's row of the landed aux tile, still packed (4 x 8 bf16)
__device__ __forceinline__ void aux_take(uint32_t aux_tile, int lane, uint4 (&a)[4]) {
    cp_async_wait_all();
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 4; ++c) a[c] = lds_v4(aux_tile + epi_off(lane, c));
    __syncwarp();
}
// this lane's row (32 floats) -> bf16 rows [row_base, +32) x cols [col0, +32) of dst, row-contiguous global stores
__device__ __forceinline__ void warp_store_rows(bf16* __restrict__ dst, long long ld, long long row_base, int col0, int M, int N,
                                                uint32_t stage, int lane, const float (&v)[32]) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
        sts_v4(stage + epi_off(lane, c), pack_bf16(v[c * 8], v[c * 8 + 1]), pack_bf16(v[c * 8 + 2], v[c * 8 + 3]),
               pack_bf16(v[c * 8 + 4], v[c * 8 + 5]), pack_bf16(v[c * 8 + 6], v[c * 8 + 7]));
    __syncwarp();
    uint4 w[4];                                  // all four shared loads first: the asm statements keep program order, and a load
#pragma unroll                                   // immediately followed by its store exposes the shared-memory latency four times
    for (int it = 0; it < 4; ++it) w[it] = lds_v4(stage + epi_off(it * 8 + (lane >> 2), lane & 3));
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int rr = it * 8 + (lane >> 2), cc = lane & 3;
        const long long grow = row_base + rr; const int gcol = col0 + cc * 8;
        if (grow < M && gcol < N) st_global_v4(dst + grow * ld + gcol, w[it].x, w[it].y, w[it].z, w[it].w);
    }
    __syncwarp();
}
__device__ __forceinline__ void unpack8(const uint4& w, float* o) {
    float2 f;
    f = unpack_bf16(w.x); o[0] = f.x; o[1] = f.y;
    f = unpack_bf16(w.y); o[2] = f.x; o[3] = f.y;
    f = unpack_bf16(w.z); o[4] = f.x; o[5] = f.y;
    f = unpack_bf16(w.w); o[6] = f.x; o[7] = f.y;
}

// one 32-row x 32-column chunk of one epilogue warp; `row` = this lane's row, row_base = first row of the warp.
// bias_s = shared address of this chunk's 32 staged bias values; aux = this lane's row of the aux operand (packed bf16).
__device__ __forceinline__ void epilogue_chunk(const GemmKernelParams& p, const uint32_t (&acc)[32], const uint4 (&aux)[4], long long row_base,
                                               int lane, int col0, uint32_t stage, uint32_t bias_s, unsigned long long seed) {
    const long long row = row_base + lane;
    float v[32];
    if (p.alpha != 1.0f) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(acc[i]) * p.alpha;
    } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(acc[i]);
    }
    const int ncols = min(32, p.N - col0);      // multiple of 8 (N % 8 == 0 is enforced); <= 0 for an out-of-range chunk
    if (ncols <= 0) return;                      // warp-uniform

    if (p.epilogue == DLE_EPI_ATOMIC_F32) {
        if (row < p.M) {
            float* o = reinterpret_cast<float*>(p.out) + row * p.ldo + col0;
#pragma unroll
            for (int i = 0; i < 32; i += 4)
                if (i < ncols) red_add_v4_f32(o + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
        return;
    }
    if (p.bias != nullptr) {                     // staged slice is zero-filled beyond N
        uint4 bw[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) bw[i] = lds_v4(bias_s + i * 16);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float b[8];
            unpack8(bw[i], b);
#pragma unroll
            for (int k = 0; k < 8; ++k) v[i * 8 + k] += b[k];
        }
    }
    if (p.epilogue == DLE_EPI_F32) {
        if (row < p.M) {
            float* o = reinterpret_cast<float*>(p.out) + row * p.ldo + col0;
#pragma unroll
            for (int i = 0; i < 32; i += 4)
                if (i < ncols) *reinterpret_cast<float4*>(o + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
        return;
    }
    if (p.epilogue == DLE_EPI_BIAS_GELU) {
        // out2 = pre-activation u (needed by gelu' in backward), out = gelu(u).  gelu is evaluated on the bf16-rounded
        // pre-activation so that backward (which only has the stored bf16 u) differentiates what forward evaluated.
        warp_store_rows(p.out2, p.ldo2, row_base, col0, p.M, p.N, stage, lane, v);
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            const uint32_t u2 = pack_bf16(v[i], v[i + 1]);       // the bf16 pair just stored
            gelu_tanh2(__uint_as_float(u2 << 16), __uint_as_float(u2 & 0xFFFF0000u), v[i], v[i + 1]);
        }
    } else if (p.epilogue == DLE_EPI_BIAS_DROPOUT_RESIDUAL) {
        if (p.drop_thresh != 0) {
            const uint32_t keep = dropout_keep32(seed, p.drop_stream, (unsigned long long)(row * (long long)p.N + col0) >> 5, p.drop_thresh);
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = ((keep >> i) & 1u) ? v[i] * p.drop_scale : 0.f;
        }
        if (p.aux != nullptr) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float a[8];
                unpack8(aux[c], a);
#pragma unroll
                for (int k = 0; k < 8; ++k) v[c * 8 + k] += a[k];
            }
        }
    } else if (p.epilogue == DLE_EPI_DGELU) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float a[8];                                     // stored pre-activation u
            unpack8(aux[c], a);
#pragma unroll
            for (int k = 0; k < 8; k += 2) {
                float g0, g1;
                gelu_tanh_grad2(a[k], a[k + 1], g0, g1);
                fmul2(v[c * 8 + k], v[c * 8 + k + 1], v[c * 8 + k], v[c * 8 + k + 1], g0, g1);
            }
        }
    } else if (p.epilogue == DLE_EPI_ADD) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float a[8];
            unpack8(aux[c], a);
#pragma unroll
            for (int k = 0; k < 8; ++k) v[c * 8 + k] += a[k];
        }
    } else if (p.epilogue == DLE_EPI_BIAS_TANH) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = tanhf(v[i]);
    }
    warp_store_rows(reinterpret_cast<bf16*>(p.out), p.ldo, row_base, col0, p.M, p.N, stage, lane, v);
    if (p.colsum_out != nullptr) {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = (row < p.M) ? __bfloat162float(__float2bfloat16_rn(v[i])) : 0.f;
        const float cs = warp_column_sums32(v, lane);
        if (lane < ncols) atomicAdd(p.colsum_out + col0 + lane, cs);
    }
}

// ----------------------------------------------------------------------------------------------
// kernel
// ----------------------------------------------------------------------------------------------
template <int BN, bool A_MN, bool B_MN, int EW>
__global__ void __launch_bounds__((GemmCfg<BN, EW>::THREADS), 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const GemmKernelParams p) {
    using Cfg = GemmCfg<BN, EW>;
    constexpr int EPI_WARPS = Cfg::EPI_WARPS, EPI_PARTS = Cfg::EPI_PARTS;
    constexpr int WARP_TMA = Cfg::WARP_TMA, WARP_MMA = Cfg::WARP_MMA, WARP_ALLOC = Cfg::WARP_ALLOC;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* epi_stage = smem + Cfg::STAGES * Cfg::STAGE_BYTES;                 // 8 warps x (out tile, aux tile), then the bias slices
    uint8_t* epi_bias = epi_stage + 2 * EPI_WARPS * EPI_TILE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(epi_bias + EPI_BIAS_BYTES);
    // Barriers exist in both CTAs at the same offsets; full_bar and tmem_empty are only used in the even (leader) CTA.
    uint64_t* full_bar = bars;                         // [STAGES]  TMA of both CTAs -> MMA
    uint64_t* empty_bar = bars + Cfg::STAGES;          // [STAGES]  MMA -> TMA of each CTA (multicast commit)
    uint64_t* tmem_full = bars + 2 * Cfg::STAGES;      // [2]       MMA -> epilogue of each CTA (multicast commit)
    uint64_t* tmem_empty = bars + 2 * Cfg::STAGES + 2; // [2]       epilogue warps of both CTAs -> MMA
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * Cfg::STAGES + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();           // 0: rows 0-127 of every pair tile, issues the MMAs; 1: rows 128-255
    const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_b);
        for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 2 * EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == WARP_ALLOC) { tmem_alloc_pair(tmem_ptr, Cfg::TMEM_COLS); tmem_relinquish_pair(); }
    tc_fence_before();
    cluster_sync();                                    // the peer's barriers are initialised before anything signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    const int total_units = p.m_tiles * p.n_tiles * p.splits;
    const int kb_per_split = (p.kb_total + p.splits - 1) / p.splits;

    // The producer and MMA warps run their loops WARP-UNIFORMLY (all 32 lanes wait on the barriers) and only the tcgen05 / TMA
    // instructions sit under elect_one(): inside an `if (lane == 0)` region ptxas cannot keep descriptors and addresses in uniform
    // registers and wraps every UTCHMMA / UTMALDG in an ELECT + R2UR + BRA.U.ANY waterfall (11-16 instructions per MMA, measured on the
    // attention kernels as an MMA-issue-bound tensor pipe at 18 %); warp-uniform flow issues consecutive MMAs back to back.
    if (warp == WARP_TMA) {
        // ===================== TMA producer (both CTAs; completions counted on the leader's full_bar) =====================
        int stage = 0; uint32_t phase = 0;
        for (int unit = pair; unit < total_units; unit += num_pairs) {
            const int tile = unit / p.splits, split = unit - tile * p.splits;
            const int m_pair = tile / p.n_tiles, n_blk = tile - m_pair * p.n_tiles;
            const int row0 = (m_pair * 2 + (int)rank) * BM, col0 = n_blk * BN + (int)rank * (BN / 2);
            const int kb0 = split * kb_per_split, kb1 = min(p.kb_total, kb0 + kb_per_split);
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                if (elect_one()) {
                    const uint32_t fb = mapa_shared(smem_u32(&full_bar[stage]), 0);
                    if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);   // both CTAs' bytes
                    uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
                    uint8_t* sb = sa + Cfg::A_BYTES;
                    if (!A_MN) {
                        tma_load_2d_pair(sa, &tmap_a, fb, kb * BK, row0);
                    } else {
#pragma unroll
                        for (int g = 0; g < BM / 64; ++g)
                            tma_load_2d_pair(sa + g * (BK * 128), &tmap_a, fb, row0 + g * 64, kb * BK);
                    }
                    if (!B_MN) {
                        tma_load_2d_pair(sb, &tmap_b, fb, kb * BK, col0);
                    } else {
#pragma unroll
                        for (int g = 0; g < BN / 128; ++g)
                            tma_load_2d_pair(sb + g * (BK * 128), &tmap_b, fb, col0 + g * 64, kb * BK);
                    }
                }
                __syncwarp();
                if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
            }
        }
        // The leader's MMA commits still arrive on this CTA's empty_bar after the last load: wait for every stage in flight so that
        // no commit targets the shared memory of a CTA that has exited.
        for (int s = 0; s < Cfg::STAGES; ++s) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
        }
    } else if (warp == WARP_MMA) {
        // ===================== MMA issuer (leader CTA only; one elected lane issues, the warp waits together) =====================
        if (rank == 0) {
            constexpr uint32_t idesc = make_idesc_bf16(2 * BM, BN, A_MN, B_MN);
            int stage = 0; uint32_t phase = 0; int it = 0;
            const uint32_t smem_base = smem_u32(smem);
            for (int unit = pair; unit < total_units; unit += num_pairs, ++it) {
                const int split = unit % p.splits;
                const int kb0 = split * kb_per_split, kb1 = min(p.kb_total, kb0 + kb_per_split);
                const int acc = it & 1; const uint32_t acc_phase = (it >> 1) & 1;
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t sa = smem_base + stage * Cfg::STAGE_BYTES;
                        const uint32_t sb = sa + Cfg::A_BYTES;
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k) {
                            // K-major:  rows of 128 B, 8-row groups 1024 B apart (SBO); advance 32 B per UMMA_K.
                            // MN-major: k-rows of 128 B (64 m/n elements), 8-k-row groups 1024 B apart (SBO),
                            //           next 64 m/n elements BK*128 B further (LBO); advance 16 k-rows = 2048 B.
                            const uint64_t da = A_MN ? make_smem_desc_sw128(sa + k * (UMMA_K * 128), BK * 128, 1024)
                                                     : make_smem_desc_sw128(sa + k * (UMMA_K * 2), 0, 1024);
                            const uint64_t db = B_MN ? make_smem_desc_sw128(sb + k * (UMMA_K * 128), BK * 128, 1024)
                                                     : make_smem_desc_sw128(sb + k * (UMMA_K * 2), 0, 1024);
                            umma_bf16_ss_pair(tmem_d, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
                        }
                        umma_commit_pair(&empty_bar[stage]);      // frees this smem stage in both CTAs when the MMAs retire
                        if (kb + 1 == kb1) umma_commit_pair(&tmem_full[acc]);     // accumulator complete -> both epilogues
                    }
                    __syncwarp();
                    if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
                }
                if (kb1 <= kb0) {                        // (cannot happen: the launcher never creates an empty split) keep the epilogue's wait finite
                    if (elect_one()) umma_commit_pair(&tmem_full[acc]);
                    __syncwarp();
                }
            }
        }
    } else if (warp < EPI_WARPS) {
        // ===================== epilogue warps (TMEM -> registers -> global), this CTA's 128 rows of the pair tile =====================
        const int q = warp & 3;                          // TMEM lane quarter this warp may access (hardware rule: warp id % 4)
        const int half = warp >> 2;                      // column part: the EPI_PARTS warps of a quarter each drain BN / EPI_PARTS columns
        constexpr int PART_COLS = BN / EPI_PARTS;        // columns per warp per tile
        constexpr int CH = PART_COLS / 32;               // 32-column chunks per warp per tile
        constexpr int EPL = PART_COLS / 32;              // bias elements staged per lane (1, 2 or 4)
        constexpr int SLICE = PART_COLS * 2;             // bytes of one staged bias slice
        const uint32_t out_tile = smem_u32(epi_stage) + warp * 2 * EPI_TILE_BYTES;
        const uint32_t aux_tile = out_tile + EPI_TILE_BYTES;
        const uint32_t tmem_empty_leader = mapa_shared(smem_u32(tmem_empty), 0);
        const unsigned long long seed = (p.drop_thresh != 0u) ? effective_seed(p.seed, p.seed_dev) : 0ull;
        const bool use_aux = p.aux != nullptr && (p.epilogue == DLE_EPI_BIAS_DROPOUT_RESIDUAL || p.epilogue == DLE_EPI_DGELU ||
                                                  p.epilogue == DLE_EPI_ADD);
        if (use_aux && pair < total_units) {             // operand of the very first chunk
            const int tile = pair / p.splits;
            const int m_pair = tile / p.n_tiles, n_blk = tile - m_pair * p.n_tiles;
            aux_prefetch(p, (long long)(m_pair * 2 + (int)rank) * BM + q * 32, n_blk * BN + half * PART_COLS, aux_tile, lane);
        }
        int it = 0;
        for (int unit = pair; unit < total_units; unit += num_pairs, ++it) {
            const int tile = unit / p.splits;
            const int m_pair = tile / p.n_tiles, n_blk = tile - m_pair * p.n_tiles;
            const int acc = it & 1; const uint32_t acc_phase = (it >> 1) & 1;
            // bias slice of this warp's column half -> shared.  The slice of tile it+1 is fetched into two registers at the top of tile it
            // and stored after its last chunk, so the global latency never sits in front of the accumulator (in the epilogue-bound
            // regime the accumulator is already waiting).  The four warps of a half write the same values into the same slice; slices
            // rotate over three tiles because a warp can run at most one tile ahead of a sibling (tmem_empty needs all arrivals).
            const uint32_t bias_s = smem_u32(epi_bias) + ((it % 3) * EPI_PARTS + half) * SLICE;
            const uint32_t bias_next = smem_u32(epi_bias) + (((it + 1) % 3) * EPI_PARTS + half) * SLICE;
            uint2 bnext = make_uint2(0u, 0u);
            const bool has_next = p.bias != nullptr && unit + num_pairs < total_units;
            if (p.bias != nullptr) {
                if (it == 0) {
                    uint2 b0 = make_uint2(0u, 0u);
                    const int col = n_blk * BN + half * PART_COLS + lane * EPL;
                    if (col < p.N) b0 = bias_load<EPL>(p.bias + col);
                    bias_stage<EPL>(bias_s, lane, b0);
                    __syncwarp();
                }
                if (has_next) {
                    const int tile2 = (unit + num_pairs) / p.splits;
                    const int n2 = tile2 - (tile2 / p.n_tiles) * p.n_tiles;
                    const int col = n2 * BN + half * PART_COLS + lane * EPL;
                    if (col < p.N) bnext = bias_load<EPL>(p.bias + col);
                }
            }
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const long long row_base = (long long)(m_pair * 2 + (int)rank) * BM + q * 32;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN;
#pragma unroll 1
            for (int cl = 0; cl < CH; ++cl) {
                const int c = half * CH + cl;
                uint32_t r[32];
                tmem_ld32(taddr + c * 32, r);
                uint4 a[4];
                if (use_aux) {
                    aux_take(aux_tile, lane, a);             // landed while the previous chunk was computed / stored
                    if (cl + 1 < CH) {
                        aux_prefetch(p, row_base, n_blk * BN + (c + 1) * 32, aux_tile, lane);
                    } else if (unit + num_pairs < total_units) {
                        const int tile2 = (unit + num_pairs) / p.splits;
                        const int m2 = tile2 / p.n_tiles, n2 = tile2 - m2 * p.n_tiles;
                        aux_prefetch(p, (long long)(m2 * 2 + (int)rank) * BM + q * 32, n2 * BN + half * PART_COLS, aux_tile, lane);
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) a[k] = make_uint4(0u, 0u, 0u, 0u);
                }
                tmem_ld_wait();
                if (row_base < p.M) epilogue_chunk(p, r, a, row_base, lane, n_blk * BN + c * 32, out_tile, bias_s + cl * 64, seed);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tmem_empty_leader + acc * 8);    // one arrival per epilogue warp of the pair
            if (has_next) {
                bias_stage<EPL>(bias_next, lane, bnext);
                __syncwarp();
            }
        }
    }

    // No CTA leaves (or frees its TMEM) while its peer can still signal its barriers or write its TMEM.
    tc_fence_before();
    cluster_sync();
    if (warp == WARP_ALLOC) { tc_fence_after(); tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS); }
}

// ----------------------------------------------------------------------------------------------
// host
// ----------------------------------------------------------------------------------------------
PFN_encodeTiled get_encode_tiled() {
    static PFN_encodeTiled fn = nullptr;
    if (fn == nullptr) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = reinterpret_cast<PFN_encodeTiled>(ptr);
    }
    return fn;
}

int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_cols, uint32_t box_rows) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (enc == nullptr) return DLE_ERR_CUDA;
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld * 2) % 16 != 0 || box_cols * 2 > 128 || box_rows > 256)
        return DLE_ERR_INVALID;
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstride[1] = {ld * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? DLE_OK : DLE_ERR_CUDA;
}

static int num_sms() {
    static int sms[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 148;
    if (sms[dev] == 0) {
        cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
        if (sms[dev] <= 0) sms[dev] = 148;
    }
    return sms[dev];
}

template <int BN, bool A_MN, bool B_MN, int EW>
static int launch_gemm_ew(const dle_gemm_args* a, cudaStream_t stream) {
    using Cfg = GemmCfg<BN, EW>;
    CUtensorMap ta, tb;
    int rc;
    // K-major operand: matrix [rows, K] -> box {64 (k), rows per CTA}; MN-major: matrix [K, rows] -> box {64 (m/n), 64 (k)}.
    // Per CTA of a pair: 128 rows of A, BN / 2 rows of B.
    rc = A_MN ? make_tmap_bf16_2d(&ta, a->A, a->K, a->M, a->lda, 64, BK) : make_tmap_bf16_2d(&ta, a->A, a->M, a->K, a->lda, BK, BM);
    if (rc != DLE_OK) return rc;
    rc = B_MN ? make_tmap_bf16_2d(&tb, a->B, a->K, a->N, a->ldb, 64, BK) : make_tmap_bf16_2d(&tb, a->B, a->N, a->K, a->ldb, BK, BN / 2);
    if (rc != DLE_OK) return rc;

    GemmKernelParams p;
    p.M = a->M; p.N = a->N; p.K = a->K;
    p.m_tiles = (a->M + 2 * BM - 1) / (2 * BM);
    p.n_tiles = (a->N + BN - 1) / BN;
    p.kb_total = (a->K + BK - 1) / BK;
    int splits = a->splits > 0 ? a->splits : 1;
    if (a->epilogue != DLE_EPI_ATOMIC_F32) splits = 1;
    if (splits > p.kb_total) splits = p.kb_total;
    // no empty split: shrink until ceil-division leaves work for the last one
    while (splits > 1 && (splits - 1) * ((p.kb_total + splits - 1) / splits) >= p.kb_total) --splits;
    p.splits = splits;
    p.epilogue = a->epilogue;
    p.bias = reinterpret_cast<const bf16*>(a->bias);
    p.aux = reinterpret_cast<const bf16*>(a->aux);
    p.out = a->out;
    p.out2 = reinterpret_cast<bf16*>(a->out2);
    p.ldo = a->ldo; p.ld_aux = a->ld_aux; p.ldo2 = a->ldo2;
    p.drop_thresh = (a->dropout_p > 0.f) ? dropout_thresh16(a->dropout_p) : 0u;
    p.drop_scale = (a->dropout_p > 0.f) ? 1.0f / (1.0f - a->dropout_p) : 1.0f;
    p.drop_stream = a->dropout_stream;
    p.seed = a->seed;
    p.seed_dev = reinterpret_cast<const unsigned long long*>(a->seed_dev);
    p.alpha = a->alpha;
    p.colsum_out = reinterpret_cast<float*>(a->colsum_out);

    auto kern = gemm_bf16_tcgen05_kernel<BN, A_MN, B_MN, EW>;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(Cfg::THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = stream;
    cfg.attrs = attr; cfg.numAttrs = 1;
    // per device (and per template instance): the shared-memory attribute, and how many pairs can be resident at once -- a persistent
    // grid larger than that would run its last pairs as a second wave
    static int pair_slots[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return DLE_ERR_CUDA;
    if (pair_slots[dev] == 0) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES) != cudaSuccess)
            return DLE_ERR_CUDA;
        int clusters = 0;
        cfg.gridDim = dim3(2 * (num_sms() / 2));
        if (cudaOccupancyMaxActiveClusters(&clusters, kern, &cfg) != cudaSuccess || clusters <= 0) return DLE_ERR_CUDA;
        pair_slots[dev] = clusters < num_sms() / 2 ? clusters : num_sms() / 2;
    }
    const int units = p.m_tiles * p.n_tiles * p.splits;
    cfg.gridDim = dim3(2 * (units < pair_slots[dev] ? units : pair_slots[dev]));
    if (cudaLaunchKernelEx(&cfg, kern, ta, tb, p) != cudaSuccess) return DLE_ERR_CUDA;
    DLE_LAUNCH_CHECK();
    return DLE_OK;
}

template <int BN, bool A_MN, bool B_MN>
static int launch_gemm(const dle_gemm_args* a, cudaStream_t stream) {
    // 16 epilogue warps only where they pay (see GemmCfg)
    if ((DLE_GEMM_EW16_EPILOGUES >> a->epilogue) & 1u) return launch_gemm_ew<BN, A_MN, B_MN, 16>(a, stream);
    return launch_gemm_ew<BN, A_MN, B_MN, 8>(a, stream);
}

}  // namespace dle

extern "C" int dle_gemm_bf16(const dle_gemm_args* a, void* stream_) {
    using namespace dle;
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
    DLE_CHECK_ARG(a != nullptr && a->A != nullptr && a->B != nullptr && a->out != nullptr);
    DLE_CHECK_ARG(a->M > 0 && a->N > 0 && a->K > 0);
    // N % 8: the epilogue stores 16-byte vectors; lda/ldb % 8: TMA row strides are multiples of 16 bytes.
    // M and K are otherwise free (TMA zero-fills out-of-bounds rows/columns of partial tiles).
    DLE_CHECK_ARG(a->N % 8 == 0 && a->ldo % 8 == 0 && a->lda % 8 == 0 && a->ldb % 8 == 0);
    DLE_CHECK_ARG(a->epilogue >= 0 && a->epilogue < DLE_EPI_COUNT);
    if (a->epilogue == DLE_EPI_BIAS_DROPOUT_RESIDUAL && a->dropout_p > 0.f) DLE_CHECK_ARG(a->N % 32 == 0);   // 32-element RNG groups
    if (a->epilogue == DLE_EPI_BIAS_GELU) DLE_CHECK_ARG(a->out2 != nullptr && a->ldo2 % 8 == 0);
    if (a->epilogue == DLE_EPI_DGELU || a->epilogue == DLE_EPI_ADD) DLE_CHECK_ARG(a->aux != nullptr);
    if (a->aux != nullptr) DLE_CHECK_ARG(a->ld_aux % 8 == 0 && (reinterpret_cast<uintptr_t>(a->aux) & 15) == 0);
    // the epilogue reads the bias slice with 4- / 8-byte loads and stores 16-byte vectors
    DLE_CHECK_ARG((reinterpret_cast<uintptr_t>(a->bias) & 7) == 0 && (reinterpret_cast<uintptr_t>(a->out) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(a->out2) & 15) == 0);
    const bool amn = a->a_layout == DLE_LAYOUT_MN, bmn = a->b_layout == DLE_LAYOUT_MN;
    // narrow-N problems (and the small-tile preference flag) take the 128-wide tile
    const bool bn128 = (a->N <= 128) || (a->tile_n == 128);
    if (bn128) {
        if (!amn && !bmn) return launch_gemm<128, false, false>(a, stream);
        if (!amn && bmn) return launch_gemm<128, false, true>(a, stream);
        if (amn && bmn) return launch_gemm<128, true, true>(a, stream);
        return launch_gemm<128, true, false>(a, stream);
    }
    if (!amn && !bmn) return launch_gemm<256, false, false>(a, stream);
    if (!amn && bmn) return launch_gemm<256, false, true>(a, stream);
    if (amn && bmn) return launch_gemm<256, true, true>(a, stream);
    return launch_gemm<256, true, false>(a, stream);
}
