// wide_tc.cu -- tensor-core GEMMs for WIDE coordinate MLPs (hidden width up to 256, e.g. BASELINE
// config 5: 63 -> 8 x 256 -> 4), where the fused small-MLP kernel (fused_tc.cu) does not apply:
// 9 x 256 x 256 bf16 weights (1.15 MB) and 128 x 256 activations per layer do not fit one CTA's
// shared memory, and the work per sample (2.86 MFLOP train) is firmly compute-bound.  So the wide
// path is LAYERWISE on the tensor cores, activations as bf16 in HBM:
//
//   forward   H_{l+1} = relu(H_l W_l + b_l)              (scripts/nerf.py:67-146)
//   backward  dZ_{l-1} = (dZ_l W_l^T) * [H_l > 0]         (reverse_diff.py rules, SURVEY.md App. B)
//   gradient  dW_l = H_l^T dZ_l, db_l = colsum(dZ_l)      (contraction over all samples)
//
// Kernels (all warp-specialised and persistent, one CTA per SM, TMA + mbarrier pipelines):
//   chain_tc_kernel  the forward pass and the adjoint pass, each ONE launch: a CTA takes blocks of its 128-sample
//                    tiles through all layers, the layer's weights in shared memory, the activations handed from
//                    layer to layer through L2; tcgen05.mma (M = 128, N <= 256, K = 16) into
//                    two TMEM accumulators, 16 epilogue warps (tcgen05.ld -> bias / ReLU + bit pattern / mask ->
//                    bf16 -> swizzled staging -> TMA store; or fp32 straight from registers on the last layer).
//                    A chain of one layer is a single GEMM (the unit-test hooks, LNB_WIDE_NO_CHAIN).
//   dw_tc_kernel     the weight gradient: the row-major bf16 activations read as MN-major operands (features
//                    contiguous), a 256 x N product accumulated in TMEM over the CTA's share of the samples, the
//                    column sums of dZ (the bias gradient) added up by the otherwise idle epilogue warps.
//   wide_reduce_all_kernel  one fixed-order reduction of every layer's per-CTA partials per step.
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdio.h>
#include <stdlib.h>

#include "lnb_internal.h"
#include "tc_ptx.cuh"

namespace {

constexpr int BM = 128;     // rows (samples) per tile
constexpr int BK = 64;      // K elements per pipeline stage = one 128-byte swizzle atom of bf16
constexpr int DW_THREADS = 192;   // weight-gradient kernel: warp 0 TMA, warp 1 MMA, warps 2..5 column sums + epilogue

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0;
    unsigned long long t0 = 0;
    for (uint32_t it = 0; !done; ++it) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity), "r"(100000u) : "memory");
        if (!done && (it & 0xFFFu) == 0xFFFu) {
            // a lost arrival must fail loudly, not hang the GPU: 20 s by the global timer (a kernel started early by
            // programmatic dependent launch legitimately spins here for as long as its predecessor runs)
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 20000000000ull) __trap();
        }
    }
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// L2 eviction-priority operands for TMA (the fixed encodings createpolicy.fractional produces for 1.0)
constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull, L2_EVICT_LAST = 0x14F0000000000000ull;
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap *map, uint32_t src, int c0, int c1, uint64_t policy)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;" ::"l"(map), "r"(src), "r"(c0), "r"(c1), "l"(policy) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, uint32_t src, int c0, int c1)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
// Programmatic dependent launch (pdl_wait / pdl_trigger): every kernel here triggers its own dependents only AFTER its
// wait, so data from two or more launches back (weights, biases) may be fetched before the wait.

// UMMA shared-memory descriptor for a 128-byte-swizzled tile whose rows are 128 B (64 bf16) apart and
// whose 8-row swizzle atoms are 1024 B apart (what a TMA box {64, rows} with SWIZZLE_128B writes).
//   K-major use  (rows = M or N, the 128 B direction = K): SBO = 1024 between 8-row groups.
//   MN-major use (rows = K, the 128 B direction = M or N): SBO = 1024 between 8-K groups, LBO = the
//   byte distance between 64-element MN atoms (= the next TMA box).
// layout_type SWIZZLE_128B = 2 (bits 61..63), version 1 (bit 46).
__device__ __forceinline__ uint64_t sw128_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}

enum { EPI_RELU_BF16 = 0,   // C = bf16(relu(acc + bias)), optionally + the ReLU pattern as bits
       EPI_MASK_BF16 = 1,   // C = bf16(bit ? acc : 0)                 (ReLU adjoint, pattern from the forward pass)
       EPI_HEAD_F32 = 2,    // C[row][0..3] = nerf/sigmoid head of (acc + bias), fp32 [M][ldc]   (last layer only)
       EPI_NONE_F32 = 3 };  // C = acc (+ bias) as fp32 [M][ldc]         (last layer only; the GEMM test hook)

constexpr int MAX_A_STAGES = 8;
constexpr int A_STAGE_BYTES = BM * BK * 2;   // 16 KB

// ---------------------------------------------------------------------------------------------
// Chain of layers in ONE persistent launch.  Tile t of layer l+1 needs only tile t of layer l (the
// same 128 samples, all columns), and the tile -> CTA map is the same for every layer, so the
// dependency is CTA-local: a CTA takes a block of G of its tiles through ALL layers of the chain
// before it moves to its next block.  What layer l wrote for those G tiles (G x 64 KB per CTA,
// G x 9.5 MB over the chip, stored evict-last) is still in L2 when layer l+1 reads it a few
// microseconds later, so HBM sees every activation tensor written once and never read back; the
// weights are reloaded from L2 once per layer per block (128 KB / G tiles), chunk by chunk as the
// previous layer's last MMAs release them.
// ---------------------------------------------------------------------------------------------
#ifdef LNB_WIDE_CLK
// debug build (LNB_WIDE_CLK=1 python -m loma_nerf_b200.build): where the chain kernel's MMA and epilogue warps wait
__device__ unsigned long long g_wide_clk[8];
#define WCLK_T0() const long long _t0 = clock64()
#define WCLK_ADD(i) atomicAdd(&g_wide_clk[i], (unsigned long long)(clock64() - _t0))
// timing experiments of the debug build only (results are invalid): LNB_WIDE_L2_HINTS bit 3 = no staging / stores,
// bit 4 = no epilogue body
#define WIDE_DEBUG_SKIP(bit) ((p.l2_hints & (bit)) != 0)
#else
#define WCLK_T0()
#define WCLK_ADD(i)
#define WIDE_DEBUG_SKIP(bit) false
#endif
constexpr int CHAIN_MAX_G = 8;
constexpr int CHAIN_THREADS = 576;   // warp 0 TMA, warp 1 MMA, warps 2..17 epilogue: the epilogue is the long pole of the chain
struct ChainLayer {
    const float *bias;         // [N] or NULL
    // ReLU pattern, one bit per element, [M][ldbits] words; word w covers columns 32w .. 32w+31 and column
    // 32w + 8g + 2j + p sits at bit 16p + 4g + j, so that the two flags of a packed bf16 pair are 16 bits
    // apart: ((word >> (4g + j)) & 0x00010001) * 0xFFFF is the pair's AND-mask
    const uint32_t *bits_in;   // EPI_MASK_BF16
    uint32_t *bits_out;        // EPI_RELU_BF16 (optional)
    float *out_f32;            // EPI_HEAD_F32, EPI_NONE_F32: [M][ldc]
    int ldbits, N, K, epi, ldc;
};
struct ChainParams {
    int M, n_layers, G, a_stages, head, l2_hints, b_region;
    ChainLayer layer[LNB_MAX_LAYERS];
};
struct ChainMaps { CUtensorMap A[LNB_MAX_LAYERS], B[LNB_MAX_LAYERS], C[LNB_MAX_LAYERS]; };

__device__ __forceinline__ void bulk_wait_group_n(int n)
{
    if (n >= 2) asm volatile("cp.async.bulk.wait_group 2;" ::: "memory");
    else if (n == 1) asm volatile("cp.async.bulk.wait_group 1;" ::: "memory");
    else asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

__global__ void __launch_bounds__(CHAIN_THREADS, 1)
chain_tc_kernel(const __grid_constant__ ChainMaps maps, const __grid_constant__ ChainParams p)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tiles = (p.M + BM - 1) / BM;
    // work units: tiles, dealt round-robin over the CTAs
    const int n_units = n_tiles, n_workers = (int)gridDim.x;
    const int unit0 = (int)blockIdx.x;
    const int n_my = unit0 < n_units ? (n_units - unit0 + n_workers - 1) / n_workers : 0;
    auto tile_of = [&](int i) { return unit0 + i * n_workers; };
    constexpr int B_CHUNK = 256 * BK * 2;     // bytes between weight chunks (uniform for all layers)
    const int AS = p.a_stages;
    uint8_t *sB = smem, *sA = smem + p.b_region;
    uint8_t *sC = sA + AS * A_STAGE_BYTES;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sC + 16 * 2048);   // 16 epilogue warps x one 32-row x 64-byte staging box
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + 8), tfull0 = smem_u32(bars + 16), tempty0 = smem_u32(bars + 18),
                   bfull0 = smem_u32(bars + 20), bempty0 = smem_u32(bars + 24), done0 = smem_u32(bars + 28);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 28 + CHAIN_MAX_G);
    float *sBias = reinterpret_cast<float *>(bars + 28 + CHAIN_MAX_G + 2);
    constexpr uint32_t acc_cols = 256;

    if (threadIdx.x == 0) {
        for (int s = 0; s < AS; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull0 + 8 * a, 1); mbar_init(tempty0 + 8 * a, 16); }   // one arrival per epilogue warp
        for (int k = 0; k < 4; ++k) { mbar_init(bfull0 + 8 * k, 1); mbar_init(bempty0 + 8 * k, 1); }
        for (int j = 0; j < CHAIN_MAX_G; ++j) mbar_init(done0 + 8 * j, 16);     // one arrival per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 2 * acc_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        // ---- TMA producer
        if (lane == 0) {
            pdl_wait();
            pdl_trigger();
            uint32_t stage = 0, phase = 0, round = 0;
            for (int blk = 0, bi = 0; blk < n_my; blk += p.G, ++bi) {
                const int g_cnt = n_my - blk < p.G ? n_my - blk : p.G;
                for (int li = 0; li < p.n_layers; ++li, ++round) {
                    // weight chunk kb always sits at kb * 32 KB whatever the layer's N, so "chunk kb released" means the same
                    // bytes for every layer
                    const int kb_count = p.layer[li].K / BK, b_rows = p.layer[li].N, b_bytes = b_rows * BK * 2;
                    for (int kb = 0; kb < 4; ++kb) {
                        // last round's MMAs on this chunk have retired.  Also for a chunk this layer does not use: its
                        // "full" barrier is advanced by a plain arrive below, and that must not overtake the MMA
                        // thread's wait for the previous phase (it can when a round has a single tile)
                        if (round > 0) mbar_wait(bempty0 + 8 * kb, (round - 1) & 1);
                        if (kb < kb_count) {
                            mbar_expect_tx(bfull0 + 8 * kb, (uint32_t)b_bytes);
                            tma_load_2d(smem_u32(sB + kb * B_CHUNK), &maps.B[li], kb * BK, 0, bfull0 + 8 * kb);
                        } else {
                            mbar_arrive(bfull0 + 8 * kb);                                   // keep the phases of unused chunks in step
                        }
                    }
                    for (int j = 0; j < g_cnt; ++j) {
                        const int tile = tile_of(blk + j);
                        if (li > 0) {   // this tile's output of the previous layer has fully left the SM (see the epilogue)
                            mbar_wait(done0 + 8 * j, (uint32_t)(bi * (p.n_layers - 1) + li - 1) & 1u);
                            asm volatile("fence.proxy.async.global;" ::: "memory");
                        }
                        for (int kb = 0; kb < kb_count; ++kb) {
                            mbar_wait(empty0 + 8 * stage, phase ^ 1);
                            mbar_expect_tx(full0 + 8 * stage, (uint32_t)A_STAGE_BYTES);
                            if (p.l2_hints & 1) tma_load_2d_hint(smem_u32(sA + stage * A_STAGE_BYTES), &maps.A[li], kb * BK, tile * BM, full0 + 8 * stage, L2_EVICT_FIRST);
                            else tma_load_2d(smem_u32(sA + stage * A_STAGE_BYTES), &maps.A[li], kb * BK, tile * BM, full0 + 8 * stage);
                            if (++stage == (uint32_t)AS) { stage = 0; phase ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer
        if (lane == 0) {
            uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0, round = 0;
            auto commit = [](uint32_t bar) { umma_commit(bar); };
#ifdef LNB_WIDE_CLK
            const long long t_begin = clock64();
#endif
            for (int blk = 0; blk < n_my; blk += p.G) {
                const int g_cnt = n_my - blk < p.G ? n_my - blk : p.G;
                for (int li = 0; li < p.n_layers; ++li, ++round) {
                    const int kb_count = p.layer[li].K / BK;
                    const uint32_t idesc = instr_desc(128, p.layer[li].N, 0, 0);
                    for (int j = 0; j < g_cnt; ++j) {
                        { WCLK_T0(); mbar_wait(tempty0 + 8 * acc, acc_phase ^ 1); WCLK_ADD(0); }
                        tc_fence_after();
                        for (int kb = 0; kb < kb_count; ++kb) {
                            if (j == 0) { WCLK_T0(); mbar_wait(bfull0 + 8 * kb, round & 1); WCLK_ADD(1); }
                            { WCLK_T0(); mbar_wait(full0 + 8 * stage, phase); WCLK_ADD(2); }
                            tc_fence_after();
                            const uint32_t a0 = smem_u32(sA + stage * A_STAGE_BYTES), b0 = smem_u32(sB + kb * B_CHUNK);
#pragma unroll
                            for (int k = 0; k < BK / 16; ++k) {
                                umma_bf16(tmem + acc * acc_cols, sw128_desc(a0 + k * 32, 16, 1024), sw128_desc(b0 + k * 32, 16, 1024), idesc,
                                               (kb > 0 || k > 0) ? 1u : 0u);
                            }
                            commit(empty0 + 8 * stage);
                            if (j == g_cnt - 1) commit(bempty0 + 8 * kb);          // this round is done with weight chunk kb
                            if (++stage == (uint32_t)AS) { stage = 0; phase ^= 1; }
                        }
                        if (j == g_cnt - 1)
                            for (int kb = kb_count; kb < 4; ++kb) commit(bempty0 + 8 * kb);
                        commit(tfull0 + 8 * acc);
                        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                    }
                }
            }
#ifdef LNB_WIDE_CLK
            atomicAdd(&g_wide_clk[3], (unsigned long long)(clock64() - t_begin));
#endif
        }
    } else {
        // ---- epilogue warps 2..17: four per TMEM lane quadrant (warp w may touch lanes 32*(w%4) .. +31), warp k of a
        // quadrant owns the 64-column chunk k of every tile and handles it as two 32-column halves: registers -> its
        // 32-row x 64-byte staging box (64-byte swizzle) -> TMA store
        const int q = warp & 3, k = (warp - 2) >> 2, et = threadIdx.x - 64;
        uint32_t acc = 0, acc_phase = 0;
        uint8_t *buf = sC + (warp - 2) * 2048;
        pdl_wait();
        for (int blk = 0; blk < n_my; blk += p.G) {
            const int g_cnt = n_my - blk < p.G ? n_my - blk : p.G;
            for (int li = 0; li < p.n_layers; ++li) {
                const ChainLayer &Ly = p.layer[li];
                const int N = Ly.N, epi = Ly.epi, c0 = k * 64;
                const bool signal = li < p.n_layers - 1;
                const int n_groups = ((epi == EPI_RELU_BF16 || epi == EPI_MASK_BF16) && c0 < N) ? 2 : 0;   // TMA stores this warp issues per tile
                asm volatile("bar.sync 1, 512;" ::: "memory");
                if (et < N) sBias[et] = Ly.bias ? __ldg(Ly.bias + et) : 0.0f;
                asm volatile("bar.sync 1, 512;" ::: "memory");
                for (int j = 0; j < g_cnt; ++j) {
                    const int tile = tile_of(blk + j);
                    const long long row = (long long)tile * BM + q * 32 + lane;
                    const bool live = row < p.M;
                    uint2 mw = make_uint2(0u, 0u);
                    if (epi == EPI_MASK_BF16 && live && c0 < N) mw = __ldg(reinterpret_cast<const uint2 *>(Ly.bits_in + row * Ly.ldbits + (c0 >> 5)));
                    { WCLK_T0(); mbar_wait(tfull0 + 8 * acc, acc_phase); if (threadIdx.x == 64) WCLK_ADD(4); }
                    tc_fence_after();
#ifdef LNB_WIDE_CLK
                    const long long t_epi = clock64();
#endif
                    const uint32_t tbase = tmem + acc * acc_cols + ((uint32_t)(q * 32) << 16);
                    if (epi == EPI_HEAD_F32 || epi == EPI_NONE_F32) {
                        // fp32 out of registers, 16 columns at a time: acc + bias, or the head's four outputs
                        for (int c = c0; c < N && c < c0 + 64; c += 16) {
                            uint32_t v[16];
                            tmem_ld16(tbase + c, v);
                            tmem_ld_wait();
                            if (!live) continue;
                            float4 *o = reinterpret_cast<float4 *>(Ly.out_f32 + row * Ly.ldc + c);
                            if (epi == EPI_HEAD_F32) {
                                float z[4];
#pragma unroll
                                for (int j = 0; j < 4; ++j) z[j] = __uint_as_float(v[j]) + sBias[j];
                                float4 h;
                                h.x = 1.0f / (1.0f + __expf(-z[0])); h.y = 1.0f / (1.0f + __expf(-z[1])); h.z = 1.0f / (1.0f + __expf(-z[2]));
                                h.w = p.head == LNB_HEAD_NERF ? fmaxf(z[3], 0.0f) : 1.0f / (1.0f + __expf(-z[3]));
                                o[0] = h;
                            } else {
#pragma unroll
                                for (int j = 0; j < 4; ++j)
                                    o[j] = make_float4(__uint_as_float(v[4 * j]) + sBias[c + 4 * j], __uint_as_float(v[4 * j + 1]) + sBias[c + 4 * j + 1],
                                                       __uint_as_float(v[4 * j + 2]) + sBias[c + 4 * j + 2], __uint_as_float(v[4 * j + 3]) + sBias[c + 4 * j + 3]);
                            }
                        }
                    } else if (c0 < N && !WIDE_DEBUG_SKIP(16)) {
                        uint32_t words[2] = {0u, 0u};
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            uint32_t v[32];
                            tmem_ld32(tbase + c0 + h * 32, v);
                            tmem_ld_wait();
                            if (WIDE_DEBUG_SKIP(8)) { if (v[0] == 0x7fc12345u) words[0] = v[1]; continue; }   // timing experiment: drain only
                            tma_store_wait_read0();          // this warp's previous store has left the box
                            __syncwarp();
                            const uint32_t wsel = h == 0 ? mw.x : mw.y;
                            uint32_t wout = 0;
#pragma unroll
                            for (int g = 0; g < 4; ++g) {   // four 16-byte pieces of this 64-byte row
                                uint4 *slot = reinterpret_cast<uint4 *>(buf + lane * 64 + ((g ^ ((lane >> 1) & 3)) << 4));
                                uint32_t pk[4];
                                if (epi == EPI_RELU_BF16) {
                                    uint32_t b8 = 0;
                                    const float4 bA = *reinterpret_cast<const float4 *>(sBias + c0 + h * 32 + g * 8), bB = *reinterpret_cast<const float4 *>(sBias + c0 + h * 32 + g * 8 + 4);
                                    const float bv[8] = {bA.x, bA.y, bA.z, bA.w, bB.x, bB.y, bB.z, bB.w};
#pragma unroll
                                    for (int c = 0; c < 4; ++c) {
                                        const float r0 = fmaxf(__uint_as_float(v[g * 8 + 2 * c]) + bv[2 * c], 0.0f);
                                        const float r1 = fmaxf(__uint_as_float(v[g * 8 + 2 * c + 1]) + bv[2 * c + 1], 0.0f);
                                        pk[c] = pack_bf16(r0, r1);
                                        b8 |= ((((pk[c] & 0x7FFF7FFFu) + 0x7FFF7FFFu) >> (15 - c)) & (0x00010001u << c));
                                    }
                                    wout |= b8 << (g * 4);
                                } else {
                                    const uint32_t b8 = wsel >> (g * 4);
#pragma unroll
                                    for (int c = 0; c < 4; ++c)
                                        pk[c] = pack_bf16(__uint_as_float(v[g * 8 + 2 * c]), __uint_as_float(v[g * 8 + 2 * c + 1])) &
                                                (((b8 >> c) & 0x00010001u) * 0xFFFFu);
                                }
                                *slot = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                            }
                            words[h] = wout;
                            fence_async_smem();
                            __syncwarp();
                            if (lane == 0) {
                                if (p.l2_hints & 2) tma_store_2d_hint(&maps.C[li], smem_u32(buf), c0 + h * 32, (int)(tile * BM + q * 32), L2_EVICT_LAST);
                                else tma_store_2d(&maps.C[li], smem_u32(buf), c0 + h * 32, (int)(tile * BM + q * 32));
                            }
                        }
                        if (epi == EPI_RELU_BF16 && Ly.bits_out && live)
                            *reinterpret_cast<uint2 *>(Ly.bits_out + row * Ly.ldbits + (c0 >> 5)) = make_uint2(words[0], words[1]);
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tempty0 + 8 * acc);
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
#ifdef LNB_WIDE_CLK
                    if (threadIdx.x == 64) atomicAdd(&g_wide_clk[5], (unsigned long long)(clock64() - t_epi));
#endif
                    // tell the producer when a tile's output is complete in memory: one tile late, so the wait
                    // is for stores issued a whole tile ago; the block's last tile is waited for outright
                    if (signal && lane == 0) {
                        WCLK_T0();
                        if (j > 0) { bulk_wait_group_n(n_groups); mbar_arrive(done0 + 8 * (j - 1)); }
                        if (j == g_cnt - 1) { bulk_wait_group_n(0); mbar_arrive(done0 + 8 * j); }
                        if (threadIdx.x == 64) WCLK_ADD(6);
                    }
                }
            }
        }
    }
    if (warp >= 2) tma_store_wait_all();
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 2 * acc_cols);
}

// ---- host helpers ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 2-D bf16 row-major [rows][cols] (cols contiguous, row pitch ld elements), box {64 cols, box_rows}, 128B swizzle
int make_map(lnb_ctx *ctx, CUtensorMap *m, const void *base, long long rows, int cols, int ld, int box_rows, int box_cols = 64)
{
    EncodeTiledFn enc = get_encode();
    if (!enc) { ctx->err = "cuTensorMapEncodeTiled is not available"; return LNB_ERR_CUDA; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};   // 64 columns: 128-byte swizzle; 32 columns: 64-byte swizzle
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { ctx->err = "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")"; return LNB_ERR_CUDA; }
    return LNB_OK;
}

// launch configuration with programmatic stream serialization (LNB_WIDE_NO_PDL=1 turns it off)
void pdl_config(cudaLaunchConfig_t *cfg, cudaLaunchAttribute *attr, int grid, int block, size_t smem, cudaStream_t stream)
{
    static const bool use_pdl = getenv("LNB_WIDE_NO_PDL") == nullptr;
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg->gridDim = dim3((unsigned)grid); cfg->blockDim = dim3((unsigned)block); cfg->dynamicSmemBytes = smem; cfg->stream = stream;
    cfg->attrs = attr; cfg->numAttrs = use_pdl ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------
// Weight gradient dW[in x out] = H^T dZ, contraction over samples.  H [rows][in_pad] and dZ
// [rows][out_pad] are the row-major bf16 activations / adjoints already in HBM; a TMA box
// {64 features, 64 samples} with the 128-byte swizzle lands as a tile whose rows are samples (the
// MMA's K) and whose 128-byte direction is the feature axis, i.e. exactly an MN-major operand.
// Each CTA owns a slab of samples and accumulates the whole [in_pad x out_pad] product in TMEM
// (two M = 128 halves x up to 256 columns = all 512 columns), then writes one fp32 partial.
// ---------------------------------------------------------------------------------------------
constexpr int DW_STAGES = 3;
struct DwParams {
    long long rows;
    int reverse;            // 64-sample blocks are dealt round-robin to the CTAs, from the first or from the last
    int l2_hints;           // bit 2: H loads evict-first
    int in_pad, out_pad;    // multiples of 64, <= 256
    float *partial;         // [grid][in_pad][out_pad]
    float *colsum;          // [grid][out_pad] column sums of dZ over the CTA's slab (bias gradient), or NULL
};

__global__ void __launch_bounds__(DW_THREADS, 1)
dw_tc_kernel(const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapZ, const DwParams p)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int a_boxes = p.in_pad / 64, b_boxes = p.out_pad / 64;
    const int a_bytes = a_boxes * 8192, b_bytes = b_boxes * 8192;       // per 64-sample stage
    uint8_t *sA = smem, *sB = smem + DW_STAGES * a_bytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sB + DW_STAGES * b_bytes);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + DW_STAGES), done0 = smem_u32(bars + 2 * DW_STAGES);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * DW_STAGES + 1);
    const int n_blocks = (int)((p.rows + 63) / 64);
    const int kb_count = (int)blockIdx.x < n_blocks ? (n_blocks - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int halves = (p.in_pad + 127) / 128;
    const uint32_t tcols = (uint32_t)(halves * p.out_pad) <= 32 ? 32 : ((halves * p.out_pad) <= 64 ? 64 : ((halves * p.out_pad) <= 128 ? 128 : ((halves * p.out_pad) <= 256 ? 256 : 512)));
    if (threadIdx.x == 0) {
        for (int s = 0; s < DW_STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 5); } // MMA commit + 4 column-sum warps
        mbar_init(done0, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(tmem_slot), tcols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    if (warp == 0 && lane == 0) {
        uint32_t stage = 0, phase = 0;
        pdl_wait();
        pdl_trigger();
        for (int kb = 0; kb < kb_count; ++kb) {
            mbar_wait(empty0 + 8 * stage, phase ^ 1);
            mbar_expect_tx(full0 + 8 * stage, (uint32_t)(a_bytes + b_bytes));
            const int blk = (int)blockIdx.x + kb * (int)gridDim.x;
            const int r0 = (p.reverse ? n_blocks - 1 - blk : blk) * 64;
            for (int b = 0; b < a_boxes; ++b)                      // rows past the end of the tensor are zero-filled by TMA
                if (p.l2_hints & 4) tma_load_2d_hint(smem_u32(sA + stage * a_bytes + b * 8192), &mapH, b * 64, r0, full0 + 8 * stage, L2_EVICT_FIRST);
                else tma_load_2d(smem_u32(sA + stage * a_bytes + b * 8192), &mapH, b * 64, r0, full0 + 8 * stage);
            for (int b = 0; b < b_boxes; ++b)
                tma_load_2d(smem_u32(sB + stage * b_bytes + b * 8192), &mapZ, b * 64, r0, full0 + 8 * stage);
            if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
        }
    } else if (warp == 1 && lane == 0) {
        const uint32_t idesc = instr_desc(128, p.out_pad, 1, 1);
        uint32_t stage = 0, phase = 0;
        for (int kb = 0; kb < kb_count; ++kb) {
            mbar_wait(full0 + 8 * stage, phase);
            tc_fence_after();
            const uint32_t a0 = smem_u32(sA + stage * a_bytes), b0 = smem_u32(sB + stage * b_bytes);
            for (int h = 0; h < halves; ++h) {
#pragma unroll
                for (int k = 0; k < 4; ++k)   // 16 samples per MMA: +2048 B (16 rows x 128 B) inside every box
                    umma_bf16(tmem + h * p.out_pad, sw128_desc(a0 + h * 2 * 8192 + k * 2048, 8192, 1024),
                              sw128_desc(b0 + k * 2048, 8192, 1024), idesc, (kb > 0 || k > 0) ? 1u : 0u);
            }
            umma_commit(empty0 + 8 * stage);
            if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(done0);
    } else if (warp >= 2) {
        // While the MMAs run, the four epilogue warps add up the columns of the dZ tiles as they pass
        // through shared memory (d_bs = colsum(dZ)): thread t owns features 2t, 2t+1, i.e. one 32-bit
        // word of every 128-byte row of box t/32; a warp reads a whole swizzled row, conflict-free.
        {
            const int t = (warp - 2) * 32 + lane, box = t >> 5, pr = t & 31;
            const bool have = box < b_boxes;
            float s0 = 0.0f, s1 = 0.0f;
            uint32_t stage = 0, phase = 0;
            for (int kb = 0; kb < kb_count; ++kb) {
                mbar_wait(full0 + 8 * stage, phase);
                if (have && p.colsum) {
                    const uint8_t *base = sB + stage * b_bytes + box * 8192 + (pr & 3) * 4;
#pragma unroll 8
                    for (int r = 0; r < 64; ++r) {
                        const uint32_t w = *reinterpret_cast<const uint32_t *>(base + r * 128 + (((pr >> 2) ^ (r & 7)) << 4));
                        s0 += __uint_as_float(w << 16);
                        s1 += __uint_as_float(w & 0xFFFF0000u);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(empty0 + 8 * stage);
                if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
            }
            if (have && p.colsum) {
                p.colsum[(size_t)blockIdx.x * p.out_pad + 2 * t] = s0;
                p.colsum[(size_t)blockIdx.x * p.out_pad + 2 * t + 1] = s1;
            }
        }
        mbar_wait(done0, 0);
        tc_fence_after();
        pdl_wait();
        const int q = warp & 3;
        float *out = p.partial + (size_t)blockIdx.x * p.in_pad * p.out_pad;
        for (int h = 0; h < halves; ++h) {
            const int feat = h * 128 + q * 32 + lane;
            for (int c0 = 0; c0 < p.out_pad; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + h * p.out_pad + c0, v);
                tmem_ld_wait();
                if (feat < p.in_pad) {
                    float4 *o = reinterpret_cast<float4 *>(out + (size_t)feat * p.out_pad + c0);
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        o[j] = kb_count ? make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]))
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, tcols);
}

// dst[k*ldw + j] += scale * sum_z partial[z][k][j] for k < in_dim, j < out_dim, for every job in ONE launch (a step
// keeps all its partials: a weight job and a bias job per layer): job j covers blocks [first_block[j], first_block[j+1]).
// A block covers 128 consecutive padded elements (32 lanes x float4) with 8 groups of partials in parallel; each group
// adds its partials in index order and the groups are combined in order, so the result is fixed.
struct ReduceJob {
    const float *partial; float *dst;
    int in_pad, out_pad, in_dim, out_dim, ldw, first_block;
};
struct ReduceJobs { ReduceJob job[2 * LNB_MAX_LAYERS]; int n_jobs, n_part; float seed_value; const float *seed_dev; };

// appends the job of partials [n_part][in_pad][out_pad]; blocks counts the launch's grid
void add_reduce_job(ReduceJobs &jobs, int &blocks, const float *partial, float *dst, int in_pad, int out_pad, int in_dim, int out_dim, int ldw)
{
    jobs.job[jobs.n_jobs++] = ReduceJob{partial, dst, in_pad, out_pad, in_dim, out_dim, ldw, blocks};
    blocks += (in_pad * out_pad + 127) / 128;
}

__global__ void __launch_bounds__(256) wide_reduce_all_kernel(const __grid_constant__ ReduceJobs jobs)
{
    __shared__ float4 acc[8][32];
    int j = 0;
    while (j + 1 < jobs.n_jobs && (int)blockIdx.x >= jobs.job[j + 1].first_block) ++j;
    const ReduceJob &J = jobs.job[j];
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int e = (((int)blockIdx.x - J.first_block) * 32 + lane) * 4;
    const int n_el = J.in_pad * J.out_pad;
    const size_t stride = (size_t)n_el;
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0;
    if (e < n_el) {
        int z = grp;
        for (; z + 8 < jobs.n_part; z += 16) {
            const float4 a = *reinterpret_cast<const float4 *>(J.partial + (size_t)z * stride + e);
            const float4 b = *reinterpret_cast<const float4 *>(J.partial + (size_t)(z + 8) * stride + e);
            s0.x += a.x; s0.y += a.y; s0.z += a.z; s0.w += a.w;
            s1.x += b.x; s1.y += b.y; s1.z += b.z; s1.w += b.w;
        }
        if (z < jobs.n_part) {
            const float4 a = *reinterpret_cast<const float4 *>(J.partial + (size_t)z * stride + e);
            s0.x += a.x; s0.y += a.y; s0.z += a.z; s0.w += a.w;
        }
    }
    acc[grp][lane] = make_float4(s0.x + s1.x, s0.y + s1.y, s0.z + s1.z, s0.w + s1.w);
    __syncthreads();
    if (grp == 0 && e < n_el) {
        float4 s = acc[0][lane];
        for (int g = 1; g < 8; ++g) { s.x += acc[g][lane].x; s.y += acc[g][lane].y; s.z += acc[g][lane].z; s.w += acc[g][lane].w; }
        const float scale = jobs.seed_value * (jobs.seed_dev ? __ldg(jobs.seed_dev) : 1.0f);
        const int k = e / J.out_pad, c = e % J.out_pad;
        if (k < J.in_dim) {
            const float v[4] = {s.x, s.y, s.z, s.w};
            for (int i = 0; i < 4; ++i)
                if (c + i < J.out_dim) J.dst[(size_t)k * J.ldw + c + i] += scale * v[i];
        }
    }
}

// dst[i][j] = bf16(j < cols ? src[i][j] : 0) for j < ldd (ldd multiple of 8): a thread makes one 16-byte store
__global__ void f32_to_bf16_rows_kernel(const float *__restrict__ src, int lds, int cols, long long rows, __nv_bfloat16 *__restrict__ dst, int ldd)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int per_row = ldd >> 3;
    if (e >= rows * per_row) return;
    const long long i = e / per_row;
    const int c8 = (int)(e % per_row) * 8;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = c8 + j < cols ? __ldg(src + i * lds + c8 + j) : 0.0f;
    *reinterpret_cast<uint4 *>(dst + i * ldd + c8) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}

// weight images: Wf[l] = [out_pad][in_pad] (forward B operand, K = in), Wb[l] = [in_pad][out_pad] (backward, K = out);
// every layer's weight images and padded bias in ONE launch: blockIdx.y = layer
struct PrepJob { const float *w, *b; __nv_bfloat16 *Wf, *Wb; float *biasP; int in_dim, out_dim, in_pad, out_pad; };
struct PrepJobs { PrepJob job[LNB_MAX_LAYERS]; int ldw; };
__global__ void wide_prep_all_kernel(const __grid_constant__ PrepJobs jobs)
{
    const PrepJob &J = jobs.job[blockIdx.y];
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < J.out_pad) J.biasP[e] = e < J.out_dim ? J.b[e] : 0.0f;
    if (e >= J.in_pad * J.out_pad) return;
    const int k = e / J.out_pad, j = e % J.out_pad;
    const float v = (k < J.in_dim && j < J.out_dim) ? J.w[(size_t)k * jobs.ldw + j] : 0.0f;
    J.Wb[(size_t)k * J.out_pad + j] = __float2bfloat16_rn(v);
    J.Wf[(size_t)j * J.in_pad + k] = __float2bfloat16_rn(v);
}

size_t dw_smem(int in_pad, int out_pad)
{
    return (size_t)DW_STAGES * ((in_pad / 64) + (out_pad / 64)) * 8192 + (2 * DW_STAGES + 4) * 8 + 16;
}

} // namespace

// One launch for a chain of layers (chain_tc_kernel): layer i computes epilogue_i(A_i B_i^T) where A_{i+1}
// is the bf16 tensor layer i wrote.  All layers share M; K multiples of 64 (<= 256), row pitches multiples
// of 8 elements; bf16 layers are multiples of 64 wide, and the last layer may instead write fp32 (the head,
// or acc + bias) with N a multiple of 16.
struct ChainDesc {
    const void *A; int lda;
    const void *B; int ldb;
    int N, K;
    const float *bias;
    const uint32_t *bits_in; uint32_t *bits_out; int ldbits;
    void *C; int ldc;
    int epi;
};

int lnb_wide_chain(lnb_ctx *ctx, const ChainDesc *d, int n, long long M, int head)
{
    LNB_ARG(n >= 1 && n <= LNB_MAX_LAYERS && M >= 0, "wide chain: layers");
    if (M == 0) return LNB_OK;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    ChainMaps maps;              // 6 KB, passed by value at launch
    ChainParams p{};
    size_t b_region = 0;
    for (int i = 0; i < n; ++i) {
        const ChainDesc &c = d[i];
        LNB_ARG(c.N >= 16 && c.N <= 256 && c.N % 16 == 0 && c.K >= 64 && c.K <= 256 && c.K % 64 == 0 && c.lda % 8 == 0 && c.ldb % 8 == 0, "wide chain: shape");
        LNB_TRY(make_map(ctx, &maps.A[i], c.A, M, c.K, c.lda, BM));
        LNB_TRY(make_map(ctx, &maps.B[i], c.B, c.N, c.K, c.ldb, c.N));
        maps.C[i] = maps.A[i];
        if (c.epi == EPI_RELU_BF16 || c.epi == EPI_MASK_BF16) {
            LNB_ARG(c.N % 64 == 0 && c.ldc % 8 == 0 && c.ldc >= c.N, "wide chain: bf16 layers are multiples of 64 wide");
            LNB_ARG((c.epi != EPI_MASK_BF16 || c.bits_in) && (!(c.bits_in || c.bits_out) || (c.ldbits * 32 >= c.N && c.ldbits <= 8)), "wide chain: ReLU bits");
            LNB_TRY(make_map(ctx, &maps.C[i], c.C, M, c.N, c.ldc, 32, 32));
        } else {
            LNB_ARG((c.epi == EPI_HEAD_F32 || c.epi == EPI_NONE_F32) && i == n - 1, "wide chain: only the last layer may write fp32");
            LNB_ARG(c.ldc % 4 == 0 && c.ldc >= (c.epi == EPI_HEAD_F32 ? 4 : c.N), "wide chain: fp32 output pitch");
        }
        ChainLayer &l = p.layer[i];
        l.bias = c.bias; l.bits_in = c.bits_in; l.bits_out = c.bits_out;
        l.out_f32 = (c.epi == EPI_HEAD_F32 || c.epi == EPI_NONE_F32) ? (float *)c.C : nullptr;
        l.ldbits = c.ldbits; l.N = c.N; l.K = c.K; l.epi = c.epi; l.ldc = c.ldc;
        const size_t chunk = 256 * BK * 2, rows = c.N;   // chunks 32 KB apart
        const size_t need = (size_t)(c.K / BK - 1) * chunk + ((rows * BK * 2 + 1023) / 1024 * 1024);
        b_region = need > b_region ? need : b_region;
    }
    static const int G = [] { const char *e = getenv("LNB_WIDE_CHAIN_G"); const int g = e ? atoi(e) : 6; return g < 1 ? 1 : (g > CHAIN_MAX_G ? CHAIN_MAX_G : g); }();
    // chain: what a layer reads is dead in L2 once read (evict-first); measured 3.04 ms per C5 step against 3.08 with
    // evict-last stores only
    static const int l2_hints = [] { const char *e = getenv("LNB_WIDE_L2_HINTS"); return e ? atoi(e) : 1; }();
    p.M = (int)M; p.n_layers = n; p.G = G; p.head = head; p.l2_hints = l2_hints; p.b_region = (int)b_region;
    long long st = (232448LL - 2048 - 16 * 2048 - (long long)b_region) / A_STAGE_BYTES;
    p.a_stages = (int)(st > MAX_A_STAGES ? MAX_A_STAGES : st);
    LNB_ARG(p.a_stages >= 2, "wide chain: shared memory");
    const size_t smem = b_region + (size_t)p.a_stages * A_STAGE_BYTES + 16 * 2048 + (28 + CHAIN_MAX_G + 2) * 8 + 1024 + 16;
    const int n_tiles = (int)((M + BM - 1) / BM);
    const int grid = n_tiles < ctx->sm_count ? n_tiles : ctx->sm_count;
    cudaLaunchConfig_t cfg{};
    cudaLaunchAttribute attr[2];
    pdl_config(&cfg, attr, grid, CHAIN_THREADS, smem, ctx->stream);
    LNB_CUDA(cudaFuncSetAttribute(chain_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lnb_prof_begin(ctx, "chain_tc_kernel");
    LNB_CUDA(cudaLaunchKernelEx(&cfg, chain_tc_kernel, maps, p));
    lnb_prof_end(ctx);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

// test hook (tests/test_gpu_wide.py), a one-layer chain: fp32 C = A * B^T (+ bias) from bf16 operands
extern "C" LNB_API int lnb_test_wide_gemm(lnb_ctx *ctx, const void *A, const void *B, long long M, int N, int K, const float *bias,
                                          float *C)
{
    if (!ctx) return LNB_ERR_ARG;
    const ChainDesc d{A, K, B, K, N, K, bias, nullptr, nullptr, 0, C, N, EPI_NONE_F32};
    return lnb_wide_chain(ctx, &d, 1, M, 0);
}

// test hook, a one-layer chain: bf16 C = relu(A B^T + bias) (+ its ReLU bit pattern into bits_out), or, when
// bits_in != NULL, C = A B^T where the bit is set and 0 elsewhere.  N a multiple of 64; bit rows are N/32 words.
extern "C" LNB_API int lnb_test_wide_gemm_bf16(lnb_ctx *ctx, const void *A, const void *B, long long M, int N, int K, const float *bias,
                                               const void *bits_in, void *bits_out, void *C)
{
    if (!ctx) return LNB_ERR_ARG;
    const ChainDesc d{A, K, B, K, N, K, bias, (const uint32_t *)bits_in, (uint32_t *)bits_out, N / 32, C, N,
                      bits_in ? EPI_MASK_BF16 : EPI_RELU_BF16};
    return lnb_wide_chain(ctx, &d, 1, M, 0);
}

// dW partials of one layer ([n_part][in_pad][out_pad] fp32) and, if colsum != NULL, the column sums of
// dZ per CTA ([n_part][out_pad])
int lnb_wide_dw(lnb_ctx *ctx, const void *H, int ldh, int in_pad, const void *dZ, int ldz, int out_pad, long long rows,
                float *partial, float *colsum, int n_part, int reverse)
{
    LNB_ARG(in_pad % 64 == 0 && in_pad >= 64 && in_pad <= 256 && out_pad % 64 == 0 && out_pad >= 64 && out_pad <= 256, "wide dW: padded widths");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    CUtensorMap mapH, mapZ;
    LNB_TRY(make_map(ctx, &mapH, H, rows, in_pad, ldh, 64));
    LNB_TRY(make_map(ctx, &mapZ, dZ, rows, out_pad, ldz, 64));
    DwParams p{};
    p.rows = rows;
    p.reverse = reverse;
    static const int l2_hints = [] { const char *e = getenv("LNB_WIDE_L2_HINTS"); return e ? atoi(e) : 2; }();
    p.l2_hints = l2_hints;
    p.in_pad = in_pad; p.out_pad = out_pad; p.partial = partial; p.colsum = colsum;
    const size_t smem = dw_smem(in_pad, out_pad);
    LNB_CUDA(cudaFuncSetAttribute(dw_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg{};
    cudaLaunchAttribute attr[1];
    pdl_config(&cfg, attr, n_part, DW_THREADS, smem, ctx->stream);
    LNB_CUDA(cudaLaunchKernelEx(&cfg, dw_tc_kernel, mapH, mapZ, p));
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

// test hook: fp32 dW[in_pad][out_pad] = H^T dZ and db[out_pad] = colsum(dZ) from bf16 H [rows][in_pad], dZ [rows][out_pad]
extern "C" LNB_API int lnb_test_wide_dw(lnb_ctx *ctx, const void *H, int in_pad, const void *dZ, int out_pad, long long rows, float *dW,
                                        float *db)
{
    if (!ctx) return LNB_ERR_ARG;
    const int n_part = ctx->sm_count;
    LNB_TRY(lnb_arena_reserve(ctx, (size_t)n_part * (in_pad + 1) * out_pad * sizeof(float) + 8192));
    float *partial = (float *)lnb_arena_take(ctx, (size_t)n_part * in_pad * out_pad * sizeof(float));
    float *bpartial = (float *)lnb_arena_take(ctx, (size_t)n_part * out_pad * sizeof(float));
    LNB_TRY(lnb_wide_dw(ctx, H, in_pad, in_pad, dZ, out_pad, out_pad, rows, partial, db ? bpartial : nullptr, n_part, (int)(rows & 1)));
    ReduceJobs jobs{};
    int blocks = 0;
    add_reduce_job(jobs, blocks, partial, dW, in_pad, out_pad, in_pad, out_pad, out_pad);
    if (db) add_reduce_job(jobs, blocks, bpartial, db, 1, out_pad, 1, out_pad, out_pad);
    jobs.n_part = n_part;
    jobs.seed_value = 1.0f;
    // the reduction adds into dW / db
    LNB_CUDA(cudaMemsetAsync(dW, 0, (size_t)in_pad * out_pad * sizeof(float), ctx->stream));
    if (db) LNB_CUDA(cudaMemsetAsync(db, 0, (size_t)out_pad * sizeof(float), ctx->stream));
    wide_reduce_all_kernel<<<blocks, 256, 0, ctx->stream>>>(jobs);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

// ---------------------------------------------------------------------------------------------
// The wide-MLP step: layerwise on the tensor cores (see the header of this file).  Produces what
// the fused kernel produces: loss, colour, d_ws, d_bs.  Returns LNB_ERR_UNSUPPORTED otherwise.
// ---------------------------------------------------------------------------------------------
static int pad64(int v) { return (v + 63) / 64 * 64; }

int lnb_wide_tc_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, const lnb_comp_args *cx)
{
    auto unsupported = [&](const char *why) {
        ctx->err = std::string("wide tensor-core path: ") + why;
        return LNB_ERR_UNSUPPORTED;
    };
    const int L = mlp->n_layers;
    if (!nerf && (a->S != 1 || a->target_w < 1 || a->target_w > 4 || a->target_w > mlp->dims[L] || (!a->X)))
        return unsupported("mlp_fit needs features, one sample per row and at most 4 output channels");
    if (L < 2 || L > LNB_MAX_LAYERS) return unsupported("needs 2..16 layers");
    for (int l = 0; l <= L; ++l)
        if (mlp->dims[l] > 256) return unsupported("layer widths above 256");
    if (mlp->dims[L] > 16) return unsupported("more than 16 output channels");
    if (a->inter || a->d_X || a->d_inter)
        return unsupported("per-layer intermediates and d_layer_input are not produced here (use the fp32 path)");
    if (!nerf && (a->d_target || a->d_color)) return unsupported("mlp_fit adjoints other than d_ws / d_bs are not produced here (use the fp32 path)");
    if (a->color && a->color_accumulate) return unsupported("colour accumulation");
    const int R = a->R, S = a->S;
    const long long N = a->n_rows > 0 ? a->n_rows : (long long)R * S;
    if (N != (long long)R * S || a->rows > N) return unsupported("needs n_rows == R*S and no extra rows");
    if (N > 0x7fffffffLL - 256) return unsupported("too many samples for one call");
    if (a->want_grad && !a->target) return unsupported("gradient without target");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    const bool cam = !a->X && !a->rays_o && a->cam;
    const bool rays = !a->X && (a->rays_o || cam);
    const bool grad = a->want_grad != 0;
    const int c_in = mlp->dims[0];
    int in_pad[LNB_MAX_LAYERS], out_pad[LNB_MAX_LAYERS];
    for (int l = 0; l < L; ++l) { in_pad[l] = pad64(mlp->dims[l]); out_pad[l] = pad64(mlp->dims[l + 1]); }
    const int n_part = ctx->sm_count;

    // ---- arena plan
    size_t need = 1 << 16;
    auto add = [&](size_t bytes) { need += (bytes + 255) / 256 * 256 + 256; };
    int max_pad = 64;
    for (int l = 0; l < L; ++l) max_pad = in_pad[l] > max_pad ? in_pad[l] : max_pad;
    for (int l = 0; l < L; ++l) {
        if (grad || l == 0) add((size_t)N * in_pad[l] * 2);      // H_l (bf16): all kept for the backward pass,
        if (grad) { add((size_t)N * out_pad[l] * 2); add((size_t)N * (in_pad[l] / 32) * 4); }   // dZ_l, ReLU bits of H_l
    }
    if (!grad) { add((size_t)N * max_pad * 2); add((size_t)N * max_pad * 2); }   // render: two buffers in turn
    if (grad) add((size_t)N * 16);                               // head adjoint fp32 [N][4]
    add((size_t)N * 16);                                         // head fp32 [N][4]
    if (rays) add((size_t)R * S * 4);
    for (int l = 0; l < L; ++l) { add((size_t)in_pad[l] * out_pad[l] * 2); add((size_t)in_pad[l] * out_pad[l] * 2); add((size_t)out_pad[l] * 4); }
    if (grad)
        for (int l = 0; l < L; ++l) { add((size_t)n_part * in_pad[l] * out_pad[l] * 4); add((size_t)n_part * out_pad[l] * 4); }
    add((size_t)R * 4 + 16); add((size_t)R * 12 + 16); add(64);
    if (grad && a->d_dists) add((size_t)N * 4);
    if (grad && (a->d_color || a->d_target)) add((size_t)R * 12 + 16);
    LNB_TRY(lnb_arena_reserve(ctx, need));
    auto take = [&](size_t bytes) { return lnb_arena_take(ctx, bytes); };
    __nv_bfloat16 *H[LNB_MAX_LAYERS], *dZ[LNB_MAX_LAYERS];
    uint32_t *bits[LNB_MAX_LAYERS];
    __nv_bfloat16 *pp[2] = {nullptr, nullptr};
    if (!grad) { pp[0] = (__nv_bfloat16 *)take((size_t)N * max_pad * 2); pp[1] = (__nv_bfloat16 *)take((size_t)N * max_pad * 2); }
    for (int l = 0; l < L; ++l) {
        H[l] = (grad || l == 0) ? (__nv_bfloat16 *)take((size_t)N * in_pad[l] * 2) : pp[(l - 1) & 1];
        dZ[l] = grad ? (__nv_bfloat16 *)take((size_t)N * out_pad[l] * 2) : nullptr;
        bits[l] = grad ? (uint32_t *)take((size_t)N * (in_pad[l] / 32) * 4) : nullptr;
    }
    float *dzh = grad ? (float *)take((size_t)N * 16) : nullptr;
    float *head = (float *)take((size_t)N * 16);
    const float *X = a->X, *dists = a->dists;
    if (rays) {   // sample positions (and view directions) and their encoding straight into the bf16 operand of layer 0
        float *de = (float *)take((size_t)R * S * 4);
        const int Ed = lnb_rays_dir_bands(c_in, a->pe_bands);
        if (N > 0 && cam)
            LNB_TRY(lnb_launch_camera_encode(ctx, a->cam, lnb_cx_views(cx), R, S, a->pe_bands, Ed, nullptr, de, H[0], in_pad[0]));
        else if (N > 0)
            LNB_TRY(lnb_launch_sample_encode_bf16(ctx, a->rays_o, a->rays_d, a->t, a->ray_dtype == LNB_RAY_F64, R, S, a->pe_bands, Ed, nullptr, de, H[0],
                                                  in_pad[0]));
        dists = de;
    }
    __nv_bfloat16 *Wf[LNB_MAX_LAYERS], *Wb[LNB_MAX_LAYERS];
    float *biasP[LNB_MAX_LAYERS];
    for (int l = 0; l < L; ++l) {
        Wf[l] = (__nv_bfloat16 *)take((size_t)in_pad[l] * out_pad[l] * 2);
        Wb[l] = (__nv_bfloat16 *)take((size_t)in_pad[l] * out_pad[l] * 2);
        biasP[l] = (float *)take((size_t)out_pad[l] * 4);
    }
    float *partial[LNB_MAX_LAYERS], *bpartial[LNB_MAX_LAYERS];
    for (int l = 0; l < L; ++l) {
        partial[l] = grad ? (float *)take((size_t)n_part * in_pad[l] * out_pad[l] * 4) : nullptr;
        bpartial[l] = grad ? (float *)take((size_t)n_part * out_pad[l] * 4) : nullptr;
    }
    float *ray_sse = (float *)take((size_t)R * 4 + 16);
    float *color = a->color ? a->color : (float *)take((size_t)R * 12 + 16);
    float *loss = a->loss ? a->loss : (float *)take(64);
    // compositing by-products and the adjoints of dists / colour / target come from the fp32 compositing kernels this path
    // shares with the exact one (their inputs, the head outputs, carry the bf16 error of the MLP)
    float *d_dists_u = (grad && a->d_dists) ? (float *)take((size_t)N * 4) : nullptr;
    float *d_color_u = (grad && (a->d_color || a->d_target)) ? (float *)take((size_t)R * 12 + 16) : nullptr;
    if (N == 0) {
        if (a->loss) LNB_TRY(lnb_launch_fill(ctx, loss, 1, 0.0f));
        return LNB_OK;
    }

    // ---- weight images, padded biases
    {
        PrepJobs pj{};
        int n_max = 0;
        for (int l = 0; l < L; ++l) {
            pj.job[l] = PrepJob{a->ws + (size_t)l * mlp->max_in * mlp->max_out, a->bs + (size_t)l * mlp->max_out, Wf[l], Wb[l], biasP[l], mlp->dims[l],
                                mlp->dims[l + 1], in_pad[l], out_pad[l]};
            n_max = in_pad[l] * out_pad[l] > n_max ? in_pad[l] * out_pad[l] : n_max;
        }
        pj.ldw = mlp->max_out;
        wide_prep_all_kernel<<<dim3((n_max + 255) / 256, L), 256, 0, ctx->stream>>>(pj);
        LNB_CHECK_LAUNCH();
    }

    // ---- forward and adjoint chain (unit seed; the seed scales d_ws / d_bs at the end): one chain_tc_kernel launch per
    // pass, or with LNB_WIDE_NO_CHAIN=1 one per layer, where no activations are handed over inside the kernel
    static const bool per_layer = getenv("LNB_WIDE_NO_CHAIN") != nullptr;
    auto run_chain = [&](const ChainDesc *cd, int n, int head_kind) {
        if (!per_layer) return lnb_wide_chain(ctx, cd, n, N, head_kind);
        for (int i = 0; i < n; ++i) LNB_TRY(lnb_wide_chain(ctx, cd + i, 1, N, head_kind));
        return (int)LNB_OK;
    };
    if (!rays) {
        const long long n = N * (in_pad[0] / 8);
        f32_to_bf16_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(X, c_in, c_in, N, H[0], in_pad[0]);
        LNB_CHECK_LAUNCH();
    }
    {
        ChainDesc cd[LNB_MAX_LAYERS];
        for (int l = 0; l < L - 1; ++l)
            cd[l] = ChainDesc{H[l], in_pad[l], Wf[l], in_pad[l], out_pad[l], in_pad[l], biasP[l], nullptr, grad ? bits[l + 1] : nullptr, in_pad[l + 1] / 32,
                              H[l + 1], out_pad[l], EPI_RELU_BF16};
        cd[L - 1] = ChainDesc{H[L - 1], in_pad[L - 1], Wf[L - 1], in_pad[L - 1], 16, in_pad[L - 1], biasP[L - 1], nullptr, nullptr, 0, head, 4, EPI_HEAD_F32};
        LNB_TRY(run_chain(cd, L, mlp->head));
    }
    if (nerf)
        LNB_TRY(lnb_launch_composite_fwd(ctx, head, 4, dists, a->target, R, S, a->rgba, a->alpha, a->cumprod, a->weights, color, 0, ray_sse, cx));
    else if (a->target)   // mlp_fit: the prediction is the sigmoid head itself, SSE over target_w channels (mlp_fit.py:140-145)
        LNB_TRY(lnb_launch_fit_loss(ctx, head, 4, a->target, R, a->target_w, ray_sse));
    if (grad) {
        if (nerf)
            LNB_TRY(lnb_launch_composite_bwd(ctx, head, 4, dists, a->target, color, R, S, dzh, 4, 4, d_dists_u, d_color_u, cx));
        else
            LNB_TRY(lnb_launch_fit_head_bwd(ctx, head, 4, a->target, R, a->target_w, R, 4, dzh, 4, nullptr));
        const long long n = N * (out_pad[L - 1] / 8);
        f32_to_bf16_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(dzh, 4, 4, N, dZ[L - 1], out_pad[L - 1]);
        LNB_CHECK_LAUNCH();
        // the adjoint chain dZ_{L-1} -> ... -> dZ_0, then the weight gradients, first the layers whose adjoints were
        // written last
        ChainDesc cd[LNB_MAX_LAYERS];
        int nc = 0;
        for (int l = L - 1; l >= 1; --l)
            cd[nc++] = ChainDesc{dZ[l], out_pad[l], Wb[l], out_pad[l], in_pad[l], out_pad[l], nullptr, bits[l], nullptr, in_pad[l] / 32, dZ[l - 1], in_pad[l],
                                 EPI_MASK_BF16};
        LNB_TRY(run_chain(cd, nc, 0));
        // serpentine order: each dW launch walks the samples in the direction opposite to the launch before it, so it
        // starts on the part of its input that the previous kernel touched last and that is still in the 126 MB L2
        // (LNB_WIDE_NO_SERPENTINE=1 turns it off)
        static const bool serpentine = getenv("LNB_WIDE_NO_SERPENTINE") == nullptr;
        for (int l = 0; l < L; ++l)
            LNB_TRY(lnb_wide_dw(ctx, H[l], in_pad[l], in_pad[l], dZ[l], out_pad[l], out_pad[l], N, partial[l], bpartial[l], n_part,
                                serpentine && l % 2 == 0));
    }
    if (a->target) LNB_TRY(lnb_launch_sum(ctx, ray_sse, R, loss));
    else if (a->loss) LNB_TRY(lnb_launch_fill(ctx, loss, 1, 0.0f));
    if (!grad) return LNB_OK;

    // ---- weight and bias gradients: one launch reduces every layer's partials into d_ws / d_bs
    ReduceJobs jobs{};
    int blocks = 0;
    for (int l = L - 1; l >= 0; --l) {
        add_reduce_job(jobs, blocks, partial[l], a->d_ws + (size_t)l * mlp->max_in * mlp->max_out, in_pad[l], out_pad[l], mlp->dims[l],
                       mlp->dims[l + 1], mlp->max_out);
        add_reduce_job(jobs, blocks, bpartial[l], a->d_bs + (size_t)l * mlp->max_out, 1, out_pad[l], 1, mlp->dims[l + 1], mlp->max_out);
    }
    jobs.n_part = n_part;
    jobs.seed_value = a->seed_mode == LNB_SEED_LOSS ? 1.0f : a->seed;
    jobs.seed_dev = a->seed_mode == LNB_SEED_LOSS ? loss : nullptr;
    wide_reduce_all_kernel<<<blocks, 256, 0, ctx->stream>>>(jobs);
    LNB_CHECK_LAUNCH();
    // += seed x unit-seed adjoint (the seed may be the loss just computed on the device)
    if (a->d_dists) LNB_TRY(lnb_launch_axpy2d(ctx, a->d_dists, S, d_dists_u, S, R, S, 1.0f, jobs.seed_value, jobs.seed_dev));
    if (a->d_color) LNB_TRY(lnb_launch_axpy2d(ctx, a->d_color, 3, d_color_u, 3, R, 3, 1.0f, jobs.seed_value, jobs.seed_dev));
    if (a->d_target) LNB_TRY(lnb_launch_axpy2d(ctx, a->d_target, 3, d_color_u, 3, R, 3, -1.0f, jobs.seed_value, jobs.seed_dev));
    return LNB_OK;
}

#ifdef LNB_WIDE_CLK
extern "C" LNB_API int lnb_test_wide_clk(unsigned long long *out8, int reset)
{
    if (out8 && cudaMemcpyFromSymbol(out8, g_wide_clk, sizeof(unsigned long long) * 8) != cudaSuccess) return LNB_ERR_CUDA;
    if (reset) { unsigned long long z[8] = {0}; if (cudaMemcpyToSymbol(g_wide_clk, z, sizeof(z)) != cudaSuccess) return LNB_ERR_CUDA; }
    return LNB_OK;
}
#endif
