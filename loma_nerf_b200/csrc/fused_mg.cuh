// fused_mg.cuh -- the fused tensor-core TRAIN step, multi-group form.  Included by fused_tc.cu inside its anonymous
// namespace (PTX wrappers, TcParams, TcLayout, the per-tile stages, SLAB / TILE / MAXL come from there).
//
// Why: a 128-sample tile takes ~10 000 cycles from features to weight gradients even alone on an SM (six dependent
// tcgen05 stages at ~555 + 145 g cycles each, three scans, five epilogues), a 4096 x 64 batch is only 13.8 tiles per
// SM, and fused_v1_kernel keeps 46 KB of activations + adjoints per tile alive, so 3-4 tiles share an SM and the launch
// is ceil(13.8 / 4) = 4-5 tile latencies long (measured: 39 us; the same kernel on a batch 8 x larger needs 25.8 us per
// 262 144 samples).  What helps is MORE TILES IN FLIGHT, i.e. less shared memory and TMEM per tile:
//   * ONE persistent CTA per SM holds up to seven independent 128-thread GROUPS; a group is what a CTA of the first
//     kernel was (thread r owns sample row r = TMEM lane r of the group's accumulator columns), synchronised with its
//     own named barrier and its own mbarriers.  The bf16 weight image is loaded once per SM instead of once per tile slot.
//   * adjoints are written IN PLACE: dZ_{l-1} = relu'(A_l) . dH_l has the shape of A_l and overwrites it, so a slot is
//     A_0 | dZ_{L-1} | A_1 .. A_{L-1} = 28 KB for the 33 -> 30 -> 30 -> 4 network instead of 46 KB.  The price: the
//     weight gradient of layer l, dW_l = A_l^T dZ_l, must be issued while both still exist -- per layer, next to the
//     dH_l MMAs, by the elected lanes of warps 1-3 (two or three K-steps each, so nobody issues for long) -- and the
//     in-place store waits for it (by then the epilogue arithmetic has hidden most of its latency).
//   * ALL groups accumulate their weight gradients into ONE set of TMEM columns (zeroed once with tcgen05.st; every
//     MMA accumulates): 7 x (32 result + 24 A-operand) columns + 80 gradient columns = 472 of the SM's 512, one partial per SM.
//   * shared memory is read by the tensor core only where an operand must be MN-major (the weight gradients) and for the
//     weights: every forward and dH MMA takes its A operand from TMEM, where the epilogue that writes A_l / dZ_l puts a
//     second copy with tcgen05.st (A_0 included, K0P / 2 columns).
//   * features mode: the fp32 tile is brought by one bulk-async copy into the slot's A_1.. region, which is dead between
//     the previous tile's last weight-gradient MMA and this tile's first epilogue -- no staging buffer.
// Forward-only launches (render) keep fused_v1_kernel: nothing is kept for a gradient there and nine 16 KB tiles
// already fit an SM.

constexpr int MG_MAX_GROUPS = 7;
constexpr int MG_MISC = 2304;       // per group: colour / target scratch, scan carries, mbarriers, MMA program
constexpr int MG_GLOBALS = 64;      // per CTA: weight-image mbarrier, TMEM base

template <int HP>
struct MgLayout {
    using LY = TcLayout<HP>;
    static constexpr int HSL = HP / 8;
    __host__ __device__ static int a0s(int c_in) { return (c_in + 8) >> 3; }   // slabs holding features 0..c_in (ones column included)
    // slot: A_0 [a0s] | dZ_{L-1} [1] | A_1 [HSL] .. A_{L-1} [HSL]
    __host__ __device__ static int dzl_off(int A0S) { return A0S * SLAB; }
    __host__ __device__ static int a_off(int l, int A0S) { return l == 0 ? 0 : (A0S + 1 + (l - 1) * HSL) * SLAB; }
    __host__ __device__ static int slot_bytes(int L, int c_in, int K0P, bool rays)
    {
        const int A0S = a0s(c_in);
        int nat = (A0S + 1 + (L - 1) * HSL) * SLAB;
        if (!rays) {   // the fp32 tile is staged from A_1 on
            const int need = a_off(1, A0S) + LY::stage_bytes(c_in, K0P);
            if (need > nat) nat = (need + 1023) / 1024 * 1024;
        }
        return nat;
    }
    __host__ __device__ static int ndw(int L) { return (L - 1) * HP + 16; }
    // per group HP result columns + the bf16 A operand of the forward / dH MMAs, whose widest is A_0 (K0P / 2 columns) or a
    // hidden layer (HP / 2)
    __host__ __device__ static int acols(int K0P) { return (K0P > HP ? K0P : HP) / 2; }
    __host__ __device__ static int tmem_need(int L, int K0P, int ng) { return ng * (HP + acols(K0P)) + ndw(L); }
    __host__ __device__ static size_t total(int L, int c_in, int K0P, bool rays, int ng)
    {
        const int A0S = a0s(c_in);
        const size_t slot = (size_t)slot_bytes(L, c_in, K0P, rays);
        const size_t t = ng * slot + LY::wimg_bytes(L, K0P) + MG_GLOBALS + (size_t)ng * MG_MISC;
        // a weight-gradient MMA reads 8 slabs (M = 64 feature rows) from the start of A_l whatever its real width (the rows
        // beyond are never read back): the last group's last such read must stay inside the allocation
        const size_t need = (ng - 1) * slot + a_off(L - 1, A0S) + 8 * SLAB;
        return t > need ? t : need;
    }
};

__device__ __forceinline__ void tmem_st16_zero(uint32_t taddr)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};" ::"r"(taddr), "r"(0u) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint4 v)   // one 8-feature slab of a row: 4 columns
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
template <int HP> constexpr int mg_max_groups() { return HP <= 32 ? MG_MAX_GROUPS : 4; }   // registers: 64 K / (groups x 128 threads)

// EXT: the extras instantiation (head_and_composite: weights, acc / depth, background), the one lnb_trainer_step_weights and
// a step with compositing extras run.  Its acc / depth scratch is the slot's dZ_{L-1} slab, dead until the head's adjoint
// is written into it (the previous tile's weight-gradient MMA that read it has been awaited in the backward loop).
// RAYS: 0 features, 1 rays or camera mode, 2 views mode (sample_inputs).
template <int RAYS, int HP, bool DIRS = false, bool EXT = false>
__global__ void __launch_bounds__(mg_max_groups<HP>() * TILE, 1) fused_mg_kernel(const TcParams p)
{
    using LY = TcLayout<HP>;
    using MG = MgLayout<HP>;
    extern __shared__ __align__(1024) uint8_t smem[];
#ifdef LNB_TC_CLK
    unsigned long long stamp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define MG_STAMP(i) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(stamp[i]))
    MG_STAMP(0);
#else
#define MG_STAMP(i)
#endif
    const int NG = (int)blockDim.x / TILE;
    const int g = (int)threadIdx.x / TILE, tid = (int)threadIdx.x % TILE, warp = tid >> 5, lane = tid & 31;
    const int L = p.L, K0P = p.K0P, c_in = p.dims[0], S = p.S;
    const int A0S = MG::a0s(c_in);
    const int slot_bytes = MG::slot_bytes(L, c_in, K0P, RAYS);
    uint8_t *const slot = smem + (size_t)g * slot_bytes;
    uint8_t *const Wbase = smem + (size_t)NG * slot_bytes;
    const float *const bias_s = reinterpret_cast<const float *>(Wbase + LY::w_off(L, L, K0P));
    uint8_t *const globals = Wbase + LY::wimg_bytes(L, K0P);
    uint8_t *const misc = globals + MG_GLOBALS + (size_t)g * MG_MISC;
    float *const stage = reinterpret_cast<float *>(slot + MG::a_off(1, A0S));   // features mode: fp32 tile, dead A_1.. region
    float *const color_s = reinterpret_cast<float *>(misc);     // [64][3]
    float *const tgt_s = color_s + 192;                         // [64][3]
    float *const tailp = tgt_s + 192;                           // [4] inclusive product at lane 31
    int *const tail_s = reinterpret_cast<int *>(tailp + 4);     // [4] sample index at lane 31
    float *const headq = tailp + 8;                             // [5] q at lane 0 of each warp
    float *const headA = tailp + 13;                            // [5]
    float *const headB = tailp + 18;                            // [5]
    float *const red_s = tailp + 24;                            // [4]
    uint64_t *const bar_p = reinterpret_cast<uint64_t *>(misc + 1664);
    const uint32_t bar_mma = smem_u32(bar_p), bar_x = smem_u32(bar_p + 1), bar_dw = smem_u32(bar_p + 2);
    const uint32_t bar_w = smem_u32(globals);
    uint32_t *const tmem_slot = reinterpret_cast<uint32_t *>(globals + 8);
    const CompScratch scratch{color_s, tgt_s, reinterpret_cast<float *>(slot + MG::dzl_off(A0S)), tailp, tail_s, headq, headA, headB};
    StageRec *const prog = reinterpret_cast<StageRec *>(misc + 1728);   // fwd l | dH l (L + l) | dW l (2L + l)

    auto a_buf = [&](int l) { return slot + MG::a_off(l, A0S); };
    uint8_t *const dzl_buf = slot + MG::dzl_off(A0S);
    // where the adjoint dZ_l lives: the last layer's in its own slab, the others in place of A_{l+1}
    auto dz_buf = [&](int l) { return l == L - 1 ? dzl_buf : a_buf(l + 1); };

    // ---- one-time setup.  Every buffer is fully rewritten each tile before an MMA reads it as data (the K padding of A_0
    // included, in TMEM); what an M = 64 weight-gradient MMA reads past a short A_l only reaches accumulator rows never read.
    if (tid == 0) {
        mbar_init(bar_mma, 1);
        mbar_init(bar_x, 1);
        mbar_init(bar_dw, 3);          // the three threads that issue a layer's weight-gradient MMAs
        if (g == 0) mbar_init(bar_w, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // features mode: a round of tiles starts on every SM at once and asks HBM for 17 KB per group -- 17 MB, 2.7 us at
        // full bandwidth.  The first tile's copy therefore goes out NOW, under the rest of the prologue (and, with PDL,
        // under the previous kernel's tail: X is never written by it), and every later tile is pulled into L2 a tile ahead.
        if (!RAYS) {
            const int t0 = g * (int)gridDim.x + (int)blockIdx.x;
            if (t0 < p.n_tiles) {
                int lead; uint32_t bytes;
                const void *src = x_src(p, t0, c_in, lead, bytes);
                mbar_expect_tx(bar_x, bytes);
                bulk_g2s(smem_u32(stage), src, bytes, bar_x);
            }
        }
    }
    // the MMA program: one record per stage, one THREAD per record (a single thread building all of them cost 3 us)
    if (tid >= 32 && tid < 32 + 3 * L) {
        const int r = tid - 32, kind = r / L, l = r % L;
        const uint32_t dcol = (uint32_t)(g * HP), acol = (uint32_t)(NG * HP + MG::ndw(L) + g * MG::acols(K0P));
        const int Np = LY::np(l, L), Kp = LY::kp(l, K0P);
        const uint32_t wl = smem_u32(Wbase + LY::w_off(l, L, K0P));
        if (kind == 0) {               // D[128 x Np] = A_l[128 x Kp] * W_l: A from TMEM (8 columns per K-step), B K-major
            prog[l] = StageRec{(uint64_t)acol, smem_desc(wl, Np * 16, 128), 8u, (uint32_t)(2 * Np * 16) >> 4,
                               instr_desc(128, Np, 0, 0), dcol, (uint32_t)(Kp / 16), 1u, 0u, 0u};
        } else if (kind == 1) {        // dH_l[128 x Kp] = dZ_l[128 x Np] * W_l^T (same W bytes, MN-major); unused for l = 0
            prog[L + l] = StageRec{(uint64_t)acol, smem_desc(wl, 128, Np * 16), 8u, 256u >> 4,
                                   instr_desc(128, Kp, 0, 1), dcol, (uint32_t)(Np / 16), 1u, 0u, 0u};       // A = dZ_l from TMEM
        } else {                       // dW_l[features x Np] += A_l^T dZ_l, K = the tile's 128 samples, both MN-major
            prog[2 * L + l] = StageRec{smem_desc(smem_u32(a_buf(l)), 128, SLAB), smem_desc(smem_u32(dz_buf(l)), 128, SLAB), 256u >> 4, 256u >> 4,
                                       instr_desc(64, Np, 1, 1), (uint32_t)(NG * HP + l * HP), (uint32_t)(TILE / 16), 0u, 0u, 0u};
        }
    }
    const uint32_t tmem_cols = tmem_alloc_cols(MG::tmem_need(L, K0P, NG));
    if (g == 0 && warp == 0) tmem_alloc(smem_u32(tmem_slot), tmem_cols);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    // the shared weight-gradient accumulator starts at zero; every MMA into it accumulates
    if (g == 0) {
        for (int c = 0; c < MG::ndw(L); c += 16) tmem_st16_zero(tmem + lane_base + (uint32_t)(NG * HP + c));
        tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // Programmatic dependent launch: all of the above overlapped the tail of the previous kernel in the stream.  Only OUR
    // reduce kernel triggers its dependents early, and the one thing of its output this kernel reads is the weight image:
    // ONE thread waits for it and issues the bulk copy of the image; the others go straight to their first tile's features
    // and meet the image at its mbarrier (which also orders their later global writes behind that kernel).  No-op without PDL.
    if (threadIdx.x == 64) {
        pdl_wait();
        const uint32_t wb = (uint32_t)LY::wimg_bytes(L, K0P);
        mbar_expect_tx(bar_w, wb);
        bulk_g2s(smem_u32(Wbase), p.wimg, wb, bar_w);
    }
    pdl_trigger();
    uint32_t phase = 0, xphase = 0, dwphase = 0;
    float loss_acc = 0.0f;
    bool dw_pending = false, have_weights = false;
    MG_STAMP(1);

    auto row_ptr = [&](uint8_t *buf, int slab) { return reinterpret_cast<uint4 *>(buf + slab * SLAB + tid * 16); };
    const uint32_t a_tm = tmem + lane_base + (uint32_t)(NG * HP + MG::ndw(L) + g * MG::acols(K0P));   // this row's bf16 A operand
    auto commit_and_wait = [&]() {
        if (tid == 0) umma_commit(bar_mma);
        mbar_wait_tight(bar_mma, phase);
        phase ^= 1;
        tc_fence_after();
    };
    auto publish_smem = [&]() { // generic-proxy smem writes -> visible to the tensor core, all threads of the group
        fence_async_smem();
        tc_fence_before();
        bar_tile(g + 1);
        tc_fence_after();
    };
    // the same for tcgen05.st -> MMA only.  The forward's shared-memory stores (A_0 .. A_{L-1}) are read by the tensor core
    // only through the weight-gradient MMAs, which are issued after the backward's first publish_smem: its proxy fence
    // covers them, so the forward needs none of its own.
    auto publish_tmem = [&]() {
        tc_fence_before();
        bar_tile(g + 1);
        tc_fence_after();
    };
    // the weight-gradient MMAs of layer l: 8 K-steps of 16 samples, dealt 3 / 3 / 2 to the elected lanes of warps 1-3; every
    // one accumulates into the shared accumulator
    auto issue_dw = [&](int l) {
        if (lane == 0 && warp > 0) {
            const uint32_t k0 = warp == 1 ? 0u : (warp == 2 ? 3u : 6u), k1 = warp == 1 ? 3u : (warp == 2 ? 6u : 8u);
            issue_steps<true>(prog + 2 * L + l, tmem, k0, k1, 1u);
            umma_commit(bar_dw);
        }
    };
    auto wait_dw = [&]() { mbar_wait_tight(bar_dw, dwphase); dwphase ^= 1; tc_fence_after(); };

    // tiles are dealt statically (tile -> group fixed): with equal tile costs nothing is gained by claiming them, and
    // nothing here then depends on the previous kernel in the stream except the weight image
    for (int tile = g * (int)gridDim.x + (int)blockIdx.x; tile < p.n_tiles; tile += (int)gridDim.x * NG) {
        const long long row0 = (long long)tile * p.rows_per_tile;
        long long rem = p.N - row0;
        const int valid = rem < p.rows_per_tile ? (int)rem : p.rows_per_tile;
        const int rays_here = valid == p.rows_per_tile ? p.G : valid / S;
        const int smp = tid % S, ray_l = tid / S;        // this thread's sample within its ray
        const bool live = tid < rays_here * S;
        // the previous tile's last weight-gradient MMAs read A_0 and A_1's buffer (dZ_0): both are rewritten below
        if (dw_pending) { wait_dw(); dw_pending = false; }
        if (!RAYS && tid == 0) {
            int lead; uint32_t bytes;
            if (have_weights) {                    // (the first tile's copy was issued in the prologue)
                const void *src = x_src(p, tile, c_in, lead, bytes);
                mbar_expect_tx(bar_x, bytes);
                bulk_g2s(smem_u32(stage), src, bytes, bar_x);
            }
            const int nxt = tile + (int)gridDim.x * NG;
            if (nxt < p.n_tiles) { const void *src = x_src(p, nxt, c_in, lead, bytes); bulk_prefetch_l2(src, bytes); }
        }
        float x[3], my_dist, tg[3], u[3];
        sample_inputs<RAYS, DIRS>(p, row0, tile * p.G, tid, smp, ray_l, live, x, my_dist, tg, u);
        // A_0 goes to shared memory (for the weight gradient, MN-major) and to TMEM (the layer-0 MMA's A operand)
        auto store_a0 = [&](int c8, uint4 q) { *row_ptr(a_buf(0), c8) = q; tmem_st4(a_tm + (uint32_t)c8 * 4u, q); };
        if (DIRS) {
            // ---- features from rays with the view direction
            pack_pe_dirs(x, u, p.pe_bands, p.dir_bands, store_a0);
        } else if (RAYS) {
            // ---- features from rays: the positional encoding, written straight into A_0
            float sn[3], cs[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) pe_sincos(x[c], &sn[c], &cs[c]);
            pack_pe(x, sn, cs, p.pe_bands, A0S, store_a0);
        } else {
            // ---- features: wait for the TMA, convert this thread's row to bf16 slabs (tcgen05.st is warp-wide: the rows
            // past `valid` store zeros in the same instruction)
            int lead; uint32_t bytes;
            (void)x_src(p, tile, c_in, lead, bytes);
            mbar_wait(bar_x, xphase);
            xphase ^= 1;
            pack_features(stage + lead + tid * c_in, c_in, tid < valid, store_a0);
        }
        // A_0's K padding in TMEM: explicit zeros (they meet zero weight rows, but stale TMEM bits could be NaN)
        for (int c8 = A0S; c8 < K0P / 8; ++c8) tmem_st4(a_tm + (uint32_t)c8 * 4u, make_uint4(0, 0, 0, 0));
        tmem_st_wait();
        if (!have_weights) {
            mbar_wait(bar_w, 0);             // weights + biases have landed (and the previous kernel has completed)
            have_weights = true;
            MG_STAMP(2);
        }
        publish_tmem(); // also: every thread is done reading `stage` (the first epilogue overwrites it)
        // ---- forward
        float hz[4];
        for (int l = 0; l < L; ++l) {
            if (tid == 0) issue_steps<true>(prog + l, tmem, 0u, 64u, 0u);
            commit_and_wait();
            const float *bl = bias_s + l * HP;
            if (l < L - 1) {
                uint8_t *an = a_buf(l + 1);
                uint32_t v[HP / 16][16];
#pragma unroll
                for (int c16 = 0; c16 < HP / 16; ++c16) tmem_ld16(tmem + lane_base + (uint32_t)(g * HP + c16 * 16), v[c16]);
                tmem_ld_wait();
                // the hidden layers' bias and the all-ones feature of the next layer's input came out of the MMA (see
                // tc_prep_kernel): ReLU + round + pack is one instruction per pair
#pragma unroll
                for (int c16 = 0; c16 < HP / 16; ++c16) {
                    uint32_t o[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = pack_relu_bf16(__uint_as_float(v[c16][2 * j]), __uint_as_float(v[c16][2 * j + 1]));
                    *row_ptr(an, c16 * 2) = make_uint4(o[0], o[1], o[2], o[3]);       // for the weight gradient (MN-major operand)
                    *row_ptr(an, c16 * 2 + 1) = make_uint4(o[4], o[5], o[6], o[7]);
                    tmem_st8(a_tm + (uint32_t)(c16 * 8), o);                          // for the next layer's MMA (A from TMEM)
                }
                tmem_st_wait();
                publish_tmem();
            } else {
                uint32_t v[16];
                tmem_ld16(tmem + lane_base + (uint32_t)(g * HP), v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 4; ++j) hz[j] = __uint_as_float(v[j]) + bl[j];
            }
        }
        // ---- head + loss + adjoint of the head's pre-activation (unit seed)
        float dz[4];
        head_and_composite<true, EXT, RAYS == 2>(p, scratch, g + 1, hz, my_dist, tg, row0, tile * p.G, valid, tid, smp, ray_l, live, loss_acc, dz);
        // ---- backward.  dZ_{L-1}: 4 live features of its one slab
        {
            const uint32_t o[8] = {pack_bf16(dz[0], dz[1]), pack_bf16(dz[2], dz[3]), 0u, 0u, 0u, 0u, 0u, 0u};
            *row_ptr(dzl_buf, 0) = make_uint4(o[0], o[1], 0u, 0u);
            tmem_st8(a_tm, o);
            tmem_st_wait();
        }
        publish_smem();
        for (int l = L - 1; l >= 1; --l) {
            if (tid == 0) issue_steps<true>(prog + L + l, tmem, 0u, 64u, 0u);
            issue_dw(l);                       // dW_l = A_l^T dZ_l while both are still there
            commit_and_wait();
            uint8_t *al = a_buf(l);
            uint32_t v[HP / 16][16];
#pragma unroll
            for (int c16 = 0; c16 < HP / 16; ++c16) tmem_ld16(tmem + lane_base + (uint32_t)(g * HP + c16 * 16), v[c16]);
            uint4 hm[HP / 8];
#pragma unroll
            for (int c8 = 0; c8 < HP / 8; ++c8) hm[c8] = *row_ptr(al, c8);
            tmem_ld_wait();
            uint4 oz[HP / 8];
            relu_adjoint<HP>(v, hm, oz);
            if (l > 1) {                       // dZ_{l-1} is the A operand of the next dH MMA
#pragma unroll
                for (int c16 = 0; c16 < HP / 16; ++c16) {
                    const uint32_t o[8] = {oz[2 * c16].x, oz[2 * c16].y, oz[2 * c16].z, oz[2 * c16].w, oz[2 * c16 + 1].x, oz[2 * c16 + 1].y, oz[2 * c16 + 1].z, oz[2 * c16 + 1].w};
                    tmem_st8(a_tm + (uint32_t)(c16 * 8), o);
                }
                tmem_st_wait();
            }
            wait_dw();                         // ... and only now may A_l become dZ_{l-1}
#pragma unroll
            for (int c8 = 0; c8 < HP / 8; ++c8) *row_ptr(al, c8) = oz[c8];
            publish_smem();
        }
        issue_dw(0);                           // dW_0 = A_0^T dZ_0 in the background; awaited at the top of the next tile
        dw_pending = true;
#ifdef LNB_TC_CLK
        if (stamp[3] == 0) MG_STAMP(3);
        MG_STAMP(4);
#endif
    }
    if (!have_weights) mbar_wait(bar_w, 0);    // a group without tiles still orders its partial writes behind the previous kernel

    // ---- epilogue: this CTA's partials.  loss, then per layer the valid (in_l+1) x out_l block.
    if (dw_pending) wait_dw();
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) loss_acc += __shfl_xor_sync(0xffffffffu, loss_acc, d);
    if (lane == 0) red_s[warp] = loss_acc;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    MG_STAMP(5);
    float *part = p.part + (size_t)blockIdx.x * p.part_stride;
    if (threadIdx.x == 0) {
        float s = 0.0f;
        for (int gg = 0; gg < NG; ++gg) {
            const float *r = reinterpret_cast<const float *>(globals + MG_GLOBALS + (size_t)gg * MG_MISC) + 384 + 24;
            s += (r[0] + r[1]) + (r[2] + r[3]);
        }
        part[0] = s;
        if (blockIdx.x == 0 && p.t_dev) p.t_dev[0] += 1; // read by the kernels that follow in the stream
    }
    // M = 64 accumulators occupy half of every lane quadrant: feature row f sits in TMEM lane 32 (f / 16) + f % 16; thread tid of
    // a group reads lane tid.  The 16-column chunks of the gradient columns are dealt round-robin to the groups.
    {
        int chunk = 0;
        for (int l = 0; l < L; ++l) {
            const int in_l = p.dims[l], out_l = p.dims[l + 1], Np = LY::np(l, L);
            float *o = part + p.part_off[l];
            for (int c16 = 0; c16 * 16 < Np; ++c16, ++chunk) {
                if (chunk % NG != g || c16 * 16 >= out_l) continue;
                uint32_t v[16];
                tmem_ld16(tmem + lane_base + (uint32_t)(NG * HP + l * HP + c16 * 16), v);
                tmem_ld_wait();
                const int f = warp * 16 + lane;
                if (lane < 16 && f <= in_l) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int col = c16 * 16 + j;
                        if (col < out_l) o[f * out_l + col] = __uint_as_float(v[j]);
                    }
                }
            }
        }
    }
    MG_STAMP(7);
    tc_fence_before();
    __syncthreads();
    if (g == 0 && warp == 0) tmem_dealloc(tmem, tmem_cols);
#ifdef LNB_TC_CLK
    MG_STAMP(6);
    if (p.dbg && tid == 0) {
        unsigned long long *o = reinterpret_cast<unsigned long long *>(p.dbg) + ((size_t)blockIdx.x * NG + g) * 8;
        for (int i = 0; i < 8; ++i) o[i] = stamp[i];
    }
#endif
}
