// Fused Swin MLP half for sm_100a:   z = y + fc2( GELU_erf( fc1( LayerNorm(y) ) ) )      (src/drct.py:510, 173-190)
//
// One persistent, warp-specialised kernel (grid = #SMs, 21 warps).  A CTA owns 128 token rows at a time; the hidden
// activations [128 x H] never leave the SM:
//   * the y tile [128 x C] arrives by TMA (128-byte swizzle, K / M tails zero-filled) into one of TWO shared-memory
//     buffers; it is the A operand of fc1, the residual of the last epilogue, and -- overwritten in place with z -- the
//     source of the TMA store of the result.  The warp that stores tile i reloads the freed buffer with tile i+2;
//   * the weights of fc1 (gamma-folded) and fc2 stream from L2 through two rings of shared-memory slots (one
//     [rows x 64] slab per slot), each fed by its own loader warp in the fixed order its consumer uses them;
//   * fc1 is computed in hidden chunks of <= 128 columns into a double-buffered TMEM accumulator (tcgen05.mma, SS);
//     16 epilogue warps turn a chunk into bf16 GELU activations (LayerNorm folded: rstd * (acc - mean * colsum) + b),
//     16 columns (one K=16 step of fc2) at a time, and write them back IN PLACE into the first 8 of those 16 TMEM
//     columns (tcgen05.st), from where fc2 consumes them as its TMEM A operand (tcgen05.mma, TS);
//   * fc2 accumulates over the chunks into a third TMEM region; the last epilogue adds bias and the residual.
// TWO MMA-issuing warps (one for fc1, one for fc2) keep the tensor core fed: the per-slab bookkeeping of one stream
// (mbarrier waits, commits) overlaps the MMAs of the other, and fc1 runs up to two chunks ahead of fc2 -- across tile
// borders -- limited only by the two chunk accumulators (barrier acc1_free, committed by the fc2 issuer).
// The 0.5 of GELU is folded into the packed fc2 weights.
#include "adsr_kernels.h"
#include "ptx.cuh"

namespace adsr {

namespace {

constexpr int kEpiWarps = 16;                 // warps 0..15: epilogue (TMEM lane quadrant = warp % 4)
constexpr int kW1LoaderWarp = 16;             // fc1 weight slabs
constexpr int kFc1Warp = 17;                  // fc1 MMA issuer
constexpr int kFc2Warp = 18;                  // fc2 MMA issuer
constexpr int kW2LoaderWarp = 19;             // fc2 weight slabs
constexpr int kTileWarp = 20;                 // the first aux warp also does: TMEM alloc, y-tile loads, z-tile stores
constexpr int kAuxWarp0 = 20;                 // warps 20..23 (TMEM lane quadrant = warp % 4): row mean / rstd two tiles ahead, folded-adjust epilogue
constexpr int kThreads = 24 * 32;             // 24 warps: 80 registers per thread (a 25th warp costs 8 of them to the allocation granularity)
constexpr int kPanelBytes = 128 * 128;        // 128 rows x 64 bf16
constexpr int kMaxHidden = 640;               // padded hidden columns (sum of chunk strides)
constexpr int kMaxN2 = 320;
constexpr int kRowStatBytes = 2 * 128 * 8;    // (rstd, -mean * rstd) of two tiles
// bias1 / colsum1 (padded hidden width each) / bias2 caches + row statistics
__host__ __device__ constexpr int const_bytes(int hidden_padded, int n2) { return (2 * hidden_padded + n2) * 4 + kRowStatBytes; }
constexpr int kSmemLimit = 232448;            // 227 KB
constexpr int kAdjSlabBytes = 32 * 128;       // folded adjust: 32 output rows x 64 bf16
constexpr int kAdjStageBytes = 4 * 32 * 64;   // folded adjust: one [32 rows x 32 bf16] staging box per aux warp (16-byte chunks swizzled)

struct __align__(16) MlpBarriers {
    uint64_t w1_full[8], w1_empty[8];
    uint64_t w2_full[8], w2_empty[8];
    uint64_t a_full[2];
    uint64_t z_ready[2];
    uint64_t acc1_full[3];
    uint64_t acc1_free[3];
    uint64_t h_ready[3][2];                   // [accumulator buffer][64-column slab of the chunk]
    uint64_t acc2_full[2];                    // [1] only with the folded adjust, whose 32-column accumulator is double-buffered
    uint64_t acc2_free[2];
    uint64_t adj_w_full;                      // folded adjust: the resident W_adj slabs have landed
    uint64_t adj_done[2];                     // folded adjust: fc1 and the y W_adj^T MMAs have finished reading the y tile in buffer b
    uint64_t rs_full[2], rs_free[2];          // (rstd, -mean * rstd) of a tile's rows in s_rowstat[tile parity]
    uint64_t res_full[2];                     // fold_res: the residual tile has replaced the (consumed) y tile in buffer b
    uint32_t tmem_base;
};

__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }

// 2 * GELU(x) for a pair:  x + |x| * (1 - erfc(|x| / sqrt 2)),  erfc(a / sqrt 2) ~ 2^(a * q(a)) with q a NEGATED quadratic:
// |error| <= 8.6e-5 after the 0.5 that lives in the fc2 weights (activations are rounded to bf16 right after).
__device__ __forceinline__ float2 gelu2_pair(float2 x) {
    const float2 a = f2(fabsf(x.x), fabsf(x.y));          // folds into |R| operand modifiers of FFMA2 / FMUL2
    float2 q = __ffma2_rn(f2(-0.027645503f, -0.027645503f), a, f2(-0.48822206f, -0.48822206f));
    q = __ffma2_rn(q, a, f2(-1.1409364f, -1.1409364f));
    const float2 m = __fmul2_rn(q, a);
    const float2 e = f2(ex2_approx(m.x), ex2_approx(m.y));
    const float2 g = __ffma2_rn(e, f2(-1.f, -1.f), f2(1.f, 1.f));
    return __ffma2_rn(a, g, x);
}

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
                 "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}

// optional timeline of CTA 0 (tools/mlp_trace.py): trace[((role * 8 + tile) * 64 + index) * 8 + k] = clock64()
template <bool TRACE>
__device__ __forceinline__ void trace_ev(long long* trace, int role, int it, int idx, int k) {
    if constexpr (TRACE) {
        if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && it < 8 && idx < 64) trace[((role * 8 + it) * 64 + idx) * 8 + k] = clock64();
    }
}

template <bool TRACE>
__global__ void __launch_bounds__(kThreads, 1) swin_mlp_kernel(const __grid_constant__ SwinMlpParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* a_buf = smem;                                            // 2 x a_buf_bytes
    uint8_t* ring1 = smem + 2 * p.a_buf_bytes;                        // w1_slots x w1_slot_bytes
    uint8_t* ring2 = ring1 + p.w1_slots * p.w1_slot_bytes;            // w2_slots x w2_slot_bytes
    uint8_t* wadj_s = ring2 + p.w2_slots * p.w2_slot_bytes;           // fused adjust: ks1 x [32 x 64] weight slabs (resident)
    uint8_t* adj_stage = wadj_s + (p.fuse_adj ? p.ks1 * kAdjSlabBytes : 0);   // folded adjust: output boxes of the aux warps
    float* s_bias1 = reinterpret_cast<float*>(adj_stage + (p.fuse_adj ? kAdjStageBytes : 0));
    float* s_colsum1 = s_bias1 + p.nc * p.hc;                         // multiples of 16 floats: float4 reads stay aligned
    float* s_bias2 = s_colsum1 + p.nc * p.hc;
    float2* s_rowstat = reinterpret_cast<float2*>(s_bias2 + p.n2);  // [2 tile parities][128 rows]: (rstd, -mean * rstd)
    MlpBarriers* bars = reinterpret_cast<MlpBarriers*>(s_rowstat + 256);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // fc1 chunk accumulators: two, or three where the TMEM columns allow (folded adjust: fc1 then runs two chunks ahead of the
    // conversion, so a chunk never waits for the fc2 of the chunk two before it)
    // fc2 accumulator of tile it: one, or (folded adjust: 32 columns) two so that the next tile's MMAs never wait for the aux warps
    auto acc2_buf = [&](int it) -> int { return p.fuse_adj ? it & 1 : 0; };
    auto acc2_phase = [&](int it) -> uint32_t { return static_cast<uint32_t>(p.fuse_adj ? it >> 1 : it) & 1u; };
    auto acc1_buf = [&](int cg) -> int { return p.n_acc1 == 3 ? cg % 3 : cg & 1; };
    auto acc1_phase = [&](int cg) -> uint32_t { return static_cast<uint32_t>(p.n_acc1 == 3 ? cg / 3 : cg >> 1) & 1u; };
    const int my_tiles = static_cast<int>(blockIdx.x) < p.m_tiles ? (p.m_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    auto tile_of = [&](int it) -> int {                                // forward, or from the last tile down (p.rev)
        const int t = it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
        return p.rev ? p.m_tiles - 1 - t : t;
    };

    if ((smem_u32(smem) & 1023u) != 0) __trap();

    for (int i = threadIdx.x; i < p.nc * p.hc; i += kThreads) {
        s_bias1[i] = p.bias1[i];
        s_colsum1[i] = p.colsum1[i];
    }
    // folded adjust: the accumulator's bias is the adjust conv's (with W_adj b2 folded in on the host)
    for (int i = threadIdx.x; i < p.n2; i += kThreads) s_bias2[i] = p.fuse_adj ? p.bias_adj[i] : p.bias2[i];

    if (warp == kFc1Warp && lane == 0) {
        for (int s = 0; s < 8; ++s) {
            mbar_init(&bars->w1_full[s], 1);
            mbar_init(&bars->w1_empty[s], 1);
            mbar_init(&bars->w2_full[s], 1);
            mbar_init(&bars->w2_empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&bars->a_full[b], 1);
            mbar_init(&bars->z_ready[b], kEpiWarps);
            mbar_init(&bars->rs_full[b], 4);
            mbar_init(&bars->rs_free[b], kEpiWarps);
            mbar_init(&bars->res_full[b], 1);
        }
        for (int b = 0; b < 3; ++b) {
            mbar_init(&bars->acc1_full[b], 1);
            mbar_init(&bars->acc1_free[b], 1);
            mbar_init(&bars->h_ready[b][0], kEpiWarps);
            mbar_init(&bars->h_ready[b][1], kEpiWarps);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&bars->acc2_full[b], 1);
            mbar_init(&bars->acc2_free[b], p.fuse_adj ? 4 : kEpiWarps);   // folded adjust: its own four warps read the accumulator
        }
        mbar_init(&bars->adj_w_full, 1);
        // folded adjust: the tile buffer is free once its fc1 and y W_adj^T MMAs (one or two issuing warps) have completed
        mbar_init(&bars->adj_done[0], (p.fuse_adj && p.adjy_fc1) ? 1 : 2);
        mbar_init(&bars->adj_done[1], (p.fuse_adj && p.adjy_fc1) ? 1 : 2);
        fence_barrier_init();
    }
    if (warp == kTileWarp) tmem_alloc<512>(&bars->tmem_base);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = bars->tmem_base;
    // programmatic dependent launch: set-up and weight loaders overlap the predecessor's tail; the warps that touch activations or
    // row statistics (tile loads / stores, epilogues) wait for it to complete
    pdl_launch_dependents();
    if (warp < kEpiWarps || warp >= kTileWarp) pdl_wait();

    // folded adjust: W_adj (y + fc2(g)) = y W_adj^T + g (W_adj W2)^T -- the fc2 ring carries the 32 rows of W_adj W2, the accumulator is
    // 32 columns wide, and the y term goes in first, straight from the tile buffer (the caller has waited for a_full / acc2_free).
    // Either MMA issuer can take it (p.adjy_fc1): the fc2 issuer's 4-MMA batches cost ~350 cycles each (profiles/r02_mma_bench.txt),
    // so for narrow blocks (3 K slabs) it is better off without these 12 MMAs; for the wide ones the fc1 issuer is the busier warp.
    auto issue_adj_y = [&](int it) {
        tc_fence_after_sync();
        if (elect_one_sync()) {
            const uint64_t a_desc = umma_desc_k_sw128(smem_u32(a_buf)) + static_cast<uint64_t>((it & 1) * static_cast<uint32_t>(p.a_buf_bytes >> 4));
            const uint64_t b_desc = umma_desc_k_sw128(smem_u32(wadj_s));
            const uint32_t idesc = umma_idesc_bf16_m128(32u);
            const uint32_t d = tmem + static_cast<uint32_t>(p.piece_col[0] + 32 * acc2_buf(it));
            for (int s = 0; s < p.ks1; ++s) {                          // straight-line groups of 4: MMAs issued from a rolled inner loop
                const int ksteps = min(4, p.k1steps - 4 * s);           // cost the issuing thread 100-280 cycles each
                const uint64_t ad = a_desc + static_cast<uint64_t>(s * (kPanelBytes >> 4)), bd = b_desc + static_cast<uint64_t>(s * (kAdjSlabBytes >> 4));
                umma_bf16(d, ad, bd, idesc, s > 0 ? 1u : 0u);
                if (ksteps > 1) umma_bf16(d, ad + 2, bd + 2, idesc, 1u);
                if (ksteps > 2) umma_bf16(d, ad + 4, bd + 4, idesc, 1u);
                if (ksteps > 3) umma_bf16(d, ad + 6, bd + 6, idesc, 1u);
            }
        }
        __syncwarp();
    };

    // The control warps below stay CONVERGED (uniform control flow, one elected lane issues): descriptors then live in
    // uniform registers and no tcgen05 / bulk-copy instruction gets wrapped in a lane-serialising loop.
    if (warp == kW1LoaderWarp) {
        // ============================================================ fc1 weight slabs: (chunk j, K slab s) in order, every tile
        int slot = 0;
        uint32_t phase = 0;
        for (int it = 0; it < my_tiles; ++it) {
            uint32_t goff = 0;
            for (int j = 0; j < p.nc; ++j) {
                const uint32_t bytes = static_cast<uint32_t>(p.hcw[j]) * 128u;
                for (int s = 0; s < p.ks1; ++s) {
                    mbar_wait(&bars->w1_empty[slot], phase ^ 1);
                    if (elect_one_sync()) {
                        mbar_arrive_expect_tx(&bars->w1_full[slot], bytes);
                        bulk_g2s(ring1 + slot * p.w1_slot_bytes, p.w1p + goff, bytes, &bars->w1_full[slot]);
                    }
                    __syncwarp();
                    goff += bytes;
                    if (++slot == p.w1_slots) { slot = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kW2LoaderWarp) {
        // ============================================================ fc2 weight slabs: (chunk j, K slab s, N piece) in order
        int slot = 0;
        uint32_t phase = 0;
        for (int it = 0; it < my_tiles; ++it) {
            uint32_t goff = 0;
            int yq = 0;
            for (int j = 0; j < p.nc; ++j) {
                const int nslab = (p.hcw[j] + 63) >> 6;
                if (p.fold_res) {                                    // wide folded conv: p.ypre[j] slabs of W_a go in front of chunk j
                    for (int q = 0; q < p.ypre[j]; ++q, ++yq) {
                        const uint32_t bytes = static_cast<uint32_t>(p.piece_rows[yq % p.n_pieces]) * 128u;
                        mbar_wait(&bars->w2_empty[slot], phase ^ 1);
                        if (elect_one_sync()) {
                            mbar_arrive_expect_tx(&bars->w2_full[slot], bytes);
                            bulk_g2s(ring2 + slot * p.w2_slot_bytes, p.w2p + goff, bytes, &bars->w2_full[slot]);
                        }
                        __syncwarp();
                        goff += bytes;
                        if (++slot == p.w2_slots) { slot = 0; phase ^= 1; }
                    }
                }
                for (int s = 0; s < nslab; ++s) {
                    for (int pc = 0; pc < p.n_pieces; ++pc) {
                        const uint32_t bytes = static_cast<uint32_t>(p.piece_rows[pc]) * 128u;
                        mbar_wait(&bars->w2_empty[slot], phase ^ 1);
                        if (elect_one_sync()) {
                            mbar_arrive_expect_tx(&bars->w2_full[slot], bytes);
                            bulk_g2s(ring2 + slot * p.w2_slot_bytes, p.w2p + goff, bytes, &bars->w2_full[slot]);
                        }
                        __syncwarp();
                        goff += bytes;
                        if (++slot == p.w2_slots) { slot = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == kFc1Warp) {
        // ============================================================ fc1 MMA issuer: acc1[cg % n_acc1] = y_tile . W1_chunk^T
        int slot = 0;
        uint32_t phase = 0;
        const uint32_t slot_units = static_cast<uint32_t>(p.w1_slot_bytes >> 4);
        const uint64_t ring_desc = umma_desc_k_sw128(smem_u32(ring1));
        const uint64_t a_desc0 = umma_desc_k_sw128(smem_u32(a_buf));
        const uint32_t a_units = static_cast<uint32_t>(p.a_buf_bytes >> 4);
        for (int it = 0; it < my_tiles; ++it) {
            trace_ev<TRACE>(p.trace, 0, it, 1, 0);
            mbar_wait(&bars->a_full[it & 1], static_cast<uint32_t>(it >> 1) & 1);
            trace_ev<TRACE>(p.trace, 0, it, 1, 1);
            const uint64_t a_desc = a_desc0 + static_cast<uint64_t>((it & 1) * a_units);
            if (p.fuse_adj && p.adjy_fc1) {
                // issued in front of the tile's fc1 chunks: the fc2 MMAs that accumulate on top are only issued after the conversion
                // of a chunk whose completion this thread commits later, so the tensor pipe sees them in the right order
                if (it == 0) mbar_wait(&bars->adj_w_full, 0);
                mbar_wait(&bars->acc2_free[acc2_buf(it)], acc2_phase(it) ^ 1);     // the aux warps have read tile it - 2
                issue_adj_y(it);
            }
            for (int j = 0; j < p.nc; ++j) {
                const int cg = it * p.nc + j;                         // running chunk counter: buffer = cg % n_acc1, use = cg / n_acc1
                const int b = acc1_buf(cg);
                const uint32_t idesc = umma_idesc_bf16_m128(static_cast<uint32_t>(p.hcw[j]));
                const uint32_t acc1 = tmem + static_cast<uint32_t>(p.acc1_col[b]);
                trace_ev<TRACE>(p.trace, 1, it, j, 0);
                mbar_wait(&bars->acc1_free[b], acc1_phase(cg) ^ 1);   // fc2 of chunk cg - n_acc1 has consumed it
                trace_ev<TRACE>(p.trace, 1, it, j, 1);
                for (int s = 0; s < p.ks1; ++s) {
                    const int ksteps = min(4, p.k1steps - 4 * s);
                    mbar_wait(&bars->w1_full[slot], phase);
                    tc_fence_after_sync();
                    if (elect_one_sync()) {
                        const uint64_t adesc = a_desc + static_cast<uint64_t>(s * (kPanelBytes >> 4));
                        const uint64_t bdesc = ring_desc + static_cast<uint64_t>(static_cast<uint32_t>(slot) * slot_units);
                        umma_bf16(acc1, adesc, bdesc, idesc, s == 0 ? 0u : 1u);
                        if (ksteps > 1) umma_bf16(acc1, adesc + 2, bdesc + 2, idesc, 1u);
                        if (ksteps > 2) umma_bf16(acc1, adesc + 4, bdesc + 4, idesc, 1u);
                        if (ksteps > 3) umma_bf16(acc1, adesc + 6, bdesc + 6, idesc, 1u);
                        umma_commit(&bars->w1_empty[slot]);
                        if (s == p.ks1 - 1) {
                            umma_commit(&bars->acc1_full[b]);
                            if ((p.fuse_adj || p.fold_res) && j == p.nc - 1) umma_commit(&bars->adj_done[it & 1]);   // last read of the y tile by fc1
                        }
                    }
                    __syncwarp();
                    if (++slot == p.w1_slots) { slot = 0; phase ^= 1; }
                }
                trace_ev<TRACE>(p.trace, 1, it, j, 2);
            }
        }
    } else if (warp == kFc2Warp) {
        // ============================================================ fc2 MMA issuer: acc2 += gelu_chunk (TMEM) . W2_chunk^T
        int slot = 0;
        uint32_t phase = 0;
        const uint32_t slot_units = static_cast<uint32_t>(p.w2_slot_bytes >> 4);
        const uint64_t ring_desc = umma_desc_k_sw128(smem_u32(ring2));
        for (int it = 0; it < my_tiles; ++it) {
            uint32_t acc2_started = 0u;                                // fold_res: bit pc = this N piece of acc2 has been written in this tile
            int yq = 0;                                                // fold_res: next (K slab, N piece) slab of W_a
            for (int j = 0; j < p.nc; ++j) {
                const int cg = it * p.nc + j;
                const int b = acc1_buf(cg);
                const int nslab = (p.hcw[j] + 63) >> 6;
                const uint32_t acc1 = tmem + static_cast<uint32_t>(p.acc1_col[b]);
                for (int s = 0; s < nslab; ++s) {
                    const int ksteps = min(4, (p.hcw[j] >> 4) - 4 * s);
                    trace_ev<TRACE>(p.trace, 3, it, 2 * j + s, 0);
                    mbar_wait(&bars->h_ready[b][s], acc1_phase(cg));
                    // the accumulator is free: plain -- the last epilogue has read the previous tile's; folded adjust -- the aux warps
                    // have read tile it - 2 (if the fc1 issuer takes the y term, it has waited for that and issued it already)
                    if (j == 0 && s == 0 && !(p.fuse_adj && p.adjy_fc1)) {
                        mbar_wait(&bars->acc2_free[acc2_buf(it)], acc2_phase(it) ^ 1);
                        if (p.fuse_adj) {
                            if (it == 0) mbar_wait(&bars->adj_w_full, 0);
                            mbar_wait(&bars->a_full[it & 1], static_cast<uint32_t>(it >> 1) & 1);
                            issue_adj_y(it);
                            if (elect_one_sync()) umma_commit(&bars->adj_done[it & 1]);
                            __syncwarp();
                        }
                        if (p.fold_res) mbar_wait(&bars->a_full[it & 1], static_cast<uint32_t>(it >> 1) & 1);
                    }
                    if (p.fold_res && s == 0) {
                        // wide folded conv: acc2 also takes y W_a^T -- the ring brings W_a as (K slab, N piece) slabs, the y panels are
                        // the (shared-memory) A operand; p.ypre[j] of them are issued in front of chunk j (see the launcher)
                        const uint64_t ya_desc = umma_desc_k_sw128(smem_u32(a_buf)) + static_cast<uint64_t>((it & 1) * static_cast<uint32_t>(p.a_buf_bytes >> 4));
                        for (int q = 0; q < p.ypre[j]; ++q, ++yq) {
                            const int ys = yq / p.n_pieces, pc = yq - ys * p.n_pieces;
                            const int yk = min(4, p.k1steps - 4 * ys);
                            const uint32_t idesc = umma_idesc_bf16_m128(static_cast<uint32_t>(p.piece_rows[pc]));
                            const uint32_t d = tmem + static_cast<uint32_t>(p.piece_col[pc]);
                            mbar_wait(&bars->w2_full[slot], phase);
                            tc_fence_after_sync();
                            if (elect_one_sync()) {
                                const uint64_t adesc = ya_desc + static_cast<uint64_t>(ys * (kPanelBytes >> 4));
                                const uint64_t bdesc = ring_desc + static_cast<uint64_t>(static_cast<uint32_t>(slot) * slot_units);
                                umma_bf16(d, adesc, bdesc, idesc, (acc2_started >> pc) & 1u);
                                if (yk > 1) umma_bf16(d, adesc + 2, bdesc + 2, idesc, 1u);
                                if (yk > 2) umma_bf16(d, adesc + 4, bdesc + 4, idesc, 1u);
                                if (yk > 3) umma_bf16(d, adesc + 6, bdesc + 6, idesc, 1u);
                                umma_commit(&bars->w2_empty[slot]);
                                if (yq == p.ks1 * p.n_pieces - 1) umma_commit(&bars->adj_done[it & 1]);   // my last read of the y tile
                            }
                            __syncwarp();
                            acc2_started |= 1u << pc;
                            if (++slot == p.w2_slots) { slot = 0; phase ^= 1; }
                        }
                    }
                    trace_ev<TRACE>(p.trace, 3, it, 2 * j + s, 1);
                    const uint32_t at = acc1 + static_cast<uint32_t>(64 * s);     // K=16 step u of the chunk lives at column 16 u
                    const uint32_t first_acc = (j == 0 && s == 0 && !p.fuse_adj) ? 0u : 1u;   // (fold_res: per N piece, acc2_started)
                    for (int pc = 0; pc < p.n_pieces; ++pc) {
                        const uint32_t idesc = umma_idesc_bf16_m128(static_cast<uint32_t>(p.piece_rows[pc]));
                        const uint32_t d = tmem + static_cast<uint32_t>(p.piece_col[pc] + 32 * acc2_buf(it));
                        mbar_wait(&bars->w2_full[slot], phase);
                        trace_ev<TRACE>(p.trace, 3, it, 2 * j + s, 5);
                        tc_fence_after_sync();
                        if (elect_one_sync()) {
                            const uint64_t bdesc = ring_desc + static_cast<uint64_t>(static_cast<uint32_t>(slot) * slot_units);
                            umma_bf16_ts(d, at, bdesc, idesc, p.fold_res ? ((acc2_started >> pc) & 1u) : first_acc);
                            if (ksteps > 1) umma_bf16_ts(d, at + 16, bdesc + 2, idesc, 1u);
                            if (ksteps > 2) umma_bf16_ts(d, at + 32, bdesc + 4, idesc, 1u);
                            if (ksteps > 3) umma_bf16_ts(d, at + 48, bdesc + 6, idesc, 1u);
                            umma_commit(&bars->w2_empty[slot]);
                            if (s == nslab - 1 && pc == p.n_pieces - 1) {
                                umma_commit(&bars->acc1_free[b]);                  // chunk accumulator may be overwritten
                                if (j == p.nc - 1) umma_commit(&bars->acc2_full[acc2_buf(it)]);  // tile complete -> last epilogue
                            }
                        }
                        __syncwarp();
                        acc2_started |= 1u << pc;
                        if (++slot == p.w2_slots) { slot = 0; phase ^= 1; }
                    }
                    trace_ev<TRACE>(p.trace, 3, it, 2 * j + s, 2);
                }
            }
        }
    } else if (warp < kEpiWarps) {
        // ============================================================ epilogue: 4 quadrants (TMEM lanes) x 4 column groups
        const int quad = warp & 3;
        const int grp = warp >> 2;
        const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
        const int r_in_tile = quad * 32 + lane;
        const uint32_t row_off = static_cast<uint32_t>(r_in_tile * 128);
        const int rsw = r_in_tile & 7;
        const bool tr = TRACE && warp == 0;

        // (rstd, -mean * rstd) of the tile's rows, produced two tiles ahead by the aux warps (the (sum, sumsq) slots were written by
        // the previous kernel: fetched cold here they cost ~2k cycles of exposed latency per tile on the clock64 timeline)
        auto row_stats = [&](int it, float& rstd, float& nrm) {
            mbar_wait(&bars->rs_full[it & 1], static_cast<uint32_t>(it >> 1) & 1);
            const float2 v = s_rowstat[(it & 1) * 128 + r_in_tile];
            rstd = v.x;
            nrm = v.y;
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->rs_free[it & 1]);
        };

        // ---- one hidden chunk: TMEM fp32 -> LN fold + bias + GELU -> bf16 into the first 8 columns of each 16-column unit
        auto epi1 = [&](int it, int j, float rstd, float nrm) {
            const int cg = it * p.nc + j;
            const int b = acc1_buf(cg);
            const int units = p.hcw[j] >> 4;                          // K=16 steps of fc2 in this chunk
            const uint32_t taddr = tmem + static_cast<uint32_t>(p.acc1_col[b]) + lane_off;
            const float2 rstd2 = f2(rstd, rstd), nrm2 = f2(nrm, nrm);
            if (tr) trace_ev<TRACE>(p.trace, 2, it, j, 0);
            mbar_wait(&bars->acc1_full[b], acc1_phase(cg));
            tc_fence_after_sync();
            if (tr) trace_ev<TRACE>(p.trace, 2, it, j, 1);
            // 16 accumulator columns -> 8 packed bf16x2 GELU activations
            auto convert16 = [&](const uint32_t (&raw)[16], int u, uint32_t (&pk)[8]) {
                const float* bp = s_bias1 + j * p.hc + 16 * u;
                const float* cp = s_colsum1 + j * p.hc + 16 * u;
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) {
                    const float4 bb = *reinterpret_cast<const float4*>(bp + 4 * q4);
                    const float4 cs = *reinterpret_cast<const float4*>(cp + 4 * q4);
                    const float2 x0 = __ffma2_rn(rstd2, f2(__uint_as_float(raw[4 * q4]), __uint_as_float(raw[4 * q4 + 1])),
                                                 __ffma2_rn(nrm2, f2(cs.x, cs.y), f2(bb.x, bb.y)));
                    const float2 x1 = __ffma2_rn(rstd2, f2(__uint_as_float(raw[4 * q4 + 2]), __uint_as_float(raw[4 * q4 + 3])),
                                                 __ffma2_rn(nrm2, f2(cs.z, cs.w), f2(bb.z, bb.w)));
                    const float2 g0 = gelu2_pair(x0), g1 = gelu2_pair(x1);
                    pk[2 * q4] = pack_bf16x2(g0.x, g0.y);
                    pk[2 * q4 + 1] = pack_bf16x2(g1.x, g1.y);
                }
            };
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {                             // h = 64-column slab of the chunk
                const int u = grp + 4 * h;
                if (u < units) {
                    uint32_t raw[16], pk[8];
                    tmem_ld16(taddr + static_cast<uint32_t>(16 * u), raw);
                    tmem_ld_wait();
                    convert16(raw, u, pk);
                    tmem_st8(taddr + static_cast<uint32_t>(16 * u), pk);
                    tmem_st_wait();
                }
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->h_ready[b][h]);
                if (tr) trace_ev<TRACE>(p.trace, 2, it, j, 2 + h);
            }
        };

        // ---- fc2: + bias + residual (the y tile in shared memory), written back in place as z
        auto epi2 = [&](int it) {
            const int ab = it & 1;
            const int units = p.n2 >> 4;
            const uint32_t a_row = smem_u32(a_buf + ab * p.a_buf_bytes) + row_off;
            const uint32_t taddr = tmem + lane_off;
            if (tr) trace_ev<TRACE>(p.trace, 2, it, 16, 0);
            // the residual: the y tile itself, or (fold_res) the tile of the residual tensor that replaced it -- TMA-written, visible to me
            mbar_wait(p.fold_res ? &bars->res_full[ab] : &bars->a_full[ab], static_cast<uint32_t>(it >> 1) & 1);
            mbar_wait(&bars->acc2_full[0], static_cast<uint32_t>(it) & 1);
            float2 ost = f2(0.f, 0.f), osq = f2(0.f, 0.f);                       // fold_res: (sum, sumsq) of my columns of the output row
            tc_fence_after_sync();
            if (tr) trace_ev<TRACE>(p.trace, 2, it, 16, 1);
#pragma unroll 1
            for (int u = grp; u < units; u += 4) {
                uint32_t raw[16];
                tmem_ld16(taddr + static_cast<uint32_t>(16 * u), raw);
                uint32_t rw[2][4];
                uint32_t saddr[2];
#pragma unroll
                for (int o = 0; o < 2; ++o) {                         // 8 columns = one 16-byte chunk of the swizzled row
                    const int c = 16 * u + 8 * o;
                    saddr[o] = a_row + static_cast<uint32_t>((c >> 6) * kPanelBytes) + static_cast<uint32_t>((((c >> 3) & 7) ^ rsw) << 4);
                    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(rw[o][0]), "=r"(rw[o][1]), "=r"(rw[o][2]), "=r"(rw[o][3])
                                 : "r"(saddr[o]));
                }
                tmem_ld_wait();
#pragma unroll
                for (int o = 0; o < 2; ++o) {
                    const int c = 16 * u + 8 * o;
                    const float4 b0 = *reinterpret_cast<const float4*>(s_bias2 + c);
                    const float4 b1 = *reinterpret_cast<const float4*>(s_bias2 + c + 4);
                    const uint32_t* a8 = &raw[8 * o];
                    const float2 v0 = __fadd2_rn(__fadd2_rn(f2(__uint_as_float(a8[0]), __uint_as_float(a8[1])), f2(b0.x, b0.y)),
                                                 f2(bf16_lo(rw[o][0]), bf16_hi(rw[o][0])));
                    const float2 v1 = __fadd2_rn(__fadd2_rn(f2(__uint_as_float(a8[2]), __uint_as_float(a8[3])), f2(b0.z, b0.w)),
                                                 f2(bf16_lo(rw[o][1]), bf16_hi(rw[o][1])));
                    const float2 v2 = __fadd2_rn(__fadd2_rn(f2(__uint_as_float(a8[4]), __uint_as_float(a8[5])), f2(b1.x, b1.y)),
                                                 f2(bf16_lo(rw[o][2]), bf16_hi(rw[o][2])));
                    const float2 v3 = __fadd2_rn(__fadd2_rn(f2(__uint_as_float(a8[6]), __uint_as_float(a8[7])), f2(b1.z, b1.w)),
                                                 f2(bf16_lo(rw[o][3]), bf16_hi(rw[o][3])));
                    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(saddr[o]), "r"(pack_bf16x2(v0.x, v0.y)),
                                 "r"(pack_bf16x2(v1.x, v1.y)), "r"(pack_bf16x2(v2.x, v2.y)), "r"(pack_bf16x2(v3.x, v3.y))
                                 : "memory");
                    if (p.fold_res) {      // pad columns: zero weights, zero bias, zero-filled residual -> exact zeros, no effect on the sums
                        ost = __fadd2_rn(ost, __fadd2_rn(__fadd2_rn(v0, v1), __fadd2_rn(v2, v3)));
                        osq = __ffma2_rn(v0, v0, osq);
                        osq = __ffma2_rn(v1, v1, osq);
                        osq = __ffma2_rn(v2, v2, osq);
                        osq = __ffma2_rn(v3, v3, osq);
                    }
                }
            }
            if (p.fold_res && p.adj_stats != nullptr) {
                // the row's (sum, sumsq): each of the four column groups leaves its partial in a slot of its own (the LayerNorm fold
                // of the consumer adds the slots up anyway) -- no exchange through shared memory, no barrier
                const int row = tile_of(it) * 128 + r_in_tile;
                if (row < p.M)
                    p.adj_stats[static_cast<long long>(row) * p.adj_stats_stride + p.adj_stats_slot0 + grp] = f2(ost.x + ost.y, osq.x + osq.y);
            }
            tc_fence_before_sync();
            fence_proxy_async_smem();                                  // my st.shared -> visible to the TMA store
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&bars->acc2_free[0]);
                mbar_arrive(&bars->z_ready[ab]);
            }
            if (tr) trace_ev<TRACE>(p.trace, 2, it, 16, 2);
        };

        // task order mirrors the MMA streams: chunk 0 of tile it+1 is turned around BEFORE the last epilogue of tile it
        // (fc1 runs ahead of fc2, so that chunk is ready while the last fc2 MMAs of tile it are still in flight)
        float rstd = 1.f, nrm = 0.f;
        if (my_tiles > 0) {
            row_stats(0, rstd, nrm);
            epi1(0, 0, rstd, nrm);
        }
        for (int it = 0; it < my_tiles; ++it) {
            for (int j = 1; j < p.nc; ++j) epi1(it, j, rstd, nrm);
            if (it + 1 < my_tiles) {
                row_stats(it + 1, rstd, nrm);
                epi1(it + 1, 0, rstd, nrm);
            }
            if (!p.fuse_adj) epi2(it);                                // folded adjust: no z, no residual pass (the aux warps finish the tile)
        }
    } else if (warp >= kAuxWarp0) {
        // ============================================================ aux warps, one per TMEM lane quadrant (thread = row of the tile):
        //  * LayerNorm row statistics: (sum, sumsq) slots -> (rstd, -mean * rstd) in shared memory, up to two tiles ahead;
        //  * folded adjust: 32 new slab columns = LReLU(acc + bias), stored at the tile's token rows, + their row statistics.  A
        //    thread holds a whole row (32 columns), so its (sum, sumsq) never leaves the thread; the 16 conversion warps never
        //    stop for this.
        const int quad = warp & 3;
        const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
        const int r_in_tile = quad * 32 + lane;
        auto produce_stats = [&](int it) {
            const int row = tile_of(it) * 128 + r_in_tile;
            float rstd = 1.f, nrm = 0.f;                              // nrm = -mean * rstd
            if (row < p.M) {
                const float2* sp = p.stats_in + static_cast<long long>(row) * p.stats_in_stride;
                float s1 = 0.f, s2 = 0.f;
                for (int k = 0; k < p.stats_in_slots; ++k) {
                    const float2 v = __ldg(sp + k);
                    s1 += v.x;
                    s2 += v.y;
                }
                const float mean = s1 * p.inv_c;
                rstd = rsqrtf(fmaxf(s2 * p.inv_c - mean * mean, 0.f) + p.ln_eps);
                nrm = -mean * rstd;
            }
            mbar_wait(&bars->rs_free[it & 1], (static_cast<uint32_t>(it >> 1) & 1) ^ 1);
            s_rowstat[(it & 1) * 128 + r_in_tile] = f2(rstd, nrm);
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->rs_full[it & 1]);
        };
        // ---- warp 20 only: y-tile loads / z-tile stores (same buffers)
        const bool tile_warp = warp == kTileWarp;
        auto load_a = [&](int it) {
            const int ab = it & 1;
            const int m0 = tile_of(it) * 128;
            if (lane == 0) {
                mbar_arrive_expect_tx(&bars->a_full[ab], static_cast<uint32_t>(p.a_buf_bytes));
                for (int pn = 0; pn < p.ks1; ++pn)
                    tma_load_2d(a_buf + ab * p.a_buf_bytes + pn * kPanelBytes, &p.tmap_y, pn * 64, m0, &bars->a_full[ab]);
            }
            __syncwarp();
        };
        if (tile_warp) {
            if (lane == 0) tma_prefetch_desc(&p.tmap_y);
            if (p.fuse_adj && lane == 0) {
                mbar_arrive_expect_tx(&bars->adj_w_full, static_cast<uint32_t>(p.ks1 * kAdjSlabBytes));
                bulk_g2s(wadj_s, p.wadj, static_cast<uint32_t>(p.ks1 * kAdjSlabBytes), &bars->adj_w_full);
            }
            if (my_tiles > 0) load_a(0);
            if (my_tiles > 1) load_a(1);
        }
        if (my_tiles > 0) produce_stats(0);
        if (my_tiles > 1) produce_stats(1);
        for (int it = 0; it < my_tiles; ++it) {
            if (it + 2 < my_tiles) produce_stats(it + 2);             // its buffer was released when tile it started
            if (tile_warp) {
                // the tile buffer is free again -- folded adjust: fc1 and the y W_adj^T MMAs have read it (nothing is stored);
                // plain: the last epilogue has turned it into z, which leaves by TMA -- fetch the tile after next
                const int ab = it & 1;
                trace_ev<TRACE>(p.trace, 0, it, 0, 0);
                if (p.fuse_adj) {
                    mbar_wait(&bars->adj_done[ab], static_cast<uint32_t>(it >> 1) & 1);
                } else {
                    const int zpan = p.fold_res ? (p.n2 + 63) >> 6 : p.ks1;     // 64-column panels of the output tile
                    if (p.fold_res) {
                        // fc1 and the y W_a^T MMAs have read the y tile: the residual tile takes its place (same panel layout; columns
                        // >= c_out are zero-filled by the tensor map), the last epilogue adds it and leaves the output in place
                        mbar_wait(&bars->adj_done[ab], static_cast<uint32_t>(it >> 1) & 1);
                        if (lane == 0) {
                            mbar_arrive_expect_tx(&bars->res_full[ab], static_cast<uint32_t>(zpan * kPanelBytes));
                            for (int pn = 0; pn < zpan; ++pn)
                                tma_load_2d(a_buf + ab * p.a_buf_bytes + pn * kPanelBytes, &p.tmap_res, pn * 64, tile_of(it) * 128, &bars->res_full[ab]);
                        }
                        __syncwarp();
                    }
                    mbar_wait(&bars->z_ready[ab], static_cast<uint32_t>(it >> 1) & 1);
                    trace_ev<TRACE>(p.trace, 0, it, 0, 1);
                    if (lane == 0) {    // bulk-group bookkeeping is per thread: the same lane stores and waits
                        for (int pn = 0; pn < zpan; ++pn)
                            tma_store_2d_box(&p.tmap_z, a_buf + ab * p.a_buf_bytes + pn * kPanelBytes, pn * 64, tile_of(it) * 128);
                        bulk_commit_group();
                        bulk_wait_group_read0();
                    }
                    __syncwarp();
                }
                trace_ev<TRACE>(p.trace, 0, it, 0, 2);
                if (it + 2 < my_tiles) load_a(it + 2);
                trace_ev<TRACE>(p.trace, 0, it, 0, 3);
            }
            if (!p.fuse_adj) continue;
            const int row = tile_of(it) * 128 + r_in_tile;
            mbar_wait(&bars->acc2_full[it & 1], acc2_phase(it));
            tc_fence_after_sync();
            uint32_t raw[32];
            const uint32_t acc2 = tmem + lane_off + static_cast<uint32_t>(p.piece_col[0] + 32 * (it & 1));
            tmem_ld16(acc2, *reinterpret_cast<uint32_t(*)[16]>(&raw[0]));
            tmem_ld16(acc2 + 16, *reinterpret_cast<uint32_t(*)[16]>(&raw[16]));
            tmem_ld_wait();
            tc_fence_before_sync();                                   // the next tile's MMAs may overwrite the accumulator
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->acc2_free[it & 1]);
            float st = 0.f, sq = 0.f;
            uint32_t pk[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                const float2 bb = *reinterpret_cast<const float2*>(s_bias2 + 2 * e);
                float v0 = __uint_as_float(raw[2 * e]) + bb.x;
                float v1 = __uint_as_float(raw[2 * e + 1]) + bb.y;
                v0 = v0 > 0.f ? v0 : v0 * p.adj_slope;
                v1 = v1 > 0.f ? v1 : v1 * p.adj_slope;
                st += v0 + v1;
                sq = fmaf(v0, v0, fmaf(v1, v1, sq));
                pk[e] = pack_bf16x2(v0, v1);
            }
            // Row-per-thread stores of the slice (8-byte pieces at a 640-byte pitch: 32 sectors per instruction) cost the conversion
            // warps ~10 % -- they share the load/store path (A/B with the stores removed).  The slice starts at column C_k, which
            // is 8 but not 16 bytes aligned, so a TMA box cannot take it; the rows are transposed through a (swizzled) staging box
            // instead and leave as 64 contiguous bytes per 8 lanes.
            __syncwarp();                                             // the previous tile's box has been read out
            const uint32_t sbox = smem_u32(adj_stage + quad * 2048);
            {
                const uint32_t srow = sbox + static_cast<uint32_t>(lane * 64);
                const uint32_t sw = static_cast<uint32_t>(lane >> 1) & 3u;
#pragma unroll
                for (uint32_t c = 0; c < 4; ++c)
                    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(srow + ((c ^ sw) << 4)), "r"(pk[4 * c]), "r"(pk[4 * c + 1]),
                                 "r"(pk[4 * c + 2]), "r"(pk[4 * c + 3])
                                 : "memory");
            }
            __syncwarp();
            {
                const uint32_t q = static_cast<uint32_t>(lane) & 7u;  // 8-byte piece of the row
                const int row0 = tile_of(it) * 128 + quad * 32;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint32_t r = static_cast<uint32_t>(4 * k + (lane >> 3));
                    uint32_t v0, v1;
                    asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];"
                                 : "=r"(v0), "=r"(v1)
                                 : "r"(sbox + r * 64u + (((q >> 1) ^ ((r >> 1) & 3u)) << 4) + ((q & 1u) << 3)));
                    if (row0 + static_cast<int>(r) < p.M)
                        *reinterpret_cast<uint2*>(p.adj_out + static_cast<long long>(row0 + static_cast<int>(r)) * p.ld_adj + p.adj_col0 + 4 * q) =
                            make_uint2(v0, v1);
                }
            }
            if (row < p.M && p.adj_stats != nullptr) {
                float2* so = p.adj_stats + static_cast<long long>(row) * p.adj_stats_stride + p.adj_stats_slot0;
                if (p.adj_stats_vec4) {
                    *reinterpret_cast<float4*>(so) = make_float4(st, sq, 0.f, 0.f);
                } else {
                    so[0] = f2(st, sq);
                    so[1] = f2(0.f, 0.f);
                }
            }
        }
        if (tile_warp && lane == 0) bulk_wait_group0();
        __syncwarp();
    }

    tc_fence_before_sync();
    __syncthreads();
    if (warp == kTileWarp) {
        tc_fence_after_sync();
        tmem_dealloc<512>(tmem);
    }
}

}  // namespace

int launch_swin_mlp(SwinMlpParams& p, const void* y, long long ldy, void* z, long long ldz, int num_sms, cudaStream_t stream) {
    if (p.M <= 0) return ADSR_OK;
    if (p.nc <= 0 || p.nc > 8 || p.n_pieces < 1 || p.n_pieces > 2) return ADSR_ERR_BAD_SHAPE;
    if (p.n2 > kMaxN2 || (p.n2 % 16) != 0 || p.nc * p.hc > kMaxHidden || (p.hc % 16) != 0) return ADSR_ERR_BAD_SHAPE;
    if (p.n2 + 2 * p.hc > 512 || p.acc1_col[0] < (p.fuse_adj ? 2 : 1) * p.n2 || p.acc1_col[1] < p.acc1_col[0] + p.hc || p.acc1_col[1] + p.hc > 512)
        return ADSR_ERR_BAD_SHAPE;
    p.acc1_col[2] = p.acc1_col[1] + p.hc;
    p.n_acc1 = p.acc1_col[2] + p.hc <= 512 ? 3 : 2;
    if (p.ks1 <= 0 || p.ks1 > 5 || p.k1steps <= 4 * (p.ks1 - 1) || p.k1steps > 4 * p.ks1) return ADSR_ERR_BAD_SHAPE;
    if (p.w1_slots < 2 || p.w1_slots > 8 || p.w2_slots < 2 || p.w2_slots > 8 || (p.w1_slot_bytes % 1024) || (p.w2_slot_bytes % 1024))
        return ADSR_ERR_BAD_SHAPE;
    int col = 0;
    for (int pc = 0; pc < p.n_pieces; ++pc) {
        if (p.piece_rows[pc] < 16 || p.piece_rows[pc] > 256 || (p.piece_rows[pc] % 16) || p.piece_col[pc] != col ||
            p.piece_rows[pc] * 128 > p.w2_slot_bytes)
            return ADSR_ERR_BAD_SHAPE;
        col += p.piece_rows[pc];
    }
    if (col != p.n2) return ADSR_ERR_BAD_SHAPE;
    for (int j = 0; j < p.nc; ++j)
        if (p.hcw[j] <= 0 || p.hcw[j] > p.hc || p.hcw[j] > 128 || (p.hcw[j] % 16) != 0 || p.hcw[j] * 128 > p.w1_slot_bytes)
            return ADSR_ERR_BAD_SHAPE;
    p.a_buf_bytes = p.ks1 * kPanelBytes;
    p.inv_c = 1.0f / static_cast<float>(p.C);
    p.adjy_fc1 = p.ks1 <= 3 ? 1 : 0;
    if (p.fuse_adj) {
        if (p.wadj == nullptr || p.bias_adj == nullptr || p.adj_out == nullptr || (p.adj_col0 % 4) || (p.ld_adj % 4) ||
            (reinterpret_cast<uintptr_t>(p.wadj) & 15) || (reinterpret_cast<uintptr_t>(p.adj_out) & 7))
            return ADSR_ERR_BAD_SHAPE;
        if (p.n2 != 32 || p.n_pieces != 1) return ADSR_ERR_BAD_SHAPE;       // the accumulator IS the 32 adjust columns
        if (p.adj_stats != nullptr && p.adj_stats_slot0 + 2 > p.adj_stats_stride) return ADSR_ERR_BAD_SHAPE;
        p.adj_stats_vec4 = ((p.adj_stats_slot0 | p.adj_stats_stride) & 1) == 0 && (reinterpret_cast<uintptr_t>(p.adj_stats) & 15) == 0;
    }
    if (p.fold_res) {
        // wide folded conv with residual: out[:, :c_out] = res[:, :c_out] + y W_a^T + g (W_a W2)^T + bias; the output tile (n2 columns)
        // takes the place of the y tile, so it must fit its panels
        if (p.fuse_adj || p.res == nullptr || p.c_out <= 0 || p.n2 != (p.c_out + 15) / 16 * 16 || (p.n2 + 63) / 64 > p.ks1 ||
            p.ld_res < p.c_out || ldz < p.c_out)
            return ADSR_ERR_BAD_SHAPE;
        if ((reinterpret_cast<uintptr_t>(p.res) & 15) || (p.ld_res % 8)) return ADSR_ERR_BAD_ALIGN;
        if (p.adj_stats != nullptr && p.adj_stats_slot0 + 4 > p.adj_stats_stride) return ADSR_ERR_BAD_SHAPE;   // four partial slots
        // where the ks1 * n_pieces slabs of W_a go in the fc2 stream (pack.pack_swin_mlp_conv_res lays it out by the same rule): all in
        // front of chunk 0.  Spreading them evenly over the chunks was measured SLOWER (188 vs 177 us at C = 308): with ~56 KB of ring
        // in flight next to two 80 KB tile buffers both rings are L2-latency bound, and the fc2 issuer then paces the whole tile
        const int ytot = p.ks1 * p.n_pieces;
        for (int j = 0; j < 8; ++j) p.ypre[j] = j == 0 ? ytot : 0;
    }
    const int smem_bytes = 2 * p.a_buf_bytes + p.w1_slots * p.w1_slot_bytes + p.w2_slots * p.w2_slot_bytes + const_bytes(p.nc * p.hc, p.n2) +
                           (p.fuse_adj ? p.ks1 * kAdjSlabBytes + kAdjStageBytes : 0) +
                           static_cast<int>(sizeof(MlpBarriers));
    if (smem_bytes > kSmemLimit) return ADSR_ERR_BAD_SHAPE;
    if ((reinterpret_cast<uintptr_t>(y) & 15) || (!p.fuse_adj && ((reinterpret_cast<uintptr_t>(z) & 15) || (ldz % 8))) || (ldy % 8) ||
        (reinterpret_cast<uintptr_t>(p.w1p) & 15) || (reinterpret_cast<uintptr_t>(p.w2p) & 15))
        return ADSR_ERR_BAD_ALIGN;
    int st = encode_tmap_rows_bf16(&p.tmap_y, y, p.M, p.C, ldy);
    if (st != ADSR_OK) return st;
    if (!p.fuse_adj) {
        st = encode_tmap_rows_bf16(&p.tmap_z, z, p.M, p.fold_res ? p.c_out : p.C, ldz);
        if (st != ADSR_OK) return st;
    }
    if (p.fold_res) {
        st = encode_tmap_rows_bf16(&p.tmap_res, p.res, p.M, p.c_out, p.ld_res);
        if (st != ADSR_OK) return st;
    }
    p.m_tiles = (p.M + 127) / 128;
    const int grid = p.m_tiles < num_sms ? p.m_tiles : num_sms;
    auto launch = [&](auto kernel) -> int {
        if (ensure_dynamic_smem(kernel, smem_bytes) != cudaSuccess) return ADSR_ERR_CUDA;
        return launch_pdl(kernel, dim3(grid), dim3(kThreads), static_cast<size_t>(smem_bytes), stream, p) == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
    };
    return p.trace != nullptr ? launch(swin_mlp_kernel<true>) : launch(swin_mlp_kernel<false>);
}

int swin_mlp_fixed_smem_bytes(int hidden_padded, int n2) { return const_bytes(hidden_padded, n2) + static_cast<int>(sizeof(MlpBarriers)); }

}  // namespace adsr
