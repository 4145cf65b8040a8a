// Fused attention half of a Swin block for sm_100a (8 x 8 windows, the DRCT-L shape):
//     y = x + proj( WindowAttention( LayerNorm(x) ) )                               (src/drct.py:478-509, 271-302)
// i.e. norm1 (folded) -> qkv Linear -> cyclic shift + window_partition -> softmax(q k^T * scale + rel-pos bias + mask) v
// -> window_reverse + un-shift -> proj Linear -> + shortcut, in ONE persistent warp-specialised kernel.  Neither the
// q|k|v rows (1.1 - 1.9 KB per token) nor the attention output ever touch HBM.
//
// A CTA owns one TILE = two consecutive windows = 128 token rows and walks over the heads:
//   * the loader warp fetches the raw x rows of the tile with 4-D TMA boxes of [R x R tokens x 64 channels] (R = 8: a whole
//     window; R = 4 when the cyclic shift makes windows wrap; closed-form index map of src/drct.py:483, 193-204) into
//     K-major 128-byte-swizzled panels (A operand of qkv); channels >= C are zero-filled by the tensor map;
//   * per head h the MMA warp computes  [q_h | k_h | v_h] = x W_h^T  (tcgen05.mma SS, N = 3 hdp) into a TMEM region (two
//     alternating regions when proj is not fused: the next head's q|k|v then runs one head ahead); the weights stream
//     from L2 through a ring of whole [3 hdp x 64] qkv slabs and a one-head-deep proj ring, each fed by its own loader warp;
//   * 16 epilogue warps apply the folded LayerNorm + bias and write q back IN PLACE into TMEM as bf16 (A operand of S), k and
//     v as bf16 into shared-memory operand panels;
//   * S = q k^T (tcgen05.mma TS, M = N = 128; the off-diagonal 64 x 64 blocks belong to the other window and are never
//     used) lands on the dead k|v accumulator columns of the region; softmax: four threads per query row, relative-position
//     bias from a shared-memory table, -100 mask from closed-form region ids (src/drct.py:449-470); unnormalised bf16
//     probabilities go back in place into TMEM;  O = P v  (TS, v as MN-major B operand) lands on the dead q columns;
//   * fuse_proj (padded heads <= 64): a persistent TMEM accumulator Y is initialised with the SHORTCUT by identity MMAs
//     (Y = x I, N = 16, straight from the resident x tile: bf16 values enter fp32 exactly); the normalised O_h is written back
//     in place as bf16 and  Y += O_h Wp_h^T  (TS) accumulates the proj Linear over the heads; the last epilogue adds the bias,
//     stages y through the idle k / v panels (coalesced 128-byte row pieces) to the ORIGINAL token rows (window_reverse +
//     un-shift are the inverse permutation) and leaves the per-row (sum, sumsq) for the norm2 fold of the MLP kernel.  Where
//     TMEM has room (the narrowest block) q|k|v has accumulator columns of its own and the next head's q|k|v is issued right
//     after S.  Otherwise (heads of 80 / 128 padded channels: TMEM cannot hold everything) two TMEM regions alternate so that
//     the next head's q|k|v runs one head ahead, the normalised O rows go through the k panel to `out` [M, nH * hdp] and the
//     row-tile GEMM applies proj.
// Single-warp issue loops are latency chains: nothing on them divides by a run-time value (one modulo per head cost 3 %).
#include "adsr_kernels.h"
#include "ptx.cuh"

namespace adsr {

namespace {

constexpr int kEpiWarps = 16;                 // warps 0..15: quadrant (TMEM lanes) = warp & 3, column group = warp >> 2
constexpr int kXLoaderWarp = 16;              // x-tile TMA loads
constexpr int kMmaWarp = 17;
constexpr int kWLoaderWarp = 18;              // qkv weight slabs, TMEM alloc
constexpr int kPLoaderWarp = 19;              // proj weight slabs
constexpr int kThreads = 20 * 32;
constexpr int kPanelBytes = 128 * 128;
constexpr int kMaxSlots = 10;
constexpr int kSmemLimit = 232448;
constexpr int kIdentBytes = 16 * 128;         // fuse_proj: identity operand slab (16 rows x 64 bf16, 128-byte swizzle)

struct __align__(8) AttnBlockBarriers {
    uint64_t w_full[kMaxSlots], w_empty[kMaxSlots];
    uint64_t p_full[4], p_empty[4];
    uint64_t x_full, x_empty;
    uint64_t qkv_full[2];                     // per TMEM region
    uint64_t qkv_ready, s_full, p_ready, o_full, o_ready;
    uint64_t proj_full, proj_free;
    uint32_t tmem_base;
};

__device__ __forceinline__ uint64_t desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
__device__ __forceinline__ uint32_t idesc_m128(uint32_t n, uint32_t b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (b_mn_major << 16) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void* src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit_() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tmem_st8_(uint32_t taddr, const uint32_t* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
                 "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st8_zero_(uint32_t taddr) {
    const uint32_t z = 0u;
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"r"(taddr), "r"(z) : "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ int region_1d_(int t, int L, int shift) { return (t >= L - 8 ? 1 : 0) + (t >= L - shift ? 1 : 0); }
__device__ __forceinline__ float2 f2_(float a, float b) { return make_float2(a, b); }

// optional timeline of CTA 0 (tools/attn_trace.py): trace[(((role * 4 + tile) * 9 + head) * 8 + k)] = clock64()
// roles: 0 = MMA warp, 1 = epilogue warp 0, 2 = x loader warp; head slot 8 = per-tile events
template <bool TRACE>
__device__ __forceinline__ void tr_ev(long long* trace, int role, int it, int h, int k) {
    if constexpr (TRACE) {
        if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && it < 4) trace[((role * 4 + it) * 9 + h) * 8 + k] = clock64();
    }
}

template <bool TRACE, bool FUSE>
__global__ void __launch_bounds__(kThreads, 1) swin_attn_kernel(const __grid_constant__ SwinAttnParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int x_bytes = p.ks * kPanelBytes;
    const int op_bytes = p.pan * kPanelBytes;
    const int nqkv = p.nH * 3 * p.hdp;
    uint8_t* x_buf = smem;                                             // [ks panels] raw x rows of the tile (A operand of qkv)
    uint8_t* k_buf = x_buf + x_bytes;                                  // [pan panels] k of the current head (K-major B operand of S)
    uint8_t* v_buf = k_buf + op_bytes;                                 // [pan panels] v of the current head (MN-major B operand of P V)
    uint8_t* ring = v_buf + op_bytes * (p.pipe ? 2 : 1);               // qkv slabs: w_slots x w_slot_bytes (pipe: the v panel alternates)
    uint8_t* pring = ring + p.w_slots * p.w_slot_bytes;                // proj slabs: p_slots x p_slot_bytes
    uint8_t* ident_s = pring + p.p_slots * p.p_slot_bytes;             // FUSE: [16 x 64] bf16 operand slab holding the 16 x 16 identity
    float* s_bq = reinterpret_cast<float*>(ident_s + (FUSE ? kIdentBytes : 0));     // [nqkv] folded qkv bias, per-head q|k|v order
    float* s_cq = s_bq + nqkv;                                         // [nqkv] column sums of the gamma-folded weights
    float* s_bp = s_cq + nqkv;                                         // [cp] proj bias
    float* s_bias = s_bp + p.cp;                                       // [nH][232] rel-pos table * log2(e)
    int* s_tok = reinterpret_cast<int*>(s_bias + p.nH * 232);          // [2][128] token row of each tile row
    float* s_max = reinterpret_cast<float*>(s_tok + 256);              // [4][128] partial row maxima
    float* s_sum = s_max + 512;                                        // [2][4][128] partial row sums, by head parity (pipe: a warp may be in
                                                                       // the next head's softmax while another still normalises this one)
    float2* s_stat = reinterpret_cast<float2*>(s_max);                 // [4][128] (sum, sumsq) partials of y -- aliases s_max | s_sum[0]
    AttnBlockBarriers* bars = reinterpret_cast<AttnBlockBarriers*>(s_sum + 1024);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int my_tiles = static_cast<int>(blockIdx.x) < p.n_tiles ? (p.n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if ((smem_u32(smem) & 1023u) != 0) __trap();
    for (int i = threadIdx.x; i < nqkv; i += kThreads) {
        s_bq[i] = p.bias_qkv[i];
        s_cq[i] = p.colsum_qkv[i];
    }
    if (FUSE)
        for (int i = threadIdx.x; i < p.cp; i += kThreads) s_bp[i] = p.bias_p[i];
    for (int i = threadIdx.x; i < 225 * p.nH; i += kThreads) {
        const int h = i % p.nH, e = i / p.nH;
        s_bias[h * 232 + e] = __ldg(p.table + i) * 1.4426950408889634f;
    }
    if (FUSE) {
        // B operand of the shortcut MMAs: row n of the K-major slab is the unit vector e_n (n < 16), i.e. out[:, n] = A[:, n]
        for (int i = threadIdx.x; i < kIdentBytes / 4; i += kThreads) reinterpret_cast<uint32_t*>(ident_s)[i] = 0u;
        __syncthreads();
        if (threadIdx.x < 16) {
            const int n = threadIdx.x;
            *reinterpret_cast<uint16_t*>(ident_s + n * 128 + (((n >> 3) ^ (n & 7)) << 4) + (n & 7) * 2) = 0x3F80;   // bf16 1.0
        }
        fence_proxy_async_smem();
    }
    if (warp == kMmaWarp && lane == 0) {
        for (int s = 0; s < kMaxSlots; ++s) {
            mbar_init(&bars->w_full[s], 1);
            mbar_init(&bars->w_empty[s], 1);
        }
        for (int s = 0; s < 4; ++s) {
            mbar_init(&bars->p_full[s], 1);
            mbar_init(&bars->p_empty[s], 1);
        }
        mbar_init(&bars->x_full, 1);
        mbar_init(&bars->x_empty, 1);
        mbar_init(&bars->qkv_full[0], 1);
        mbar_init(&bars->qkv_full[1], 1);
        mbar_init(&bars->qkv_ready, kEpiWarps);
        mbar_init(&bars->s_full, 1);
        mbar_init(&bars->p_ready, kEpiWarps);
        mbar_init(&bars->o_full, 1);
        mbar_init(&bars->o_ready, kEpiWarps);
        mbar_init(&bars->proj_full, 1);
        mbar_init(&bars->proj_free, kEpiWarps);
        fence_barrier_init();
    }
    if (warp == kWLoaderWarp) tmem_alloc<512>(&bars->tmem_base);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = bars->tmem_base;
    // programmatic dependent launch: the set-up above and the weight loaders run under the predecessor's tail; every warp that reads
    // or writes activations / row statistics (x loader, epilogue warps) first waits for the predecessor to complete
    pdl_launch_dependents();
    if (warp < kEpiWarps || warp == kXLoaderWarp) pdl_wait();
    const int uq = p.hdp >> 4;                                         // 16-column units (= K16 steps) per head operand
    const int nwx = p.W >> 3, nW = (p.H >> 3) * nwx;

    if (warp == kXLoaderWarp) {
        // ============================================================ x tile: one TMA box per (window, R x R token block, panel).
        // Tile row of a token = window * 64 + block * R*R + y' * R + x'  (block-major slot order; R = 8: the usual y * 8 + x).
        // Attention is invariant under a permutation of a window's tokens as long as the bias / mask / output row use the
        // same slot -> (y, x) map, which the epilogue warps do.
        if (lane == 0) tma_prefetch_desc(&p.tmap_x);
        const int R = p.box_r, nb = 8 / R;
        const int combos = 2 * nb * nb;
        int qslot = 0;                                                 // pipelined heads: consumer cursor of the qkv weight ring
        uint32_t qph = 0;
        for (int it = 0; it < my_tiles; ++it) {
            const int tile = it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
            tr_ev<TRACE>(p.trace, 2, it, 8, 0);
            mbar_wait(&bars->x_empty, (static_cast<uint32_t>(it) & 1) ^ 1);
            tr_ev<TRACE>(p.trace, 2, it, 8, 1);
            if (lane == 0) mbar_arrive_expect_tx(&bars->x_full, static_cast<uint32_t>(x_bytes));
            __syncwarp();
            for (int cb = lane; cb < combos; cb += 32) {
                const int w2 = cb / (nb * nb), blk = cb - w2 * nb * nb;
                const int by = blk / nb, bx = blk - by * nb;
                const int win = tile * 2 + w2;
                const int b = win / nW, w = win - b * nW;
                int y = (w / nwx) * 8 + by * R + p.shift; if (y >= p.H) y -= p.H;
                int x = (w % nwx) * 8 + bx * R + p.shift; if (x >= p.W) x -= p.W;
                uint8_t* dst = x_buf + (w2 * 64 + blk * R * R) * 128;
                for (int pn = 0; pn < p.ks; ++pn) tma_load_4d(dst + pn * kPanelBytes, &p.tmap_x, pn * 64, x, y, b, &bars->x_full);
            }
            __syncwarp();
            tr_ev<TRACE>(p.trace, 2, it, 8, 2);
            if (FUSE && p.pipe) {
                // pipelined heads: this warp also issues the q|k|v MMAs of the tile it has just requested (accumulator columns of
                // their own; head g may start once the conversion warps have read head g - 1 out of them).  The same split for the
                // two-region attention-only plans (S / P V no longer polled between q|k|v steps) gained 1 %: not kept.
                mbar_wait(&bars->x_full, static_cast<uint32_t>(it) & 1);
                const uint64_t x_desc = umma_desc_k_sw128(smem_u32(x_buf));
                const uint64_t ring_desc = umma_desc_k_sw128(smem_u32(ring));
                const uint32_t slot_units = static_cast<uint32_t>(p.w_slot_bytes >> 4);
                for (int h = 0; h < p.nH; ++h) {
                    const int g = it * p.nH + h;
                    const uint32_t acc = tmem + static_cast<uint32_t>(p.col_acc);
                    // head g may start once the conversion warps have read head g - 1 out of the accumulator columns.  (Gating on "S of head
                    // g - 1 issued / completed" instead, so that these bulk MMAs queue behind the latency-critical S, was measured slower:
                    // 221 / 218 vs 209 us -- they then sit in front of P V.)
                    // (this warp is never two phases behind: qkv_ready of head g needs the q|k|v it is about to issue)
                    if (g > 0) mbar_wait(&bars->qkv_ready, static_cast<uint32_t>(g - 1) & 1);
                    tr_ev<TRACE>(p.trace, 2, it, h, 4);
                    // (K slab, N piece) steps of 4 MMAs: one batch of 12 in a single elected region was measured at ~280 cycles per MMA
                    for (int qs = 0; qs < p.ks; ++qs) {
                        const int ksteps = min(4, p.k16 - 4 * qs);
                        uint32_t dcol = 0;
                        for (int pc = 0; pc < p.qkv_pieces; ++pc) {
                            mbar_wait(&bars->w_full[qslot], qph);
                            tc_fence_after_sync();
                            if (elect_one_sync()) {
                                const uint64_t adesc = x_desc + static_cast<uint64_t>(qs * (kPanelBytes >> 4));
                                const uint64_t bdesc = ring_desc + static_cast<uint64_t>(static_cast<uint32_t>(qslot) * slot_units);
                                const uint32_t idesc = idesc_m128(static_cast<uint32_t>(p.qp_rows[pc]), 0);
                                umma_bf16(acc + dcol, adesc, bdesc, idesc, qs > 0 ? 1u : 0u);
                                if (ksteps > 1) umma_bf16(acc + dcol, adesc + 2, bdesc + 2, idesc, 1u);
                                if (ksteps > 2) umma_bf16(acc + dcol, adesc + 4, bdesc + 4, idesc, 1u);
                                if (ksteps > 3) umma_bf16(acc + dcol, adesc + 6, bdesc + 6, idesc, 1u);
                                umma_commit(&bars->w_empty[qslot]);
                                if (qs == p.ks - 1 && pc == p.qkv_pieces - 1) {
                                    umma_commit(&bars->qkv_full[0]);
                                    if (h == p.nH - 1) umma_commit(&bars->x_empty);      // the x tile is no longer an operand
                                }
                            }
                            __syncwarp();
                            dcol += static_cast<uint32_t>(p.qp_rows[pc]);
                            if (++qslot == p.w_slots) { qslot = 0; qph ^= 1; }
                        }
                    }
                    tr_ev<TRACE>(p.trace, 2, it, h, 5);
                }
            }
        }
    } else if (warp == kWLoaderWarp) {
        // ============================================================ qkv weight slabs: (head, K slab, N piece) in order, every tile
        int slot = 0;
        uint32_t phase = 0;
        const size_t slab_bytes = static_cast<size_t>(3 * p.hdp) * 128u;
        for (int it = 0; it < my_tiles; ++it) {
            for (int hs = 0; hs < p.nH * p.ks; ++hs) {
                int row0 = 0;
                for (int pc = 0; pc < p.qkv_pieces; ++pc) {
                    const uint32_t bytes = static_cast<uint32_t>(p.qp_rows[pc]) * 128u;
                    mbar_wait(&bars->w_empty[slot], phase ^ 1);
                    if (elect_one_sync()) {
                        mbar_arrive_expect_tx(&bars->w_full[slot], bytes);
                        bulk_g2s(ring + slot * p.w_slot_bytes, p.w1p + static_cast<size_t>(hs) * slab_bytes + static_cast<size_t>(row0) * 128u, bytes,
                                 &bars->w_full[slot]);
                    }
                    __syncwarp();
                    row0 += p.qp_rows[pc];
                    if (++slot == p.w_slots) { slot = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kPLoaderWarp) {
        // ============================================================ proj weight slabs: (head, N piece) in order, every tile
        if (FUSE) {
            int slot = 0;
            uint32_t phase = 0;
            const size_t pslab_bytes = static_cast<size_t>(p.cp) * 128u;
            for (int it = 0; it < my_tiles; ++it) {
                for (int h = 0; h < p.nH; ++h) {
                    int row0 = 0;
                    for (int pc = 0; pc < p.n_pp; ++pc) {
                        const uint32_t bytes = static_cast<uint32_t>(p.pp_rows[pc]) * 128u;
                        mbar_wait(&bars->p_empty[slot], phase ^ 1);
                        if (elect_one_sync()) {
                            mbar_arrive_expect_tx(&bars->p_full[slot], bytes);
                            bulk_g2s(pring + slot * p.p_slot_bytes, p.w2p + static_cast<size_t>(h) * pslab_bytes + static_cast<size_t>(row0) * 128u, bytes,
                                     &bars->p_full[slot]);
                        }
                        __syncwarp();
                        row0 += p.pp_rows[pc];
                        if (++slot == p.p_slots) { slot = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // ============================================================ MMA issuer (converged warp, one elected lane issues).
        // The tensor pipe executes in issue order, which is what lets S overlay the dead k|v accumulator columns, O the dead
        // q columns and the proj accumulator the dead regions.
        const uint32_t idesc_s = idesc_m128(128, 0);
        const uint32_t idesc_pv = idesc_m128(static_cast<uint32_t>(p.hdp), 1);
        const uint64_t x_desc = umma_desc_k_sw128(smem_u32(x_buf));
        const uint32_t k_addr = smem_u32(k_buf), v_addr = smem_u32(v_buf);
        const uint64_t k_desc = umma_desc_k_sw128(k_addr);
        const uint64_t ring_desc = umma_desc_k_sw128(smem_u32(ring));
        const uint32_t slot_units = static_cast<uint32_t>(p.w_slot_bytes >> 4);
        const uint64_t pring_desc = umma_desc_k_sw128(smem_u32(pring));
        const uint32_t pslot_units = static_cast<uint32_t>(p.p_slot_bytes >> 4);
        int slot = 0, pslot = 0;
        uint32_t wph = 0, pph = 0;
        int o_waited = 0;                                              // o_ready phases consumed so far (they complete in head order)
        auto ensure_o = [&](int g) {                                   // the epilogue is done with O (and the region) of head counter g
            while (o_waited <= g) {
                mbar_wait(&bars->o_ready, static_cast<uint32_t>(o_waited) & 1);
                ++o_waited;
            }
            tc_fence_after_sync();
        };
        auto region_of = [&](int g) -> uint32_t {                      // fuse_proj: one region behind the proj accumulator
            return tmem + static_cast<uint32_t>(FUSE ? p.cp : (p.nreg == 2 ? (g & 1) : 0) * p.rsz);
        };

        // q|k|v of one head is issued in (K slab, N piece) steps so that the short S / P V MMAs of the current head can cut in
        // between the steps of the next head's q|k|v (the tensor pipe runs in issue order)
        int q_g = 0, q_step = 0, q_s = 0, q_pc = 0;
        const int q_steps = p.ks * p.qkv_pieces;
        const uint32_t idesc_q0 = idesc_m128(static_cast<uint32_t>(p.qp_rows[0]), 0);
        const uint32_t idesc_q1 = idesc_m128(static_cast<uint32_t>(p.qp_rows[1] > 0 ? p.qp_rows[1] : 16), 0);
        uint32_t q_dst = 0;                                            // region of head q_g
        uint32_t q_full_idx = 0;
        bool q_last_head = false;
        auto ready = [&](uint64_t* bar, uint32_t parity) -> bool {     // one lane polls, the warp stays converged
            uint32_t ok = 0;
            if (lane == 0) ok = mbar_test_wait(bar, parity) ? 1u : 0u;
            return __shfl_sync(0xffffffffu, ok, 0) != 0;
        };
        auto qkv_step = [&]() {                                        // precondition: the ring slot has landed
            tc_fence_after_sync();
            if (elect_one_sync()) {
                const int ksteps = min(4, p.k16 - 4 * q_s);
                const uint32_t d = q_pc ? q_dst + static_cast<uint32_t>(p.qp_rows[0]) : q_dst;
                const uint64_t adesc = x_desc + static_cast<uint64_t>(q_s * (kPanelBytes >> 4));
                const uint64_t bdesc = ring_desc + static_cast<uint64_t>(static_cast<uint32_t>(slot) * slot_units);
                const uint32_t idesc = q_pc ? idesc_q1 : idesc_q0;
                umma_bf16(d, adesc, bdesc, idesc, q_s > 0 ? 1u : 0u);
                if (ksteps > 1) umma_bf16(d, adesc + 2, bdesc + 2, idesc, 1u);
                if (ksteps > 2) umma_bf16(d, adesc + 4, bdesc + 4, idesc, 1u);
                if (ksteps > 3) umma_bf16(d, adesc + 6, bdesc + 6, idesc, 1u);
                umma_commit(&bars->w_empty[slot]);
                if (q_step == q_steps - 1) {
                    umma_commit(&bars->qkv_full[q_full_idx]);
                    if (q_last_head) umma_commit(&bars->x_empty);      // the x tile is no longer an operand
                }
            }
            __syncwarp();
            ++q_step;
            if (++q_pc == p.qkv_pieces) { q_pc = 0; ++q_s; }
            if (++slot == p.w_slots) { slot = 0; wph ^= 1; }
        };
        auto qkv_begin = [&](int g, int head) {               // head = g % nH, known to every caller (no division on this path)
            q_g = g; q_step = 0; q_s = 0; q_pc = 0;
            q_dst = (FUSE && p.col_acc >= 0) ? tmem + static_cast<uint32_t>(p.col_acc) : region_of(g);
            q_full_idx = (!FUSE && p.nreg == 2) ? static_cast<uint32_t>(g & 1) : 0u;
            q_last_head = head == p.nH - 1;
        };
        auto qkv_finish = [&]() {
            while (q_step < q_steps) {
                mbar_wait(&bars->w_full[slot], wph);
                qkv_step();
            }
        };
        q_step = q_steps;                                              // nothing pending

        if (my_tiles > 0 && !(FUSE && p.pipe)) {
            mbar_wait(&bars->x_full, 0);
            qkv_begin(0, 0);
            qkv_finish();
        }
        for (int it = 0; it < my_tiles; ++it) {
            for (int h = 0; h < p.nH; ++h) {
                const int g = it * p.nH + h;
                const uint32_t par = static_cast<uint32_t>(g) & 1;
                const bool next_in_tile = h + 1 < p.nH;
                const bool more_tiles = it + 1 < my_tiles;
                const uint32_t t_r = region_of(g);
                const uint32_t t_s = t_r + static_cast<uint32_t>(p.hdp);
                const uint32_t t_o = FUSE ? tmem + static_cast<uint32_t>(p.col_o) : t_r;
                auto issue_s = [&]() {
                    // S = q k^T : q bf16 in TMEM (unit u at column 16 u of the region), k panel in shared memory
                    tc_fence_after_sync();
                    if (elect_one_sync()) {
#pragma unroll
                        for (int u = 0; u < 8; ++u) {                  // straight-line issue: a rolled loop costs ~100 cycles per MMA
                            if (u < uq)
                                umma_bf16_ts(t_s, t_r + static_cast<uint32_t>(16 * u),
                                             k_desc + static_cast<uint64_t>(((u >> 2) * kPanelBytes + (u & 3) * 32) >> 4), idesc_s, u == 0 ? 0u : 1u);
                        }
                        umma_commit(&bars->s_full);
                    }
                    __syncwarp();
                };
                auto issue_pv = [&]() {
                    // O = P v : P bf16 in TMEM (16 keys per step = 8 packed columns), v rows as MN-major B operand; without proj
                    // fusion O lands on the q columns (q was consumed by S, which has completed: the softmax ran on it)
                    tc_fence_after_sync();
                    if (elect_one_sync()) {
#pragma unroll
                        for (int k = 0; k < 8; ++k)
                            umma_bf16_ts(t_o, t_s + static_cast<uint32_t>(8 * k), desc_mn_sw128(v_addr + (p.pipe ? static_cast<uint32_t>((g & 1) * op_bytes) : 0u) + static_cast<uint32_t>(k * 2048), kPanelBytes),
                                         idesc_pv, k == 0 ? 0u : 1u);
                        umma_commit(&bars->o_full);
                    }
                    __syncwarp();
                };
                tr_ev<TRACE>(p.trace, 0, it, h, 0);
                if (FUSE && p.pipe) {
                    // pipelined heads (separate q|k|v accumulator columns): S of head h + 1 goes in front of the proj MMAs of head h, right
                    // behind P V of head h -- the conversion warps have turned head h + 1 around by then.  The q|k|v MMAs are issued by
                    // the x-loader warp: with them this warp's issue time per head (3.7 k cycles) was the bottleneck of the pipeline
                    auto issue_proj_shortcut = [&]() {
                        // the accumulator starts as the shortcut: Y[:, 16 g .. 16 g + 15] = x[:, same columns] * I (x tile still
                        // resident; bf16 values enter the fp32 accumulator exactly), the proj MMAs of every head accumulate on top
                        mbar_wait(&bars->proj_free, (static_cast<uint32_t>(it) & 1) ^ 1);
                        tc_fence_after_sync();
                        if (elect_one_sync()) {
                            const uint64_t idesc_b = umma_desc_k_sw128(smem_u32(ident_s));
                            const uint32_t idesc16 = idesc_m128(16u, 0);
                            const int n16 = p.cp >> 4;
#pragma unroll
                            for (int gcol = 0; gcol < 20; ++gcol)             // cp <= 320
                                if (gcol < n16)
                                    umma_bf16(tmem + static_cast<uint32_t>(16 * gcol),
                                              x_desc + static_cast<uint64_t>((gcol >> 2) * (kPanelBytes >> 4) + (gcol & 3) * 2), idesc_b, idesc16, 0u);
                        }
                        __syncwarp();
                    };
                    if (h == 0) {
                        mbar_wait(&bars->qkv_ready, par);
                        tr_ev<TRACE>(p.trace, 0, it, h, 2);
                        issue_s();
                        issue_proj_shortcut();
                    }
                    mbar_wait(&bars->p_ready, par);
                    tr_ev<TRACE>(p.trace, 0, it, h, 3);
                    issue_pv();
                    tr_ev<TRACE>(p.trace, 0, it, h, 4);
                    if (next_in_tile) {
                        // S of the next head: same code as issue_s() with the next head's counters (its region is the same one)
                        mbar_wait(&bars->qkv_ready, par ^ 1);
                        tc_fence_after_sync();
                        if (elect_one_sync()) {
#pragma unroll
                            for (int u = 0; u < 8; ++u)
                                if (u < uq)
                                    umma_bf16_ts(t_s, t_r + static_cast<uint32_t>(16 * u),
                                                 k_desc + static_cast<uint64_t>(((u >> 2) * kPanelBytes + (u & 3) * 32) >> 4), idesc_s, u == 0 ? 0u : 1u);
                            umma_commit(&bars->s_full);
                        }
                        __syncwarp();
                    }
                    tr_ev<TRACE>(p.trace, 0, it, h, 1);
                    ensure_o(g);
                    uint32_t dcol = 0;
                    for (int pc = 0; pc < p.n_pp; ++pc) {
                        mbar_wait(&bars->p_full[pslot], pph);
                        tc_fence_after_sync();
                        if (elect_one_sync()) {
                            const uint64_t bdesc = pring_desc + static_cast<uint64_t>(static_cast<uint32_t>(pslot) * pslot_units);
                            const uint32_t idesc = idesc_m128(static_cast<uint32_t>(p.pp_rows[pc]), 0);
#pragma unroll
                            for (int u = 0; u < 4; ++u)                // fuse_proj: hdp <= 64
                                if (u < uq) umma_bf16_ts(tmem + dcol, t_o + static_cast<uint32_t>(16 * u), bdesc + 2 * u, idesc, 1u);
                            umma_commit(&bars->p_empty[pslot]);
                            if (h == p.nH - 1 && pc == p.n_pp - 1) umma_commit(&bars->proj_full);
                        }
                        __syncwarp();
                        dcol += static_cast<uint32_t>(p.pp_rows[pc]);
                        if (++pslot == p.p_slots) { pslot = 0; pph ^= 1; }
                    }
                    tr_ev<TRACE>(p.trace, 0, it, h, 5);
                } else if (FUSE) {
                    // one region: S / P overlay the k|v accumulators, so the next head's q|k|v follows P V in the pipe; it runs
                    // while the epilogue normalises O, whose bf16 copy then feeds  Y += O_h Wp_h^T  (persistent accumulator)
                    mbar_wait(&bars->qkv_ready, par);
                    tr_ev<TRACE>(p.trace, 0, it, h, 2);
                    issue_s();
                    if (h == 0) {   // issued under the softmax of head 0: the MMA warp and the tensor pipe are idle then (it used to delay S of head 1)
                        // the accumulator starts as the shortcut: Y[:, 16 g .. 16 g + 15] = x[:, same columns] * I (x tile still
                        // resident; bf16 values enter the fp32 accumulator exactly), the proj MMAs of every head accumulate on top
                        mbar_wait(&bars->proj_free, (static_cast<uint32_t>(it) & 1) ^ 1);
                        tc_fence_after_sync();
                        if (elect_one_sync()) {
                            const uint64_t idesc_b = umma_desc_k_sw128(smem_u32(ident_s));
                            const uint32_t idesc16 = idesc_m128(16u, 0);
                            const int n16 = p.cp >> 4;
#pragma unroll
                            for (int gcol = 0; gcol < 20; ++gcol)             // cp <= 320
                                if (gcol < n16)
                                    umma_bf16(tmem + static_cast<uint32_t>(16 * gcol),
                                              x_desc + static_cast<uint64_t>((gcol >> 2) * (kPanelBytes >> 4) + (gcol & 3) * 2), idesc_b, idesc16, 0u);
                        }
                        __syncwarp();
                    }
                    const bool acc_sep = p.col_acc >= 0;               // q|k|v has its own accumulator columns (spare TMEM): the next
                    if (acc_sep && next_in_tile) {                     // head's q|k|v need not wait for P V, it runs under the softmax
                        qkv_begin(g + 1, next_in_tile ? h + 1 : 0);
                        qkv_finish();
                    }
                    mbar_wait(&bars->p_ready, par);
                    tr_ev<TRACE>(p.trace, 0, it, h, 3);
                    issue_pv();
                    tr_ev<TRACE>(p.trace, 0, it, h, 4);
                    if (!acc_sep && next_in_tile) {
                        qkv_begin(g + 1, next_in_tile ? h + 1 : 0);
                        qkv_finish();
                    }
                    tr_ev<TRACE>(p.trace, 0, it, h, 1);
                    ensure_o(g);
                    uint32_t dcol = 0;
                    for (int pc = 0; pc < p.n_pp; ++pc) {
                        mbar_wait(&bars->p_full[pslot], pph);
                        tc_fence_after_sync();
                        if (elect_one_sync()) {
                            const uint64_t bdesc = pring_desc + static_cast<uint64_t>(static_cast<uint32_t>(pslot) * pslot_units);
                            const uint32_t idesc = idesc_m128(static_cast<uint32_t>(p.pp_rows[pc]), 0);
#pragma unroll
                            for (int u = 0; u < 4; ++u)                // fuse_proj: hdp <= 64
                                if (u < uq) umma_bf16_ts(tmem + dcol, t_o + static_cast<uint32_t>(16 * u), bdesc + 2 * u, idesc, 1u);
                            umma_commit(&bars->p_empty[pslot]);
                            if (h == p.nH - 1 && pc == p.n_pp - 1) umma_commit(&bars->proj_full);
                        }
                        __syncwarp();
                        dcol += static_cast<uint32_t>(p.pp_rows[pc]);
                        if (++pslot == p.p_slots) { pslot = 0; pph ^= 1; }
                    }
                    tr_ev<TRACE>(p.trace, 0, it, h, 5);
                    if (!next_in_tile && more_tiles) {
                        mbar_wait(&bars->x_full, static_cast<uint32_t>(it + 1) & 1);
                        qkv_begin(g + 1, next_in_tile ? h + 1 : 0);                              // next tile's first head: overlaps the last epilogue of this tile
                        qkv_finish();
                    }
                } else if (p.nreg == 2) {
                    // the other region was last used by head g - 1: once its O has been read it takes the next head's q|k|v, which
                    // the tensor pipe computes while the epilogue warps turn head g around (also across tile borders)
                    if (g >= 1) ensure_o(g - 1);
                    const bool look = next_in_tile || more_tiles;
                    bool began = false;
                    if (next_in_tile) { qkv_begin(g + 1, next_in_tile ? h + 1 : 0); began = true; }
                    bool s_done = false, pv_done = false;
                    while (!pv_done) {
                        if (!s_done) {
                            if (ready(&bars->qkv_ready, par)) { tr_ev<TRACE>(p.trace, 0, it, h, 2); issue_s(); s_done = true; continue; }
                        } else if (ready(&bars->p_ready, par)) {
                            tr_ev<TRACE>(p.trace, 0, it, h, 3);
                            issue_pv();
                            pv_done = true;
                            continue;
                        }
                        if (look && !began && ready(&bars->x_full, static_cast<uint32_t>(it + 1) & 1)) { qkv_begin(g + 1, next_in_tile ? h + 1 : 0); began = true; }
                        if (began && q_step < q_steps && ready(&bars->w_full[slot], wph)) qkv_step();
                    }
                    tr_ev<TRACE>(p.trace, 0, it, h, 4);
                    if (look) {
                        if (!began) {
                            mbar_wait(&bars->x_full, static_cast<uint32_t>(it + 1) & 1);
                            qkv_begin(g + 1, next_in_tile ? h + 1 : 0);
                        }
                        qkv_finish();
                    }
                    tr_ev<TRACE>(p.trace, 0, it, h, 1);
                } else {
                    mbar_wait(&bars->qkv_ready, par);
                    tr_ev<TRACE>(p.trace, 0, it, h, 2);
                    issue_s();
                    mbar_wait(&bars->p_ready, par);
                    tr_ev<TRACE>(p.trace, 0, it, h, 3);
                    issue_pv();
                    tr_ev<TRACE>(p.trace, 0, it, h, 4);
                    ensure_o(g);                                       // single region: strictly one head after the other
                    if (next_in_tile || more_tiles) {
                        if (!next_in_tile) mbar_wait(&bars->x_full, static_cast<uint32_t>(it + 1) & 1);
                        qkv_begin(g + 1, next_in_tile ? h + 1 : 0);
                        qkv_finish();
                    }
                }
            }
        }
    } else if (warp < kEpiWarps) {
        // ============================================================ epilogue / softmax warps
        const int quad = warp & 3, grp = warp >> 2;
        const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
        const int r = quad * 32 + lane;                                // tile row; window = r >> 6, slot = r & 63
        const int rsw = r & 7;
        const int n = r & 63;
        const uint32_t kcol0 = static_cast<uint32_t>((r >> 6) * 64);   // my window's keys inside the 128 S columns
        // slot -> (y, x) inside the window (block-major for R = 4, see the x loader); my 16 keys are slots 16 grp .. 16 grp + 15:
        // R = 8: key rows 2 grp, 2 grp + 1;  R = 4: the 4 x 4 block grp
        const bool blk4 = p.box_r == 4;
        const int ny = blk4 ? ((n >> 5) << 2) + ((n >> 2) & 3) : (n >> 3);
        const int nx = blk4 ? (((n >> 4) & 1) << 2) + (n & 3) : (n & 7);
        const int ky0 = blk4 ? (grp >> 1) * 4 : 2 * grp, kx0 = blk4 ? (grp & 1) * 4 : 0;   // first key of my 16
        const int qb = (ny - ky0 + 7) * 15 + (nx - kx0 + 7);           // bias index of that key; key (ky0 + dy, kx0 + dx): - (15 dy + dx)
        const uint32_t k_row = smem_u32(k_buf) + static_cast<uint32_t>(r * 128);
        const uint32_t v_row = smem_u32(v_buf) + static_cast<uint32_t>(r * 128);
        const float2 sc2 = f2_(p.scale_log2e, p.scale_log2e);
        const uint32_t t_base = tmem + lane_off;
        const int t128 = grp * 32 + lane;
        const uint32_t cpr_magic = (65536u + static_cast<uint32_t>(p.hdp >> 3) - 1u) / static_cast<uint32_t>(p.hdp >> 3);   // id / (hdp / 8), id < 512

        // ---- per-tile set-up of my row: slot -> token (closed form of roll + window_partition), the mask bits of my 16 keys and the
        // LayerNorm statistics.  The (sum, sumsq) slots are a COLD global load (written by the previous kernel), so the set-up of
        // tile it + 1 runs while tile it waits for its first S anyway (the load latency disappears in that wait)
        auto row_setup = [&](int tile, int& tok_o, uint32_t& mbits_o, float& rstd_o, float& nrm_o) {
            const int win = tile * 2 + (r >> 6);
            const int b = win / nW, w = win - b * nW;
            const int wy = (w / nwx) * 8, wx = (w % nwx) * 8;
            const int ys = wy + ny, xs = wx + nx;
            int y = ys + p.shift; if (y >= p.H) y -= p.H;
            int x = xs + p.shift; if (x >= p.W) x -= p.W;
            const int tok = (b * p.H + y) * p.W + x;
            uint32_t mbits = 0xffffu;
            if (p.shift > 0) {
                // key k lies in my mask region iff its row AND its column do (region id = 3 ry + rx, src/drct.py:449-470)
                const int my_ry = region_1d_(ys, p.H, p.shift), my_rx = region_1d_(xs, p.W, p.shift);
                const int kw = blk4 ? 4 : 8, kh = 16 / kw;             // my keys: kh rows of kw
                uint32_t xmask = 0;
                for (int j = 0; j < kw; ++j) xmask |= (region_1d_(wx + kx0 + j, p.W, p.shift) == my_rx ? 1u : 0u) << j;
                mbits = 0u;
                for (int i = 0; i < kh; ++i)
                    if (region_1d_(wy + ky0 + i, p.H, p.shift) == my_ry) mbits |= xmask << (i * kw);
            }
            const float2* sp = p.stats_in + static_cast<long long>(tok) * p.stats_in_stride;
            float s1 = 0.f, s2 = 0.f;
            for (int k = 0; k < p.stats_in_slots; ++k) {
                const float2 v = __ldg(sp + k);
                s1 += v.x;
                s2 += v.y;
            }
            const float inv_c = 1.0f / static_cast<float>(p.C);
            const float mean = s1 * inv_c;
            const float rs = rsqrtf(fmaxf(s2 * inv_c - mean * mean, 0.f) + p.ln_eps);
            tok_o = tok; mbits_o = mbits; rstd_o = rs; nrm_o = -mean * rs;
        };
        int tok = 0;
        uint32_t mbits = 0xffffu;
        float rstd = 0.f, nrm = 0.f;
        // p.early_setup (plans whose next q|k|v runs ahead, so that a tile does NOT start with a long wait that would hide the loads):
        // the set-up of tile it + 1 runs while tile it waits for its first S; otherwise it runs at the tile top, under the
        // q|k|v wait, with the statistics pulled into L1 one tile ahead
        int tok_n = 0;
        uint32_t mbits_n = 0xffffu;
        float rstd_n = 0.f, nrm_n = 0.f;
        const bool early = p.early_setup != 0;
        if (early && my_tiles > 0) row_setup(static_cast<int>(blockIdx.x), tok, mbits, rstd, nrm);

        for (int it = 0; it < my_tiles; ++it) {
            const int tile = it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
            const int mb = it & 1;
            if (!early) {
              if (grp == 1 && it + 1 < my_tiles) {
                // the (sum, sumsq) slots of my row in the NEXT tile: fetched cold at the tile start they cost ~2k cycles of exposed
                // latency, so their line is pulled into L1 a whole tile ahead (same closed-form token map)
                const int win = (tile + static_cast<int>(gridDim.x)) * 2 + (r >> 6);
                const int b = win / nW, w = win - b * nW;
                int y = (w / nwx) * 8 + ny + p.shift; if (y >= p.H) y -= p.H;
                int x = (w % nwx) * 8 + nx + p.shift; if (x >= p.W) x -= p.W;
                const char* np_ = reinterpret_cast<const char*>(p.stats_in + static_cast<long long>((b * p.H + y) * p.W + x) * p.stats_in_stride);
                for (int o = 0; o < p.stats_in_slots * 8; o += 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(np_ + o));
              }
              row_setup(tile, tok, mbits, rstd, nrm);
            }
            if (grp == 0) s_tok[mb * 128 + r] = tok;
            const float2 rstd2 = f2_(rstd, rstd), nrm2 = f2_(nrm, nrm);

            // The three stages of a head.  Usual order: convert(h), softmax(h), normalise(h).  Pipelined order (p.pipe: blocks whose
            // next q|k|v has accumulator columns of its own, so it is complete while the softmax runs): convert(h + 1) goes BETWEEN
            // softmax(h) and normalise(h) -- it runs under P V of head h (q columns and the k panel are dead once S has completed,
            // the v panel alternates), and normalise(h) then runs under S of head h + 1: on the clock64 timeline of block 1 the
            // conversion warps waited 0.46 k cycles for S and 0.54 k for P V in every head of 4.0 k.
            auto stage_convert = [&](int h) {
                const int g = it * p.nH + h;
                const uint32_t par = static_cast<uint32_t>(g) & 1;
                const int reg = (!FUSE && p.nreg == 2) ? (g & 1) : 0;
                const uint32_t t_r = t_base + static_cast<uint32_t>(FUSE ? p.cp : reg * p.rsz);
                const uint32_t t_s = t_r + static_cast<uint32_t>(p.hdp);
                const uint32_t t_o = FUSE ? t_base + static_cast<uint32_t>(p.col_o) : t_r;
                const uint32_t t_acc = (FUSE && p.col_acc >= 0) ? t_base + static_cast<uint32_t>(p.col_acc) : t_r;   // q|k|v accumulators
                (void)par; (void)t_s; (void)t_o; (void)t_acc;
                // ---- q | k | v of head h: folded LayerNorm + bias -> bf16; q in place (TMEM), k / v into the operand panels
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, h, 0);
                mbar_wait(&bars->qkv_full[reg], static_cast<uint32_t>((!FUSE && p.nreg == 2) ? (g >> 1) : g) & 1);
                tc_fence_after_sync();
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, h, 1);
                for (int u = grp; u < 3 * uq; u += 4) {
                    uint32_t raw[16];
                    tmem_ld16(t_acc + static_cast<uint32_t>(16 * u), raw);
                    tmem_ld_wait();
                    const float* bp = s_bq + h * 3 * p.hdp + 16 * u;
                    const float* cp = s_cq + h * 3 * p.hdp + 16 * u;
                    uint32_t pk[8];
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) {
                        const float4 bb = *reinterpret_cast<const float4*>(bp + 4 * q4);
                        const float4 cs = *reinterpret_cast<const float4*>(cp + 4 * q4);
                        const float2 x0 = __ffma2_rn(rstd2, f2_(__uint_as_float(raw[4 * q4]), __uint_as_float(raw[4 * q4 + 1])),
                                                     __ffma2_rn(nrm2, f2_(cs.x, cs.y), f2_(bb.x, bb.y)));
                        const float2 x1 = __ffma2_rn(rstd2, f2_(__uint_as_float(raw[4 * q4 + 2]), __uint_as_float(raw[4 * q4 + 3])),
                                                     __ffma2_rn(nrm2, f2_(cs.z, cs.w), f2_(bb.z, bb.w)));
                        pk[2 * q4] = pack_bf16x2(x0.x, x0.y);
                        pk[2 * q4 + 1] = pack_bf16x2(x1.x, x1.y);
                    }
                    if (u < uq) {
                        tmem_st8_(t_r + static_cast<uint32_t>(16 * u), pk);
                    } else {
                        const bool is_k = u < 2 * uq;
                        const int cu = u - (is_k ? uq : 2 * uq);       // unit inside the operand: columns 16 cu .. 16 cu + 15
                        const uint32_t rowa = (is_k ? k_row : v_row + (p.pipe ? static_cast<uint32_t>((g & 1) * op_bytes) : 0u)) + static_cast<uint32_t>((cu >> 2) * kPanelBytes);
                        const int c0 = (2 * cu) & 7;
                        st_shared_v4(rowa + static_cast<uint32_t>(((c0 ^ rsw) << 4)), pk[0], pk[1], pk[2], pk[3]);
                        st_shared_v4(rowa + static_cast<uint32_t>((((c0 + 1) ^ rsw) << 4)), pk[4], pk[5], pk[6], pk[7]);
                    }
                }
                tmem_st_wait();
                fence_proxy_async_smem();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->qkv_ready);
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, h, 2);

            };
            auto stage_softmax = [&](int h) {
                const int g = it * p.nH + h;
                const uint32_t par = static_cast<uint32_t>(g) & 1;
                const int reg = (!FUSE && p.nreg == 2) ? (g & 1) : 0;
                const uint32_t t_r = t_base + static_cast<uint32_t>(FUSE ? p.cp : reg * p.rsz);
                const uint32_t t_s = t_r + static_cast<uint32_t>(p.hdp);
                const uint32_t t_o = FUSE ? t_base + static_cast<uint32_t>(p.col_o) : t_r;
                const uint32_t t_acc = (FUSE && p.col_acc >= 0) ? t_base + static_cast<uint32_t>(p.col_acc) : t_r;   // q|k|v accumulators
                (void)par; (void)t_s; (void)t_o; (void)t_acc;
                // ---- softmax over my window's 64 keys, 16 per thread
                if (early && h == 0 && it + 1 < my_tiles) row_setup(tile + static_cast<int>(gridDim.x), tok_n, mbits_n, rstd_n, nrm_n);
                mbar_wait(&bars->s_full, par);
                tc_fence_after_sync();
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, h, 3);
                float t[16];
                float mx = -INFINITY;
                {
                    uint32_t raw[16];
                    tmem_ld16(t_s + kcol0 + static_cast<uint32_t>(16 * grp), raw);
                    tmem_ld_wait();
                    const float* bias = s_bias + h * 232 + qb;
                    if (blk4) {
#pragma unroll
                        for (int k = 0; k < 16; k += 2) {
                            const float2 bv = f2_(bias[-((k >> 2) * 15 + (k & 3))], bias[-(((k + 1) >> 2) * 15 + ((k + 1) & 3))]);
                            const float2 v = __ffma2_rn(f2_(__uint_as_float(raw[k]), __uint_as_float(raw[k + 1])), sc2, bv);
                            t[k] = v.x;
                            t[k + 1] = v.y;
                            mx = fmaxf(mx, fmaxf(v.x, v.y));
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < 16; k += 2) {
                            const float2 bv = f2_(bias[-((k >> 3) * 15 + (k & 7))], bias[-(((k + 1) >> 3) * 15 + ((k + 1) & 7))]);
                            const float2 v = __ffma2_rn(f2_(__uint_as_float(raw[k]), __uint_as_float(raw[k + 1])), sc2, bv);
                            t[k] = v.x;
                            t[k + 1] = v.y;
                            mx = fmaxf(mx, fmaxf(v.x, v.y));
                        }
                    }
                }
                s_max[grp * 128 + r] = mx;
                named_bar_sync(1 + quad, 128);
                mx = fmaxf(fmaxf(s_max[r], s_max[128 + r]), fmaxf(s_max[256 + r], s_max[384 + r]));
                {
                    const float2 nmx = f2_(-mx, -mx);
                    float2 acc = f2_(0.f, 0.f);
                    uint32_t pk[8];
#ifndef ADSR_NO_FASTPATH
                    if (__all_sync(0xffffffffu, mbits == 0xffffu)) {     // no key of this warp's rows is masked (warp-uniform: a divergent
                                                                         // branch would run the exponentials twice)
#pragma unroll
                        for (int k = 0; k < 16; k += 2) {
                            const float2 d = __fadd2_rn(f2_(t[k], t[k + 1]), nmx);
                            const float2 e = f2_(ex2_approx(d.x), ex2_approx(d.y));
                            acc = __fadd2_rn(acc, e);
                            pk[k >> 1] = pack_bf16x2(e.x, e.y);
                        }
                    } else
#endif
                    {
#pragma unroll
                        for (int k = 0; k < 16; k += 2) {
                            const float2 d = __fadd2_rn(f2_(t[k], t[k + 1]), nmx);
                            float2 e = f2_(ex2_approx(d.x), ex2_approx(d.y));
                            // keys of another mask region get -100 in the reference: their probability is exp(-100) ~ 0
                            if (!((mbits >> k) & 1u)) e.x = 0.f;
                            if (!((mbits >> (k + 1)) & 1u)) e.y = 0.f;
                            acc = __fadd2_rn(acc, e);
                            pk[k >> 1] = pack_bf16x2(e.x, e.y);
                        }
                    }
                    s_sum[(g & 1) * 512 + grp * 128 + r] = acc.x + acc.y;
                    // P in place: key j of the tile -> packed column j / 2; the same keys' slots of the OTHER window get zeros
                    tmem_st8_(t_s + ((kcol0 + static_cast<uint32_t>(16 * grp)) >> 1), pk);
                    tmem_st8_zero_(t_s + (((64u - kcol0) + static_cast<uint32_t>(16 * grp)) >> 1));
                }
                tmem_st_wait();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->p_ready);
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, h, 4);

            };
            auto stage_normalise = [&](int h) {
                const int g = it * p.nH + h;
                const uint32_t par = static_cast<uint32_t>(g) & 1;
                const int reg = (!FUSE && p.nreg == 2) ? (g & 1) : 0;
                const uint32_t t_r = t_base + static_cast<uint32_t>(FUSE ? p.cp : reg * p.rsz);
                const uint32_t t_s = t_r + static_cast<uint32_t>(p.hdp);
                const uint32_t t_o = FUSE ? t_base + static_cast<uint32_t>(p.col_o) : t_r;
                const uint32_t t_acc = (FUSE && p.col_acc >= 0) ? t_base + static_cast<uint32_t>(p.col_acc) : t_r;   // q|k|v accumulators
                (void)par; (void)t_s; (void)t_o; (void)t_acc;
                // ---- O = P v done: normalise; fuse_proj: pack into the persistent bf16 operand, else store the rows
                mbar_wait(&bars->o_full, par);
                tc_fence_after_sync();
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, h, 5);
                {
                    const float* ss = s_sum + (g & 1) * 512;
                    const float inv = 1.0f / ((ss[r] + ss[128 + r]) + (ss[256 + r] + ss[384 + r]));
                    const float2 inv2 = f2_(inv, inv);
                    for (int u = grp; u < uq; u += 4) {
                        uint32_t raw[16];
                        tmem_ld16(t_o + static_cast<uint32_t>(16 * u), raw);
                        tmem_ld_wait();
                        uint32_t pk[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const float2 v = __fmul2_rn(f2_(__uint_as_float(raw[2 * e]), __uint_as_float(raw[2 * e + 1])), inv2);
                            pk[e] = pack_bf16x2(v.x, v.y);
                        }
                        if (FUSE) {
                            tmem_st8_(t_o + static_cast<uint32_t>(16 * u), pk);        // in place: A operand of the proj MMAs
                        } else {
                            // stage the row piece in the k panel (dead: S has completed; same swizzled row layout as k itself)
                            const uint32_t rowa = k_row + static_cast<uint32_t>((u >> 2) * kPanelBytes);
                            const int c0 = (2 * u) & 7;
                            st_shared_v4(rowa + static_cast<uint32_t>(((c0 ^ rsw) << 4)), pk[0], pk[1], pk[2], pk[3]);
                            st_shared_v4(rowa + static_cast<uint32_t>((((c0 + 1) ^ rsw) << 4)), pk[4], pk[5], pk[6], pk[7]);
                        }
                    }
                }
                tmem_st_wait();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->o_ready);            // O has left TMEM: the region may be reused
                if (!FUSE) {
                    // attention rows -> out[token, h * hdp ...]: the quadrant's 32 staged rows are copied out by its four warps,
                    // consecutive lanes along a row (coalesced 16-byte pieces instead of one 32-byte piece per lane and row)
                    named_bar_sync(1 + quad, 128);                       // the quadrant's rows (and s_tok) are complete
                    const int cpr = p.hdp >> 3;                          // 16-byte chunks per row
                    const uint32_t kq = smem_u32(k_buf);
                    for (int id = t128; id < 32 * cpr; id += 128) {
                        const int rl = static_cast<int>((static_cast<uint32_t>(id) * cpr_magic) >> 16), ch = id - rl * cpr;
                        const int rq = quad * 32 + rl;
                        uint4 val;
                        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                                     : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w)
                                     : "r"(kq + static_cast<uint32_t>((ch >> 3) * kPanelBytes + rq * 128 + (((ch & 7) ^ (rq & 7)) << 4))));
                        *reinterpret_cast<uint4*>(p.out + static_cast<long long>(s_tok[mb * 128 + rq]) * p.ldo + h * p.hdp + ch * 8) = val;
                    }
                    named_bar_sync(1 + quad, 128);                       // copied out: the next head may overwrite the k panel
                }
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, h, 6);
            };
            if (FUSE && p.pipe) {
                stage_convert(0);
                for (int h = 0; h < p.nH; ++h) {
                    stage_softmax(h);
                    if (h + 1 < p.nH) stage_convert(h + 1);
                    stage_normalise(h);
                }
            } else {
                for (int h = 0; h < p.nH; ++h) {
                    stage_convert(h);
                    stage_softmax(h);
                    stage_normalise(h);
                }
            }

            if (FUSE) {
                // ---- y = accumulator (shortcut + proj) + bias -> original token rows; (sum, sumsq) of the row for norm2.
                // 64-column chunks are staged in the idle k / v panels so that every global access is a coalesced 128-byte row
                // piece: the epilogue writes its 16 columns, then the quadrant's four warps copy the 32 panel rows out.  A quadrant
                // only touches its own panel rows, so quadrant-wide named barriers are all the sync needed.
                const int nch = (p.cp + 63) >> 6;
                const uint32_t panel0 = smem_u32(k_buf), panel1 = smem_u32(v_buf);
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, 8, 0);
                mbar_wait(&bars->proj_full, static_cast<uint32_t>(it) & 1);
                tc_fence_after_sync();
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, 8, 1);
                float2 st = f2_(0.f, 0.f), sq = f2_(0.f, 0.f);
                for (int c2 = 0; c2 < nch; c2 += 2) {                   // two 64-column chunks (= both panels) per barrier round
#pragma unroll
                    for (int pp = 0; pp < 2; ++pp) {
                        const int col0 = 64 * (c2 + pp) + 16 * grp;
                        if (col0 < p.cp) {
                            uint32_t raw[16];
                            tmem_ld16(t_base + static_cast<uint32_t>(col0), raw);
                            tmem_ld_wait();
                            const uint32_t rowa = (pp ? panel1 : panel0) + static_cast<uint32_t>(r * 128);
#pragma unroll
                            for (int o = 0; o < 2; ++o) {
                                const float4 b0 = *reinterpret_cast<const float4*>(s_bp + col0 + 8 * o);
                                const float4 b1 = *reinterpret_cast<const float4*>(s_bp + col0 + 8 * o + 4);
                                const uint32_t* a8 = &raw[8 * o];
                                const float2 v0 = __fadd2_rn(f2_(__uint_as_float(a8[0]), __uint_as_float(a8[1])), f2_(b0.x, b0.y));
                                const float2 v1 = __fadd2_rn(f2_(__uint_as_float(a8[2]), __uint_as_float(a8[3])), f2_(b0.z, b0.w));
                                const float2 v2 = __fadd2_rn(f2_(__uint_as_float(a8[4]), __uint_as_float(a8[5])), f2_(b1.x, b1.y));
                                const float2 v3 = __fadd2_rn(f2_(__uint_as_float(a8[6]), __uint_as_float(a8[7])), f2_(b1.z, b1.w));
                                // columns >= C: zero weight rows, zero bias, zero-filled x -> exact zeros, no effect on the sums
                                st = __fadd2_rn(st, __fadd2_rn(__fadd2_rn(v0, v1), __fadd2_rn(v2, v3)));
                                sq = __ffma2_rn(v0, v0, sq);
                                sq = __ffma2_rn(v1, v1, sq);
                                sq = __ffma2_rn(v2, v2, sq);
                                sq = __ffma2_rn(v3, v3, sq);
                                st_shared_v4(rowa + static_cast<uint32_t>((((2 * grp + o) ^ rsw) << 4)), pack_bf16x2(v0.x, v0.y),
                                             pack_bf16x2(v1.x, v1.y), pack_bf16x2(v2.x, v2.y), pack_bf16x2(v3.x, v3.y));
                            }
                        }
                    }
                    if (c2 + 2 >= nch) {                                 // the accumulator has been read: the next tile may start it over
                        tc_fence_before_sync();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&bars->proj_free);
                    }
                    named_bar_sync(1 + quad, 128);                       // the quadrant's y chunks (and s_tok) are complete
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int pp = i >> 1;
                        const int id = t128 + 128 * (i & 1);
                        const int rq = quad * 32 + (id >> 3), j = id & 7;
                        const int col = 64 * (c2 + pp) + 8 * j;
                        const int nvalid = p.C - col;
                        if (nvalid > 0) {
                            uint4 val;
                            asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                                         : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w)
                                         : "r"((pp ? panel1 : panel0) + static_cast<uint32_t>(rq * 128) + static_cast<uint32_t>(((j ^ (rq & 7)) << 4))));
                            __nv_bfloat16* dst = p.out + static_cast<long long>(s_tok[mb * 128 + rq]) * p.ldo + col;
                            if (nvalid >= 8) {
                                *reinterpret_cast<uint4*>(dst) = val;
                            } else {
                                const uint32_t w4[4] = {val.x, val.y, val.z, val.w};
#pragma unroll
                                for (int e = 0; e < 8; ++e)
                                    if (e < nvalid) reinterpret_cast<uint16_t*>(dst)[e] = static_cast<uint16_t>((w4[e >> 1] >> (16 * (e & 1))) & 0xffffu);
                            }
                        }
                    }
                    if (c2 + 2 < nch) named_bar_sync(1 + quad, 128);     // copied out: the next round may overwrite the panels
                }
                if (warp == 0) tr_ev<TRACE>(p.trace, 1, it, 8, 2);
                if (p.stats_out != nullptr) {
                    s_stat[grp * 128 + r] = f2_(st.x + st.y, sq.x + sq.y);
                    named_bar_sync(1 + quad, 128);
                    if (grp == 0) {
                        const float2 a = s_stat[r], b = s_stat[128 + r], c = s_stat[256 + r], d = s_stat[384 + r];
                        p.stats_out[static_cast<long long>(tok) * p.stats_out_stride + p.stats_out_slot0] =
                            f2_((a.x + b.x) + (c.x + d.x), (a.y + b.y) + (c.y + d.y));
                    }
                }
                named_bar_sync(1 + quad, 128);   // panels copied out / s_stat consumed before the next tile's k, v, s_max, s_sum writes
            }
            if (early) { tok = tok_n; mbits = mbits_n; rstd = rstd_n; nrm = nrm_n; }
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (warp == kWLoaderWarp) {
        tc_fence_after_sync();
        tmem_dealloc<512>(tmem);
    }
}

int fixed_smem_bytes(int nH, int hdp, int cp) {       // kIdentBytes is only used with fuse_proj; reserving it always keeps this simple
    return kIdentBytes + (2 * nH * 3 * hdp + cp + nH * 232) * 4 + 256 * 4 + 3 * 512 * 4 + static_cast<int>(sizeof(AttnBlockBarriers)) + 64;
}

int round16(int v) { return (v + 15) / 16 * 16; }

}  // namespace

// Static plan of the fused kernel for one block shape.  Returns 0 = not covered (use the separate kernels),
// 1 = qkv + attention fused (out = attention rows [M, nH * hdp], proj by the row-tile GEMM), 2 = whole attention half.
int swin_attn_plan(SwinAttnParams& p, int C, int nH, int hdp, int allow_proj) {
    if (C <= 0 || C > 320 || nH < 1 || nH > 8 || hdp < 32 || hdp > 128 || (hdp % 16) || nH * 3 * hdp > 1024) return 0;
    p.C = C; p.nH = nH; p.hdp = hdp;
    p.ks = (C + 63) / 64;
    p.k16 = (C + 15) / 16;
    p.pan = (hdp + 63) / 64;
    p.cp = round16(C);
    // attention only: a TMEM region hosts a head from start to end -- q|k|v accumulators (3 hdp) -> q bf16 in place + S / P over
    // the dead k|v columns (hdp + 128) -> O over the dead q columns; two regions let the next head's q|k|v run one head ahead.
    // fuse_proj: [proj accumulator cp | region hdp + 128 | O hdp]; q|k|v (3 hdp <= hdp + 128) reuses the region head after head.
    p.rsz = 3 * hdp > hdp + 128 ? 3 * hdp : hdp + 128;
    if (p.rsz > 512) return 0;
    p.fuse_proj = (allow_proj && hdp <= 64 && p.cp + 2 * hdp + 128 <= 512) ? 1 : 0;
    p.nreg = (!p.fuse_proj && 2 * p.rsz <= 512) ? 2 : 1;
    p.col_o = p.fuse_proj ? p.cp + hdp + 128 : 0;
    // spare TMEM (the narrowest block): q|k|v gets accumulator columns of its own behind O, so that the next head's q|k|v MMAs can
    // be issued as soon as S is (they no longer overwrite P) instead of after P V
    p.col_acc = (p.fuse_proj && p.cp + 2 * hdp + 128 + 3 * hdp <= 512) ? p.cp + 2 * hdp + 128 : -1;
    p.early_setup = p.col_acc >= 0 ? 1 : 0;
    // ... and then the heads are pipelined: the conversion of head h + 1 runs under P V of head h (second v panel), the
    // normalisation of head h under S of head h + 1
    p.pipe = p.col_acc >= 0 ? 1 : 0;
    // a [3 hdp x 64] qkv slab is one ring slot and one issue step (every step costs ~400 cycles of wait / commit bookkeeping on
    // top of its MMAs, so steps are kept as large as the MMA N limit of 256 allows); 3 hdp > 256: two N pieces
    const int n3 = 3 * hdp;
    p.qkv_pieces = n3 <= 256 ? 1 : 2;
    p.qp_rows[0] = p.qkv_pieces == 1 ? n3 : round16(n3 / 2);
    p.qp_rows[1] = n3 - p.qp_rows[0];
    p.qp_rows[2] = p.qp_rows[3] = 0;
    p.w_slot_bytes = (p.qp_rows[0] * 128 + 1023) / 1024 * 1024;        // qp_rows[0] >= qp_rows[1]
    p.n_pp = 0;
    p.p_slots = 0;
    p.p_slot_bytes = 0;
    for (int i = 0; i < 4; ++i) p.pp_rows[i] = 0;
    if (p.fuse_proj) {                                                 // a head's proj slab [cp x 64]: one MMA N piece, or two when cp > 256
        p.n_pp = p.cp <= 256 ? 1 : 2;
        p.pp_rows[0] = p.n_pp == 1 ? p.cp : round16(p.cp / 2);
        p.pp_rows[1] = p.cp - p.pp_rows[0];
        p.p_slot_bytes = (p.pp_rows[0] * 128 + 1023) / 1024 * 1024;
        p.p_slots = p.n_pp;                                            // the ring holds one head's proj weights: fetched a head ahead
    }
    const int avail = kSmemLimit - p.ks * kPanelBytes - (2 + p.pipe) * p.pan * kPanelBytes - fixed_smem_bytes(nH, hdp, p.cp) - p.p_slots * p.p_slot_bytes;
    p.w_slots = avail / p.w_slot_bytes;
    if (p.w_slots > kMaxSlots) p.w_slots = kMaxSlots;
    if (p.w_slots < 2) return 0;
    return p.fuse_proj ? 2 : 1;
}

int launch_swin_attn(SwinAttnParams& p, int num_sms, cudaStream_t stream) {
    const int nW = (p.H / 8) * (p.W / 8);
    if ((p.H % 8) || (p.W % 8) || ((p.B * nW) & 1) || p.shift < 0 || p.shift >= 8) return ADSR_ERR_BAD_SHAPE;
    if ((reinterpret_cast<uintptr_t>(p.x) & 15) || (reinterpret_cast<uintptr_t>(p.out) & 15) || (p.ldx % 8) || (p.ldo % 8) ||
        (reinterpret_cast<uintptr_t>(p.w1p) & 15) || (reinterpret_cast<uintptr_t>(p.w2p) & 15))
        return ADSR_ERR_BAD_ALIGN;
    if (p.ldx < (p.C + 7) / 8 * 8) return ADSR_ERR_BAD_SHAPE;
    if (p.fuse_proj ? p.ldo < (p.C + 7) / 8 * 8 : p.ldo < p.nH * p.hdp) return ADSR_ERR_BAD_SHAPE;
    p.n_tiles = p.B * nW / 2;
    if (p.shift != 0 && p.shift != 4) return ADSR_ERR_BAD_SHAPE;      // square token boxes of side 8 / 4 cover these two
    p.box_r = p.shift == 0 ? 8 : 4;
    const int st = encode_tmap_nhwc_box_bf16(&p.tmap_x, p.x, p.B, p.H, p.W, p.C, p.ldx, p.box_r);
    if (st != ADSR_OK) return st;
    const int smem_bytes = p.ks * kPanelBytes + (2 + p.pipe) * p.pan * kPanelBytes + p.w_slots * p.w_slot_bytes + p.p_slots * p.p_slot_bytes +
                           fixed_smem_bytes(p.nH, p.hdp, p.cp);
    if (smem_bytes > kSmemLimit) return ADSR_ERR_BAD_SHAPE;
    const int grid = p.n_tiles < num_sms ? p.n_tiles : num_sms;
    auto launch = [&](auto kernel) -> int {
        if (ensure_dynamic_smem(kernel, smem_bytes) != cudaSuccess) return ADSR_ERR_CUDA;
        return launch_pdl(kernel, dim3(grid), dim3(kThreads), static_cast<size_t>(smem_bytes), stream, p) == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
    };
    if (p.trace != nullptr) return p.fuse_proj ? launch(swin_attn_kernel<true, true>) : launch(swin_attn_kernel<true, false>);
    return p.fuse_proj ? launch(swin_attn_kernel<false, true>) : launch(swin_attn_kernel<false, false>);
}

}  // namespace adsr
