// tcgen05 / TMEM GEMM and implicit-GEMM 3x3 convolution for sm_100a.
//
// One persistent, warp-specialised kernel (grid = #SMs, 16 warps).  Per 128-row output tile the K dimension is
// streamed through a 4-deep shared-memory ring; each ring stage holds
//   * an A tile  [128 rows x 64 bf16]  (K-major, 128-byte swizzle): in GEMM mode it arrives by TMA
//     (cp.async.bulk.tensor, out-of-bounds K columns / M rows zero-filled by the hardware); in conv mode 4 producer
//     warps gather the 3x3 taps of an NHWC image with zero padding (implicit GEMM, im2col never materialised), and
//   * a  B tile  [BN rows  x 64 bf16]  = pre-swizzled weight image fetched with ONE bulk async copy per stage
//     (weights are packed once at load time into exactly the shared-memory image the tensor core wants).
// A single elected thread issues tcgen05.mma (M=128, N=BN<=256, K=16, bf16 -> fp32) into one of two TMEM accumulator
// buffers; 8 epilogue warps drain the other buffer with tcgen05.ld.  The row-owner thread does all the math in fp32
// (folded LayerNorm, bias, GELU / LeakyReLU / ReLU, alpha, residual), rounds once to bf16 and can emit the row's
// (sum, sum of squares) for the NEXT LayerNorm.
//
// This kernel has the TMA epilogue (row-major outputs with a residual, at 16-byte aligned columns, BN % 32 == 0): every
// warp owns a double-buffered 32x32 bf16 staging tile in the 64-byte-swizzle layout.  The residual tile is TMA-LOADED
// into it (one chunk ahead), the row owner adds it from shared memory and writes the result back in place, one lane
// TMA-STORES the box.  No address arithmetic, predicates or global load/store instructions in the hot loop; M / N edges
// are clipped by the TMA unit.  Every other output (no residual, PixelShuffle(2) stores, slab slices at 8-byte aligned
// columns) goes to the manual-epilogue kernel of tc_gemm_manual.cu; launch_tc_gemm below picks one of the two.
//
// Replaces (reference call sites): nn.Linear qkv/proj/fc1/fc2 (src/drct.py:278,300,185-188) with the LayerNorms in front
// of qkv / fc1 (src/drct.py:481,510), the 1x1 adjust convs (src/drct.py:334-374, 389-393), conv_after_body /
// conv_before_upsample / Upsample convs + PixelShuffle (src/drct.py:837,844-845,702-705) and every 3x3 conv of DRN.
#include "adsr_kernels.h"
#include "ptx.cuh"

namespace adsr {

namespace {

constexpr int kStages = 4;
constexpr int kAStageBytes = 128 * 128;       // 128 rows x 64 bf16
constexpr int kBStageBytes = 256 * 128;       // up to 256 rows x 64 bf16
constexpr int kNumThreads = 512;              // 16 warps: loader, MMA, TMEM alloc, spare, 8 epilogue, 4 producers
constexpr int kEpiWarps = 8;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kTmemCols = 512;                // 2 accumulator buffers x 256 fp32 columns
constexpr int kStageTileBytes = 32 * 64;      // 32 rows x 32 bf16 staging tile
constexpr int kRingBytes = kStages * (kAStageBytes + kBStageBytes);
constexpr int kStagingBytes = kEpiWarps * 2 * kStageTileBytes;     // double-buffered per warp
constexpr int kSmemBytes = kRingBytes + kStagingBytes + 512 /*barriers*/;

struct __align__(8) RingBarriers {
    uint64_t full[kStages];
    uint64_t empty[kStages];
    uint64_t tmem_full[2];
    uint64_t tmem_empty[2];
    uint64_t res_full[kEpiWarps][2];   // residual tile of a warp's staging buffer has landed
    uint32_t tmem_base;
};

// exact-erf GELU to 8e-7 absolute: erf(z) = 1 - 2^-p(z) with a degree-5 fit of p (z = |x|/sqrt 2 folded
// into the coefficients), so gelu(x) = 0.5 * (x + |x| - |x| * 2^-q(|x|)): 5 FMA + 1 MUFU + 3.
__device__ __forceinline__ float gelu_erf(float x) {
    const float a = fabsf(x);
    float q = 4.88103149e-4f;                    // c5 / 2^2.5
    q = fmaf(q, a, -7.19872210e-3f);             // c4 / 4
    q = fmaf(q, a, 5.21466284e-2f);              // c3 / 2^1.5
    q = fmaf(q, a, 4.59595859e-1f);              // c2 / 2
    q = fmaf(q, a, 1.15100050e+0f);              // c1 / sqrt 2
    const float e = exp2f(-q * a);
    return 0.5f * (x + fmaf(-a, e, a));
}

template <int ACT>
__device__ __forceinline__ float apply_act(float v, float slope) {
    if constexpr (ACT == ADSR_ACT_LRELU) return v > 0.f ? v : v * slope;
    if constexpr (ACT == ADSR_ACT_GELU) return gelu_erf(v);
    if constexpr (ACT == ADSR_ACT_RELU) return fmaxf(v, 0.f);
    return v;
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

// TMA store of a 2-D box from shared memory (bulk async group) and the group bookkeeping
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {      // <= N most recent groups may still be READING shared memory
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

template <int ACT, bool STATS>
__global__ void __launch_bounds__(kNumThreads, 1) tc_gemm_kernel(const __grid_constant__ TcGemmParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + kStages * kAStageBytes;
    uint8_t* smem_stg = smem + kRingBytes;                                   // [8 warps][2][32 rows][64 B]
    RingBarriers* bars = reinterpret_cast<RingBarriers*>(smem_stg + kStagingBytes);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    // Tile schedule (identical in every warp role): tiles are dealt round-robin (tile = it * grid + cta) with N fastest,
    // so the N tiles of one row block run on neighbouring CTAs at the same time and share the A tile through L2.
    const int total_tiles = p.m_tiles * p.n_tiles;
    const int my_tiles = blockIdx.x < total_tiles ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
#define ADSR_TILE_COORDS(it_)                                                            \
    const int lin_ = (it_) * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x); \
    const int m_tile = lin_ / p.n_tiles;                                                  \
    const int n_tile = lin_ % p.n_tiles;

    if ((smem_u32(smem) & 1023u) != 0) __trap();   // swizzle-128B operands need 1024 B alignment

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&bars->full[s], p.use_tma ? 1 : 128 + 1);   // (128 producer threads +) the copy issuer
            mbar_init(&bars->empty[s], 1);                         // one tcgen05.commit
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&bars->tmem_full[b], 1);
            mbar_init(&bars->tmem_empty[b], kEpiThreads);
        }
        for (int w = 0; w < kEpiWarps; ++w) {
            mbar_init(&bars->res_full[w][0], 1);
            mbar_init(&bars->res_full[w][1], 1);
        }
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc<kTmemCols>(&bars->tmem_base);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == 0) {
        // ================================ loader: TMA A tile + bulk-copied B tile per ring stage =====
        {   // converged warp, one elected lane issues (keeps descriptors in uniform registers)
            const uint32_t b_bytes = static_cast<uint32_t>(p.BN) * 128u;
            const uint32_t tx_bytes = b_bytes + (p.use_tma ? static_cast<uint32_t>(kAStageBytes) : 0u);
            if (p.use_tma && lane == 0) tma_prefetch_desc(&p.tmap_a);
            int stage = 0;
            uint32_t phase = 0;
            for (int it = 0; it < my_tiles; ++it) {
                ADSR_TILE_COORDS(it)
                const int m0 = m_tile * 128;
                const uint8_t* src = p.Bp + static_cast<size_t>(n_tile) * p.num_k_stages * b_bytes;
                for (int ks = 0; ks < p.num_k_stages; ++ks) {
                    mbar_wait(&bars->empty[stage], phase ^ 1);
                    if (elect_one_sync()) {
                        mbar_arrive_expect_tx(&bars->full[stage], tx_bytes);
                        if (p.use_tma) tma_load_2d(smem_a + stage * kAStageBytes, &p.tmap_a, ks * 64, m0, &bars->full[stage]);
                        bulk_g2s(smem_b + stage * kBStageBytes, src + static_cast<size_t>(ks) * b_bytes, b_bytes,
                                 &bars->full[stage]);
                    }
                    __syncwarp();
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer (single thread) ================================
        {   // converged warp, one elected lane issues
            const uint32_t idesc = umma_idesc_bf16_m128(static_cast<uint32_t>(p.BN));
            int stage = 0;
            uint32_t phase = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const int buf = it & 1;
                const uint32_t use = static_cast<uint32_t>(it >> 1);
                mbar_wait(&bars->tmem_empty[buf], (use & 1) ^ 1);
                tc_fence_after_sync();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(buf * 256);
                for (int ks = 0; ks < p.num_k_stages; ++ks) {
                    int steps;
                    if (p.conv) {
                        steps = p.k16_per_tap - 4 * (ks % p.stages_per_tap);
                    } else {
                        steps = p.k16_total - 4 * ks;
                    }
                    steps = steps > 4 ? 4 : steps;
                    mbar_wait(&bars->full[stage], phase);
                    tc_fence_after_sync();
                    const uint64_t adesc = umma_desc_k_sw128(smem_u32(smem_a + stage * kAStageBytes));
                    const uint64_t bdesc = umma_desc_k_sw128(smem_u32(smem_b + stage * kBStageBytes));
                    if (elect_one_sync()) {
                        // advance 16 bf16 = 32 B along K inside the 128 B swizzle row: +2 in 16-byte units
                        umma_bf16(d_tmem, adesc, bdesc, idesc, ks != 0 ? 1u : 0u);
                        if (steps > 1) umma_bf16(d_tmem, adesc + 2, bdesc + 2, idesc, 1u);
                        if (steps > 2) umma_bf16(d_tmem, adesc + 4, bdesc + 4, idesc, 1u);
                        if (steps > 3) umma_bf16(d_tmem, adesc + 6, bdesc + 6, idesc, 1u);
                        umma_commit(&bars->empty[stage]);      // frees the ring slot when the MMAs retire
                        if (ks == p.num_k_stages - 1) umma_commit(&bars->tmem_full[buf]);   // accumulator complete -> epilogue
                    }
                    __syncwarp();
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp >= 4 && warp < 4 + kEpiWarps) {
        // ================================ epilogue ====================================================
        // quadrant q = warp & 3 owns TMEM lanes / tile rows 32q..32q+31 (thread = row); the two warps of a quadrant take
        // alternate 32-column chunks.
        const int ew = warp - 4;
        const int quad = warp & 3;
        const int half = ew >> 2;
        uint8_t* stg = smem_stg + ew * 2 * kStageTileBytes;    // this warp's two staging tiles
        const int wsw = (lane >> 1) & 3;                       // 64-byte swizzle phase of my row
        const int n_chunks = (p.BN + 31) >> 5;
        const bool has_res = p.res != nullptr;
        int g = 0;                                             // chunks processed by this warp (staging buffer = g & 1)

        // (tile index, chunk) of the first chunk at or after (it, ch) that this warp really stores
        auto next_chunk = [&](int it, int ch, int& it_out, int& ch_out) -> bool {
            while (it < my_tiles) {
                const int lin = it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
                const int nb = (lin % p.n_tiles) * p.BN;
                const int lim = min(p.n_store, nb + p.BN);
                if (ch < n_chunks && nb + ch * 32 < lim) { it_out = it; ch_out = ch; return true; }
                ++it;
                ch = half;
            }
            return false;
        };
        auto issue_res_load = [&](int it, int ch, int bufi) {     // lane 0 only
            const int lin = it * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
            const int mt = lin / p.n_tiles, nt = lin % p.n_tiles;
            uint64_t* bar = &bars->res_full[ew][bufi];
            mbar_arrive_expect_tx(bar, kStageTileBytes);
            tma_load_2d(stg + bufi * kStageTileBytes, &p.tmap_res, nt * p.BN + ch * 32, mt * 128 + quad * 32, bar);
        };
        if (has_res && lane == 0) {
            int it0, ch0;
            if (next_chunk(0, half, it0, ch0)) issue_res_load(it0, ch0, 0);
        }

        for (int it = 0; it < my_tiles; ++it) {
            ADSR_TILE_COORDS(it)
            const int buf = it & 1;
            const uint32_t use = static_cast<uint32_t>(it >> 1);
            const int n_base = n_tile * p.BN;
            const int n_lim = min(p.n_store, n_base + p.BN);   // never write into the next N tile's columns
            const int row0 = m_tile * 128 + quad * 32;
            const int row = row0 + lane;                       // the row this thread owns
            const bool row_ok = row < p.M;
            // LayerNorm statistics of my row: partial (sum, sumsq) slots written by the producing kernel(s)
            float ln_mean = 0.f, ln_rstd = 1.f;
            if (p.ln_fold && row_ok) {
                const float2* sp = p.stats_in + static_cast<long long>(row) * p.stats_in_stride;
                float s1 = 0.f, s2 = 0.f;
                for (int k = 0; k < p.stats_in_slots; ++k) {
                    const float2 v = __ldg(sp + k);
                    s1 += v.x;
                    s2 += v.y;
                }
                const float inv_c = 1.0f / static_cast<float>(p.ln_C);
                ln_mean = s1 * inv_c;
                ln_rstd = rsqrtf(fmaxf(s2 * inv_c - ln_mean * ln_mean, 0.f) + p.ln_eps);
            }
            mbar_wait(&bars->tmem_full[buf], use & 1);
            tc_fence_after_sync();
            const uint32_t taddr = tmem_base + static_cast<uint32_t>(buf * 256) + (static_cast<uint32_t>(quad * 32) << 16);
            float st_sum = 0.f, st_sq = 0.f;

            for (int ch = half; ch < n_chunks; ch += 2) {
                const int c0 = ch * 32;
                const int n0 = n_base + c0;
                if (n0 >= n_lim) continue;                      // warp-uniform: nothing of this chunk is stored
                uint8_t* sbuf = stg + (g & 1) * kStageTileBytes;
                const uint32_t sbuf_row = smem_u32(sbuf) + static_cast<uint32_t>(lane * 64);

                uint32_t raw[32];
                __syncwarp();                                   // tcgen05.ld is .sync.aligned
                tmem_ld32(taddr + static_cast<uint32_t>(c0), raw);
                tmem_ld_wait();

                if (has_res) {
                    // prefetch the residual tile of my NEXT chunk into the other staging buffer; the store that last
                    // used that buffer (chunk g-1) must have finished reading it
                    if (lane == 0) {
                        int it2, ch2;
                        if (next_chunk(it, ch + 2, it2, ch2)) {
                            bulk_wait_read<0>();
                            issue_res_load(it2, ch2, (g + 1) & 1);
                        }
                    }
                    mbar_wait(&bars->res_full[ew][g & 1], static_cast<uint32_t>(g >> 1) & 1);   // my residual tile landed
                } else {
                    if (lane == 0) bulk_wait_read<1>();         // the store of chunk g-2 has finished reading this buffer
                    __syncwarp();
                }

                // ---- fp32 math per element, one rounding to bf16; logical 16-byte chunk j of my row holds columns 8j..8j+7
                uint32_t pk[16];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint32_t rw[4] = {0u, 0u, 0u, 0u};
                    if (has_res) {
                        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                                     : "=r"(rw[0]), "=r"(rw[1]), "=r"(rw[2]), "=r"(rw[3])
                                     : "r"(sbuf_row + static_cast<uint32_t>((j ^ wsw) << 4)));
                    }
#pragma unroll
                    for (int h2 = 0; h2 < 2; ++h2) {
                        const int q4 = 2 * j + h2;              // group of 4 columns
                        const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + 4 * q4));   // L1-resident, warp-uniform
                        float a[4] = {__uint_as_float(raw[4 * q4 + 0]), __uint_as_float(raw[4 * q4 + 1]),
                                      __uint_as_float(raw[4 * q4 + 2]), __uint_as_float(raw[4 * q4 + 3])};
                        const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
                        if (p.ln_fold) {                        // LN(x) W^T = rstd * (x W'^T - mean * colsum)
                            const float4 cs = __ldg(reinterpret_cast<const float4*>(p.colsum + n0 + 4 * q4));
                            const float cv[4] = {cs.x, cs.y, cs.z, cs.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e) a[e] = ln_rstd * fmaf(-ln_mean, cv[e], a[e]);
                        }
                        float v[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            v[e] = apply_act<ACT>(a[e] + bv[e], p.slope) * p.alpha;
                            if (has_res) {
                                const uint32_t w2 = rw[2 * h2 + (e >> 1)];
                                v[e] += (e & 1) ? bf16_hi(w2) : bf16_lo(w2);
                            }
                            // (columns >= N need no masking: zero weight rows, zero bias / colsum and a zero-filled
                            //  residual make them exact zeros, and act(0) = 0 for every activation used)
                            if (STATS) { st_sum += v[e]; st_sq = fmaf(v[e], v[e], st_sq); }
                        }
                        pk[2 * q4] = pack_bf16x2(v[0], v[1]);
                        pk[2 * q4 + 1] = pack_bf16x2(v[2], v[3]);
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(sbuf_row + static_cast<uint32_t>((j ^ wsw) << 4)),
                                 "r"(pk[4 * j]), "r"(pk[4 * j + 1]), "r"(pk[4 * j + 2]), "r"(pk[4 * j + 3])
                                 : "memory");
                }

                fence_proxy_async_smem();                       // my st.shared must be visible to the TMA (async proxy)
                __syncwarp();
                if (lane == 0) {
                    tma_store_2d(&p.tmap_out, sbuf, p.ocol0 + n0, row0);   // rows >= M / columns >= ocol0+n_store clipped
                    bulk_commit();
                }
                ++g;
            }
            // partial LayerNorm statistics of my row for the consumer of this output (deterministic slot, no atomics)
            if (STATS && row_ok)
                p.stats_out[static_cast<long long>(row) * p.stats_out_stride + p.stats_out_slot0 + n_tile * 2 + half] =
                    make_float2(st_sum, st_sq);
            __syncwarp();
            tc_fence_before_sync();
            mbar_arrive(&bars->tmem_empty[buf]);
        }
        if (lane == 0) bulk_wait_all();                         // all my stores have left shared memory and are complete
    } else if (warp >= 4 + kEpiWarps && !p.use_tma) {
        // ================================ conv mode: A producers (4 warps, 128 threads) ===============
        const int pw = warp - (4 + kEpiWarps);
        const int chunk = lane & 7;                            // 16-byte chunk inside the 128 B row
        const int rsub = pw * 4 + (lane >> 3);                 // row inside each 16-row step
        const uint32_t sw_off = static_cast<uint32_t>(rsub * 128 + ((chunk ^ (rsub & 7)) << 4));
        int stage = 0;
        uint32_t phase = 0;
        for (int it = 0; it < my_tiles; ++it) {
            ADSR_TILE_COORDS(it)
            (void)n_tile;
            const int m0 = m_tile * 128;
            // per-row source bookkeeping (8 rows per thread: r = step*16 + rsub)
            long long row_off[8];
            int oy[8], ox[8];
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                const int m = m0 + s * 16 + rsub;
                if (m >= p.M) {
                    row_off[s] = -1; oy[s] = 0; ox[s] = 0;
                } else if (p.conv) {
                    const int hw = p.Hout * p.Wout;
                    const int b = m / hw;
                    const int rem = m - b * hw;
                    oy[s] = rem / p.Wout;
                    ox[s] = rem - oy[s] * p.Wout;
                    row_off[s] = static_cast<long long>(b) * p.Hin * p.Win;   // pixel index of image start
                } else {
                    row_off[s] = static_cast<long long>(m) * p.lda; oy[s] = 0; ox[s] = 0;
                }
            }
            for (int ks = 0; ks < p.num_k_stages; ++ks) {
                uint4 v[8];
                if (p.conv) {
                    const int tap = ks / p.stages_per_tap;
                    const int col = (ks - tap * p.stages_per_tap) * 64 + chunk * 8;
                    const int dy = tap / 3 - 1, dx = tap % 3 - 1;
                    const bool col_ok = col < p.K8;
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        const int iy = oy[s] * p.stride + dy, ix = ox[s] * p.stride + dx;
                        const bool ok = col_ok && row_off[s] >= 0 && iy >= 0 && iy < p.Hin && ix >= 0 && ix < p.Win;
                        if (ok) {
                            const long long pix = row_off[s] + static_cast<long long>(iy) * p.Win + ix;
                            v[s] = __ldg(reinterpret_cast<const uint4*>(p.A + pix * p.lda + col));
                        } else {
                            v[s] = make_uint4(0, 0, 0, 0);
                        }
                    }
                } else {
                    const int col = ks * 64 + chunk * 8;
                    const bool col_ok = col < p.K8;
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        if (col_ok && row_off[s] >= 0) {
                            v[s] = __ldg(reinterpret_cast<const uint4*>(p.A + row_off[s] + col));
                        } else {
                            v[s] = make_uint4(0, 0, 0, 0);
                        }
                    }
                }
                mbar_wait(&bars->empty[stage], phase ^ 1);
                uint8_t* dst = smem_a + stage * kAStageBytes + sw_off;
#pragma unroll
                for (int s = 0; s < 8; ++s) *reinterpret_cast<uint4*>(dst + s * 16 * 128) = v[s];
                fence_proxy_async_smem();
                mbar_arrive(&bars->full[stage]);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after_sync();
        tmem_dealloc<kTmemCols>(tmem_base);
    }
}

using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                              const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode_fn() {
    static EncodeFn encode = nullptr;
    if (encode == nullptr) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess || fn == nullptr)
            return nullptr;
        encode = reinterpret_cast<EncodeFn>(fn);
    }
    return encode;
}

int encode_2d(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld_elems, int box_cols,
              int box_rows, CUtensorMapSwizzle swz) {
    EncodeFn encode = get_encode_fn();
    if (encode == nullptr) return ADSR_ERR_CUDA;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld_elems) * 2};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? ADSR_OK : ADSR_ERR_CUDA;
}

}  // namespace

int encode_tmap_rows_bf16(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld_elems) {
    return encode_2d(map, base, rows, cols, ld_elems, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B);
}

// token rows viewed as the NHWC image [B, H, W, C]: boxes of R x R tokens x 64 channels (the window pieces of swin_attn.cu);
// a box lands as R*R rows of 128 bytes (x fastest) in the 128-byte-swizzle operand layout
int encode_tmap_nhwc_box_bf16(CUtensorMap* map, const void* base, int B, int H, int W, int C, long long ld_elems, int R) {
    return encode_tmap_nhwc_box2_bf16(map, base, B, H, W, C, ld_elems, R, R);
}

// general form: boxes of box_w x box_h tokens x 64 channels (box_w tokens of a row are contiguous in shared memory)
int encode_tmap_nhwc_box2_bf16(CUtensorMap* map, const void* base, int B, int H, int W, int C, long long ld_elems, int box_w, int box_h) {
    return encode_tmap_nhwc_box3_bf16(map, base, B, H, W, C, ld_elems, 64, box_w, box_h);
}

// box_c channels per token: 64 (128-byte swizzle), 32 (64-byte swizzle) or 16 (32-byte swizzle) -- the swizzle span equals the row
int encode_tmap_nhwc_box3_bf16(CUtensorMap* map, const void* base, int B, int H, int W, int C, long long ld_elems, int box_c, int box_w,
                               int box_h) {
    EncodeFn encode = get_encode_fn();
    if (encode == nullptr) return ADSR_ERR_CUDA;
    const CUtensorMapSwizzle sw = box_c == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : box_c == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    if (box_c != 64 && box_c != 32 && box_c != 16) return ADSR_ERR_BAD_SHAPE;
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(B)};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(ld_elems) * 2, static_cast<cuuint64_t>(ld_elems) * 2 * W,
                                   static_cast<cuuint64_t>(ld_elems) * 2 * W * H};
    const cuuint32_t box[4] = {static_cast<cuuint32_t>(box_c), static_cast<cuuint32_t>(box_w), static_cast<cuuint32_t>(box_h), 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? ADSR_OK : ADSR_ERR_CUDA;
}

// 32 x 32 bf16 boxes in the 64-byte-swizzle layout of the epilogue staging tiles (residual loads / output stores)
int encode_tmap_epilogue_bf16(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld_elems) {
    return encode_2d(map, base, rows, cols, ld_elems, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B);
}

int launch_tc_gemm(TcGemmParams& p, int num_sms, cudaStream_t stream) {
    if (p.M <= 0) return ADSR_OK;
    if (p.BN < 16 || p.BN > 256 || (p.BN % 16) != 0) return ADSR_ERR_BAD_SHAPE;
    if ((p.lda % 8) != 0 || (p.ldo % 4) != 0 || (p.ocol0 % 4) != 0) return ADSR_ERR_BAD_SHAPE;
    if ((reinterpret_cast<uintptr_t>(p.A) & 15) || (reinterpret_cast<uintptr_t>(p.Bp) & 15)) return ADSR_ERR_BAD_ALIGN;
    if (p.res != nullptr && ((p.ldres % 8) != 0 || (reinterpret_cast<uintptr_t>(p.res) & 15))) return ADSR_ERR_BAD_ALIGN;
    if (p.out_mode == ADSR_OUT_ROWS && (p.ocol0 % 8) == 0 &&
        ((reinterpret_cast<uintptr_t>(p.out) & 15) || (p.ldo % 8) != 0))
        return ADSR_ERR_BAD_ALIGN;
    if (p.num_k_stages <= 0 || p.n_tiles <= 0 || (p.n_store % 4) != 0) return ADSR_ERR_BAD_SHAPE;
    if (p.ln_fold && (p.colsum == nullptr || p.stats_in == nullptr || p.ln_C <= 0 || p.stats_in_slots <= 0)) return ADSR_ERR_BAD_SHAPE;
    if (p.stats_out != nullptr && p.out_mode != ADSR_OUT_ROWS) return ADSR_ERR_BAD_SHAPE;
    if (p.out_mode == ADSR_OUT_PIXEL_SHUFFLE2 &&
        ((p.BN % 32) != 0 || (p.ldo % 8) != 0 || (reinterpret_cast<uintptr_t>(p.out) & 15)))
        return ADSR_ERR_BAD_SHAPE;

    // short-K row outputs packed with BN = 128: the row-tile kernel (tc_gemm_rows.cu)
    if (tc_gemm_rows_eligible(p)) return launch_tc_gemm_rows(p, num_sms, stream);

    // TMA epilogue when there is a residual to add (row-major output at a 16-byte aligned column, chunks never straddle
    // N tiles).  Without a residual the manual epilogue is faster today: with two staging tiles per warp the TMA-store
    // latency caps the store bandwidth of wide outputs (measured 1.9 vs 2.4 TB/s on the qkv shape).
    p.epi_tma = (p.res != nullptr && p.out_mode == ADSR_OUT_ROWS && (p.ocol0 % 8) == 0 && (p.BN % 32) == 0 &&
                 (p.n_store % 8) == 0) ? 1 : 0;
    if (p.epi_tma) {
        int st = encode_tmap_epilogue_bf16(&p.tmap_out, p.out, p.M, p.ocol0 + p.n_store, p.ldo);
        if (st != ADSR_OK) return st;
        if (p.res != nullptr) {
            st = encode_tmap_epilogue_bf16(&p.tmap_res, p.res, p.M, p.N, p.ldres);
            if (st != ADSR_OK) return st;
        }
    } else if (p.stats_out != nullptr && p.res != nullptr) {
        return ADSR_ERR_BAD_SHAPE;     // the manual epilogue adds the residual after the statistics are taken
    }

    const int units = p.m_tiles * p.n_tiles;
    const int grid = units < num_sms ? units : num_sms;
    // stride-1 convolutions whose 128-pixel tiles are whole image rows: the A stages come by 4-D TMA boxes (manual-epilogue kernel)
    p.conv_tma = 0;
    if (p.conv && p.stride == 1 && p.Hout == p.Hin && p.Wout == p.Win && p.Win <= 128 && (128 % p.Win) == 0 &&
        ((p.Hin * p.Win) % 128) == 0 && !p.ln_fold && p.stats_out == nullptr && (reinterpret_cast<uintptr_t>(p.A) & 15) == 0) {
        const int B = p.M / (p.Hin * p.Win);
        if (encode_tmap_nhwc_box2_bf16(&p.tmap_a, p.A, B, p.Hin, p.Win, p.K8, p.lda, p.Win, 128 / p.Win) == ADSR_OK) {
            p.conv_tma = 1;
            p.epi_tma = 0;
            return launch_tc_gemm_manual(p, grid, stream);
        }
    }
    auto launch = [&](auto kernel) -> int {
        if (ensure_dynamic_smem(kernel, kSmemBytes) != cudaSuccess) return ADSR_ERR_CUDA;
        kernel<<<grid, kNumThreads, kSmemBytes, stream>>>(p);
        return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
    };
    if (!p.epi_tma) return launch_tc_gemm_manual(p, grid, stream);
    const bool st = p.stats_out != nullptr;
    switch (p.act) {
        case ADSR_ACT_NONE: return st ? launch(tc_gemm_kernel<ADSR_ACT_NONE, true>) : launch(tc_gemm_kernel<ADSR_ACT_NONE, false>);
        case ADSR_ACT_LRELU: return st ? launch(tc_gemm_kernel<ADSR_ACT_LRELU, true>) : launch(tc_gemm_kernel<ADSR_ACT_LRELU, false>);
        case ADSR_ACT_GELU: return st ? launch(tc_gemm_kernel<ADSR_ACT_GELU, true>) : launch(tc_gemm_kernel<ADSR_ACT_GELU, false>);
        case ADSR_ACT_RELU: return st ? launch(tc_gemm_kernel<ADSR_ACT_RELU, true>) : launch(tc_gemm_kernel<ADSR_ACT_RELU, false>);
    }
    return ADSR_ERR_BAD_SHAPE;
}

}  // namespace adsr
