// Internal declarations shared by the .cu translation units (not part of the public C ABI).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/adsr_b200.h"

namespace adsr {

// Opt-in dynamic shared memory of a kernel: only ever RAISED.  The limit is per-function state, not part of a launch: a launcher that
// sets it to each launch's own size leaves the LAST size behind, and a tool that re-launches the kernel nodes of a captured CUDA graph
// one by one (ncu) then fails the nodes that need more than the last captured launch did.
template <typename Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, int bytes) {
    cudaFuncAttributes attr;
    const cudaError_t e = cudaFuncGetAttributes(&attr, kernel);
    if (e != cudaSuccess) return e;
    if (attr.maxDynamicSharedSizeBytes >= bytes) return cudaSuccess;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}


// Programmatic dependent launch (PDL): the kernel may become resident while the previous kernel of the stream is still draining; it
// must execute pdl_wait() before touching anything the previous kernel wrote (or still reads).  Used by the three kernels of DRN's
// RCAB chain (320 of the 333 launches of a DRN-L step), whose prologues (barrier init, TMEM allocation, resident weights) then
// overlap the tail of their predecessor.  ADSR_PDL=0 in the environment falls back to plain stream order.
bool pdl_enabled();
template <typename Kernel, typename... Args>
inline cudaError_t launch_pdl(Kernel kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// SSIM of one pixel from its five window sums (x, y, x^2, y^2, xy) and 1 / (ws * ws), shared by the three scorer kernels
// (scoring.cu) and the 1 - SSIM map (anomaly_maps.cu).  Every operation is rounded on its own (no FMA contraction), so the kernels
// give the same bits for the same window sums, and for an identical pair (sums 0 == 1, 2 == 3 == 4) the numerator and the
// denominator are the same double: exactly 1.
__device__ __forceinline__ double ssim_term(const double (&sum)[5], double inv_n, double C1, double C2) {
    const double mu1 = __dmul_rn(sum[0], inv_n), mu2 = __dmul_rn(sum[1], inv_n);
    const double m11 = __dmul_rn(mu1, mu1), m22 = __dmul_rn(mu2, mu2), m12 = __dmul_rn(mu1, mu2);
    const double s1 = __dsub_rn(__dmul_rn(sum[2], inv_n), m11), s2 = __dsub_rn(__dmul_rn(sum[3], inv_n), m22),
                 s12 = __dsub_rn(__dmul_rn(sum[4], inv_n), m12);
    return __ddiv_rn(__dmul_rn(__dadd_rn(__dmul_rn(2.0, m12), C1), __dadd_rn(__dmul_rn(2.0, s12), C2)),
                     __dmul_rn(__dadd_rn(__dadd_rn(m11, m22), C1), __dadd_rn(__dadd_rn(s1, s2), C2)));
}
#endif

struct TcGemmParams {
    CUtensorMap tmap_a;    // GEMM mode: [M rows x K cols] bf16, box 128 x 64, 128-byte swizzle (first: 64 B aligned)
    CUtensorMap tmap_out;  // TMA epilogue: output  [M x (ocol0 + n_store)], box 32 x 32, 64-byte swizzle
    CUtensorMap tmap_res;  // TMA epilogue: residual [M x N], same box (columns >= N read as zero)
    int use_tma;           // 1 = A tiles arrive by TMA (GEMM), 0 = producer warps gather them (conv)
    int conv_tma;          // conv, stride 1, 128-pixel tiles made of whole image rows: tmap_a is the NHWC image [B, H, W, C] and every
                           // (tap, channel panel) stage is ONE 4-D TMA box shifted by the tap (zero fill outside the image)
    int epi_tma;           // set by launch_tc_gemm: 1 = TMA epilogue, 0 = manual epilogue
    // A operand: token rows (GEMM) or NHWC image (implicit-GEMM conv)
    const __nv_bfloat16* A;
    long long lda;       // row / pixel pitch in elements (multiple of 8)
    int M;               // output rows (tokens or output pixels)
    int K8;              // readable K columns per row (GEMM) or channels per pixel (conv), rounded up to 8
    int num_k_stages;    // 64-wide K stages streamed per tile
    int k16_total;       // GEMM: number of K=16 MMA steps
    int conv;            // 0 = GEMM, 1 = 3x3 conv
    int Hin, Win, Hout, Wout, stride;
    int stages_per_tap, k16_per_tap;
    // B operand: packed weight image
    const uint8_t* Bp;
    int n_tiles, BN, m_tiles;
    // LayerNorm folded into the GEMM: A holds RAW rows, the weights carry gamma, the epilogue applies
    //   out = rstd_m * (acc - mean_m * colsum_n) + bias_n
    // with (sum, sumsq) of row m read from `stats_in` (stats_in_slots partial slots per row, written by the
    // epilogue(s) of the kernel(s) that produced A).
    int ln_fold;          // 0 / 1
    int ln_C;             // number of columns the statistics run over (= K)
    float ln_eps;
    const float* colsum;  // [n_tiles * BN]  s_n = sum_k gamma_k W_nk (of the bf16-rounded packed weights)
    const float2* stats_in;
    int stats_in_slots, stats_in_stride;
    // producer side: per-row partial (sum, sumsq) of THIS kernel's output -> stats_out[row*stride + slot0 + n_tile*2 + half]
    float2* stats_out;
    int stats_out_slot0, stats_out_stride;
    // epilogue
    const float* bias;
    int N, n_store, act;
    float slope, alpha;
    const __nv_bfloat16* res;
    long long ldres;
    __nv_bfloat16* out;
    long long ldo;
    int ocol0, out_mode;
    int rev_tiles;       // row-tile kernel: walk the M tiles from the last one down (the rows the producer of A wrote last are still in L2)
};

int launch_tc_gemm(TcGemmParams& p, int num_sms, cudaStream_t stream);
int launch_tc_gemm_manual(const TcGemmParams& p, int grid, cudaStream_t stream);   // tc_gemm_manual.cu
bool tc_gemm_rows_eligible(const TcGemmParams& p);                                  // tc_gemm_rows.cu
int launch_tc_gemm_rows(TcGemmParams& p, int num_sms, cudaStream_t stream);
// Encodes the TMA descriptor of a row-major bf16 matrix (driver entry point resolved at run time).
int encode_tmap_rows_bf16(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld_elems);

// ---- tcgen05 window attention for 8x8 windows (attention_tc.cu); ADSR_ERR_BAD_SHAPE = shape not covered, use the mma.sync kernel
int launch_window_attention_tc(const void* qkv, long long ldq, void* out, long long ldo, const float* table, int B, int H, int W,
                               int shift, int nH, int hd, int hdp, int num_sms, cudaStream_t stream);

// ---- tcgen05 window attention for 16x16 windows (attention_tc16.cu: DRCT-L at 64 px LR); ADSR_ERR_BAD_SHAPE = shape not covered
int launch_window_attention_tc16(const void* qkv, long long ldq, void* out, long long ldo, const float* table, int B, int H, int W,
                                 int shift, int nH, int hd, int hdp, int num_sms, cudaStream_t stream);

// ---- fused Swin MLP (swin_mlp.cu)
struct SwinMlpParams {
    CUtensorMap tmap_y;   // [M x C] bf16, box 64 x 128, 128-byte swizzle (loads)
    CUtensorMap tmap_z;   // same geometry on the output (stores)
    const uint8_t* w1p;   // fc1 slabs [hcw[j] rows x 64 bf16] in (chunk j, K slab s) order
    const uint8_t* w2p;   // fc2 slabs [piece rows x 64 bf16] in (chunk j, K slab s, piece) order
    const float* bias1;   // [nc * hc]  beta W1^T + b1, chunk-strided
    const float* colsum1; // [nc * hc]  sum_k gamma_k W1[n,k] of the bf16-rounded packed weights
    const float* bias2;   // [n2]
    const float2* stats_in;
    int stats_in_slots, stats_in_stride;
    float ln_eps;
    int C, M, m_tiles;
    float inv_c;          // 1 / C (set by the launcher)
    int rev;              // walk the row tiles from the last one down (what the producer wrote last is still in L2)
    int ks1, k1steps;     // 64-wide panels / K=16 steps of the y tile
    int nc, hc;           // hidden chunks, chunk stride in bias1 / colsum1 (= TMEM columns per fc1 accumulator)
    int hcw[8];           // MMA N of each chunk (multiple of 16, <= 128)
    int n2;               // fc2 accumulator columns (C rounded up to 16)
    int n_pieces;         // the fc2 N dimension is issued in 1 or 2 pieces (each <= 256 rows)
    int piece_rows[2], piece_col[2];
    int acc1_col[3];      // TMEM columns of the fc1 chunk accumulators ([2] = [1] + hc, used when n_acc1 == 3)
    int n_acc1;           // 2 or 3 (set by the launcher)
    // wide folded 1x1 conv WITH residual (adjust5 of the RDG, src/drct.py:394-396: x + 0.2 adjust5(z)):
    //   out[:, :c_out] = res[:, :c_out] + y W_a^T + g (W_a W2)^T + bias2   (the conv's scale and both biases folded in on the host);
    // W_a leads the fc2 ring of every tile as (K slab, N piece) slabs, the residual tile replaces the consumed y tile in shared memory,
    // the last epilogue adds it in place and also leaves the row's (sum, sumsq) in adj_stats (optional).  z itself never exists.
    int fold_res;
    int ypre[8];          // W_a slabs issued in front of chunk j (set by the launcher)
    int c_out;
    const __nv_bfloat16* res;
    long long ld_res;
    CUtensorMap tmap_res;
    int adjy_fc1;         // folded adjust: the fc1 (1) or the fc2 (0) issuer starts the accumulator with y W_adj^T (set by the launcher)
    int w1_slots, w1_slot_bytes, w2_slots, w2_slot_bytes, a_buf_bytes;
    long long* trace;     // optional [4 roles][8 tiles][64][8] clock64 timeline of CTA 0 (tools/mlp_trace.py), else nullptr
    // optional adjust 1x1 conv (src/drct.py:389-393) FOLDED into fc2: adj_out[:, adj_col0 + n] = LReLU(z W_adj^T + b)[n], n < 32, computed
    // as y W_adj^T + g (W_adj W2)^T + (b_adj + W_adj b2): the fc2 ring carries the 32 rows of W_adj W2 (n2 = 32), the accumulator
    // starts with y W_adj^T, and z itself never exists
    int fuse_adj;
    const uint8_t* wadj;  // ks1 slabs [32 rows x 64 bf16], 128-byte swizzle; resident in shared memory
    const float* bias_adj;   // [32]
    __nv_bfloat16* adj_out;
    long long ld_adj;
    int adj_col0;
    float adj_slope;
    float2* adj_stats;    // per-row (sum, sumsq) of the 32 new columns -> adj_stats[row * stride + slot0] (slot0 + 1 is zeroed)
    int adj_stats_slot0, adj_stats_stride;
    int adj_stats_vec4;   // the two slots of a row form one aligned 16-byte store (set by the launcher)
};
int swin_mlp_fixed_smem_bytes(int hidden_padded, int n2);
int launch_swin_mlp(SwinMlpParams& p, const void* y, long long ldy, void* z, long long ldz, int num_sms, cudaStream_t stream);

// ---- fused attention half of a Swin block (swin_attn.cu)
struct SwinAttnParams {
    CUtensorMap tmap_x;       // x as [B, H, W, C] bf16, box 64 channels x R x R tokens, 128-byte swizzle (x-tile loads)
    const __nv_bfloat16* x;   // [M, >= C] raw token rows: A operand of the (norm1-folded) qkv Linear and the shortcut
    long long ldx;
    __nv_bfloat16* out;       // fuse_proj: y [M, >= C] = x + proj(attention);  else attention rows [M, nH * hdp]
    long long ldo;
    const uint8_t* w1p;       // qkv slabs [3 hdp rows (q_h | k_h | v_h) x 64 bf16] in (head, K slab) order, gamma folded
    const uint8_t* w2p;       // proj slabs [cp rows x 64 bf16] (K = the head's hdp channels), one per head
    const float* bias_qkv;    // [nH * 3 * hdp]  W beta + b in the slab row order
    const float* colsum_qkv;  // [nH * 3 * hdp]  sum_k gamma_k W_nk of the bf16-rounded packed weights
    const float* bias_p;      // [cp]
    const float* table;       // [225, nH] relative position bias table
    const float2* stats_in;   // per-row (sum, sumsq) partials of x
    int stats_in_slots, stats_in_stride;
    float2* stats_out;        // per-row (sum, sumsq) of y -> stats_out[row * stride + slot0]   (fuse_proj only; may be null)
    int stats_out_slot0, stats_out_stride;
    float ln_eps, scale_log2e;
    int B, H, W, C, shift, nH, hdp;
    int n_tiles;              // window pairs
    int box_r;                // side of the square token boxes a window is fetched in: 8 (no shift) or 4 (shift 4, wrapped windows)
    int ks, k16;              // 64-wide panels / K=16 steps of the x tile
    int pan;                  // 64-column panels per k / v operand
    int fuse_proj;
    int cp;                   // proj accumulator columns (C rounded up to 16)
    int n_pp, pp_rows[4];     // a head's proj slab is issued in n_pp N pieces (each fits a ring slot)
    int qkv_pieces, qp_rows[4];  // a qkv slab is one ring slot / issue step; two N pieces when 3 hdp > 256
    int rsz, nreg;            // TMEM: columns per head region, number of regions (2 = next head's q|k|v runs one head ahead)
    int col_o;                // TMEM column of O (fuse_proj: behind the region; else O overlays the region's q columns)
    int col_acc;              // fuse_proj with spare TMEM: separate q|k|v accumulator columns, else -1 (accumulators = the region)
    int pipe;                 // heads pipelined: convert(h + 1) between softmax(h) and normalise(h) (needs col_acc >= 0; second v panel)
    int early_setup;          // per-row tile set-up (token, mask bits, LayerNorm statistics) one tile ahead, under the first S wait
    int w_slots, w_slot_bytes;   // qkv weight ring
    int p_slots, p_slot_bytes;   // proj weight ring (fuse_proj)
    long long* trace;         // optional clock64 timeline of CTA 0 (tools/attn_trace.py), else nullptr
};
int encode_tmap_nhwc_box_bf16(CUtensorMap* map, const void* base, int B, int H, int W, int C, long long ld_elems, int R);
int encode_tmap_nhwc_box2_bf16(CUtensorMap* map, const void* base, int B, int H, int W, int C, long long ld_elems, int box_w, int box_h);
int encode_tmap_nhwc_box3_bf16(CUtensorMap* map, const void* base, int B, int H, int W, int C, long long ld_elems, int box_c, int box_w,
                               int box_h);
int swin_attn_plan(SwinAttnParams& p, int C, int nH, int hdp, int allow_proj);   // 0 = not covered, 1 = qkv + attention, 2 = + proj
int launch_swin_attn(SwinAttnParams& p, int num_sms, cudaStream_t stream);

// ---- halo-tile 3x3 conv with resident weights (conv_halo.cu)
struct ConvHaloParams {
    CUtensorMap tmap_in;      // input as [B, H, W, C] bf16, box 64 channels x (W + 2) x box_rows, 128-byte swizzle
    CUtensorMap tmap_tail;    // same image, box 16 channels, 32-byte swizzle: the last K = 16 step when Cin = 64 + (<= 16) channels
    const uint8_t* wp;        // slabs [BN rows x 64 bf16], K index = tap * 16 k16_per_tap + channel (compact), 128-byte swizzle
    const float* bias;        // [BN]
    __nv_bfloat16* out;
    long long ldo;
    int ocol0, n_store;
    float* chan_part;         // optional [n_tiles * 4, BN] per-(tile, row quadrant) column sums of the outputs (fp32, before bf16 rounding)
    int B, H, W, Cin, N, BN;
    int act;
    float slope;
    // set by launch_conv_halo
    int k16_per_tap, full_panels, tail, slabs, Wh, box_rows, box_bytes, panel_bytes, tail_box_bytes, tail_bytes, n_abuf, tiles_per_img,
        n_tiles;
};
int launch_conv_halo(ConvHaloParams& p, const void* in, long long ld_in, int num_sms, cudaStream_t stream);

}  // namespace adsr
