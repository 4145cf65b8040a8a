#include <cstdlib>
// extern "C" entry points that only marshal arguments (the kernels live in the other .cu files).
#include <string.h>

#include "adsr_kernels.h"

using namespace adsr;

extern "C" int adsr_abi_version(void) { return ADSR_ABI_VERSION; }

namespace adsr {
bool pdl_enabled() {
    static const bool on = [] {
        const char* e = getenv("ADSR_PDL");
        return !(e != nullptr && e[0] == '0');
    }();
    return on;
}
}  // namespace adsr

extern "C" const char* adsr_status_string(int status) {
    switch (status) {
        case ADSR_OK: return "ok";
        case ADSR_ERR_BAD_SHAPE: return "unsupported shape";
        case ADSR_ERR_BAD_ALIGN: return "misaligned pointer or pitch";
        case ADSR_ERR_LAUNCH: return "kernel launch failed";
        case ADSR_ERR_CUDA: return "CUDA runtime call failed";
        case ADSR_ERR_ARCH: return "device is not sm_100";
    }
    return "unknown status";
}

extern "C" int adsr_device_check(int* host_num_sms) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return ADSR_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return ADSR_ERR_CUDA;
    if (host_num_sms) *host_num_sms = prop.multiProcessorCount;
    return prop.major == 10 ? ADSR_OK : ADSR_ERR_ARCH;
}

extern "C" int adsr_tc_gemm_bf16(const void* A, int64_t lda, int M, int K, const void* w_packed, const float* bias_padded,
                                 int N, int BN, int n_tiles, int act, float slope, float alpha, const void* res,
                                 int64_t ldres, void* out, int64_t ldo, int ocol0, int n_store,
                                 const float* ln_colsum, float ln_eps, const float* ln_stats_in, int stats_in_slots,
                                 int stats_in_stride, float* stats_out, int stats_out_slot0, int stats_out_stride,
                                 int reverse_tiles, int num_sms, void* stream) {
    if (M <= 0) return ADSR_OK;
    if (K <= 0 || N <= 0 || n_store > n_tiles * BN || lda < K) return ADSR_ERR_BAD_SHAPE;
    TcGemmParams p{};
    p.rev_tiles = reverse_tiles != 0;
    p.A = static_cast<const __nv_bfloat16*>(A);
    p.lda = lda;
    p.M = M;
    p.K8 = (K + 7) & ~7;
    p.k16_total = (K + 15) / 16;
    p.num_k_stages = (K + 63) / 64;
    p.conv = 0;
    p.Hin = p.Win = p.Hout = p.Wout = 1;
    p.stride = 1;
    p.stages_per_tap = 1;
    p.k16_per_tap = 0;
    p.Bp = static_cast<const uint8_t*>(w_packed);
    p.n_tiles = n_tiles;
    p.BN = BN;
    p.m_tiles = (M + 127) / 128;
    p.bias = bias_padded;
    p.N = N;
    p.n_store = n_store;
    p.act = act;
    p.slope = slope;
    p.alpha = alpha;
    p.res = static_cast<const __nv_bfloat16*>(res);
    p.ldres = ldres;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.ldo = ldo;
    p.ocol0 = ocol0;
    p.out_mode = ADSR_OUT_ROWS;
    p.ln_fold = ln_colsum != nullptr;
    p.ln_C = K;
    p.ln_eps = ln_eps;
    p.colsum = ln_colsum;
    p.stats_in = reinterpret_cast<const float2*>(ln_stats_in);
    p.stats_in_slots = stats_in_slots;
    p.stats_in_stride = stats_in_stride;
    p.stats_out = reinterpret_cast<float2*>(stats_out);
    p.stats_out_slot0 = stats_out_slot0;
    p.stats_out_stride = stats_out_stride;
    if (p.ln_fold && ln_stats_in == nullptr) return ADSR_ERR_BAD_SHAPE;
    if (stats_out != nullptr && stats_out_slot0 + 2 * n_tiles > stats_out_stride) return ADSR_ERR_BAD_SHAPE;
    // A tiles come by TMA: tensor = [M rows x K cols]; columns >= K and rows >= M are zero-filled by the hardware
    p.use_tma = 1;
    if ((reinterpret_cast<uintptr_t>(A) & 15) || (lda % 8)) return ADSR_ERR_BAD_ALIGN;
    const int st = encode_tmap_rows_bf16(&p.tmap_a, A, M, K, lda);
    if (st != ADSR_OK) return st;
    return launch_tc_gemm(p, num_sms, static_cast<cudaStream_t>(stream));
}

extern "C" int adsr_conv3x3_halo_bf16(const void* in, int64_t ld_in, int B, int H, int W, int Cin, const void* w_compact,
                                      const float* bias_padded, int N, int BN, int act, float slope, void* out, int64_t ldo,
                                      int ocol0, int n_store, float* chan_part, int num_sms, void* stream) {
    if (B <= 0) return ADSR_OK;
    if (in == nullptr || w_compact == nullptr || bias_padded == nullptr || out == nullptr) return ADSR_ERR_BAD_SHAPE;
    if (ld_in < ((Cin + 7) & ~7)) return ADSR_ERR_BAD_SHAPE;
    ConvHaloParams p{};
    p.wp = static_cast<const uint8_t*>(w_compact);
    p.bias = bias_padded;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.ldo = ldo;
    p.ocol0 = ocol0;
    p.n_store = n_store;
    p.chan_part = chan_part;
    p.B = B;
    p.H = H;
    p.W = W;
    p.Cin = Cin;
    p.N = N;
    p.BN = BN;
    p.act = act;
    p.slope = slope;
    return launch_conv_halo(p, in, ld_in, num_sms, static_cast<cudaStream_t>(stream));
}

extern "C" int adsr_conv3x3_igemm_bf16(const void* in, int64_t ld_in, int B, int Hin, int Win, int Cin, int stride,
                                       const void* w_packed, const float* bias_padded, int N, int BN, int n_tiles, int act,
                                       float slope, float alpha, const void* res, int64_t ldres, void* out, int64_t ldo,
                                       int ocol0, int out_mode, int n_store, int num_sms, void* stream) {
    if (B <= 0) return ADSR_OK;
    if (Cin <= 0 || N <= 0 || (stride != 1 && stride != 2) || n_store > n_tiles * BN || ld_in < ((Cin + 7) & ~7))
        return ADSR_ERR_BAD_SHAPE;
    if (out_mode == ADSR_OUT_PIXEL_SHUFFLE2 && ((N % 4) || stride != 1 || res != nullptr || ocol0 != 0)) return ADSR_ERR_BAD_SHAPE;
    TcGemmParams p{};
    p.A = static_cast<const __nv_bfloat16*>(in);
    p.lda = ld_in;
    p.Hin = Hin;
    p.Win = Win;
    p.stride = stride;
    p.Hout = (Hin + 2 - 3) / stride + 1;
    p.Wout = (Win + 2 - 3) / stride + 1;
    p.M = B * p.Hout * p.Wout;
    p.K8 = (Cin + 7) & ~7;
    p.conv = 1;
    p.stages_per_tap = (Cin + 63) / 64;
    p.k16_per_tap = (Cin + 15) / 16;
    p.num_k_stages = 9 * p.stages_per_tap;
    p.k16_total = 0;
    p.Bp = static_cast<const uint8_t*>(w_packed);
    p.n_tiles = n_tiles;
    p.BN = BN;
    p.m_tiles = (p.M + 127) / 128;
    p.bias = bias_padded;
    p.N = N;
    p.n_store = n_store;
    p.act = act;
    p.slope = slope;
    p.alpha = alpha;
    p.res = static_cast<const __nv_bfloat16*>(res);
    p.ldres = ldres;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.ldo = ldo;
    p.ocol0 = ocol0;
    p.out_mode = out_mode;
    return launch_tc_gemm(p, num_sms, static_cast<cudaStream_t>(stream));
}

// tuning hook (not part of the public header): device buffer that receives the CTA-0 timeline of the next fused-MLP launches
static long long* g_mlp_trace = nullptr;
extern "C" void adsr_debug_set_mlp_trace(void* device_buffer) { g_mlp_trace = static_cast<long long*>(device_buffer); }

static int swin_mlp_common(SwinMlpParams& p, const void* y, int64_t ldy, int M, int C, const void* w1_packed, const void* w2_packed,
                           const float* bias1, const float* colsum1, const float* bias2, const int32_t* plan, int plan_len,
                           float ln_eps, const float* ln_stats_in, int stats_in_slots, int stats_in_stride) {
    if (plan == nullptr || plan_len < 22 || C <= 0 || ldy < C || ln_stats_in == nullptr || stats_in_slots <= 0) return ADSR_ERR_BAD_SHAPE;
    p.ks1 = plan[0]; p.k1steps = plan[1]; p.nc = plan[2]; p.hc = plan[3]; p.n2 = plan[4];
    p.acc1_col[0] = plan[5]; p.acc1_col[1] = plan[6];
    p.n_pieces = plan[7]; p.piece_rows[0] = plan[8]; p.piece_rows[1] = plan[9];
    p.piece_col[0] = 0; p.piece_col[1] = plan[8];
    p.w1_slots = plan[10]; p.w1_slot_bytes = plan[11]; p.w2_slots = plan[12]; p.w2_slot_bytes = plan[13];
    for (int j = 0; j < 8; ++j) p.hcw[j] = plan[14 + j];
    // plan[23] = 1: folded adjust -- the fc2 ring carries W_adj W2 (32 rows), so the accumulator is 32 columns, not C;
    // plan[23] = 2: wide folded conv with residual -- n2 = the conv's output channels rounded up to 16 (checked by the launcher)
    const int fold = plan_len >= 24 ? plan[23] : 0;
    if (p.ks1 != (C + 63) / 64 || p.k1steps != (C + 15) / 16 || (fold == 0 && p.n2 != (C + 15) / 16 * 16) || (fold == 1 && p.n2 != 32))
        return ADSR_ERR_BAD_SHAPE;
    p.w1p = static_cast<const uint8_t*>(w1_packed);
    p.w2p = static_cast<const uint8_t*>(w2_packed);
    p.bias1 = bias1; p.colsum1 = colsum1; p.bias2 = bias2;
    p.stats_in = reinterpret_cast<const float2*>(ln_stats_in);
    p.stats_in_slots = stats_in_slots; p.stats_in_stride = stats_in_stride;
    p.ln_eps = ln_eps; p.C = C; p.M = M;
    p.trace = g_mlp_trace;
    return ADSR_OK;
}

extern "C" int adsr_swin_mlp_bf16(const void* y, int64_t ldy, int M, int C, const void* w1_packed, const void* w2_packed,
                                  const float* bias1, const float* colsum1, const float* bias2, const int32_t* plan, int plan_len,
                                  float ln_eps, const float* ln_stats_in, int stats_in_slots, int stats_in_stride, void* z,
                                  int64_t ldz, int reverse_tiles, int num_sms, void* stream) {
    if (M <= 0) return ADSR_OK;
    if (ldz < C || (plan != nullptr && plan_len >= 24 && plan[23] != 0)) return ADSR_ERR_BAD_SHAPE;   // a folded-adjust pack has no z
    SwinMlpParams p{};
    p.rev = reverse_tiles != 0;
    const int st = swin_mlp_common(p, y, ldy, M, C, w1_packed, w2_packed, bias1, colsum1, bias2, plan, plan_len, ln_eps, ln_stats_in,
                                   stats_in_slots, stats_in_stride);
    if (st != ADSR_OK) return st;
    return launch_swin_mlp(p, y, ldy, z, ldz, num_sms, static_cast<cudaStream_t>(stream));
}

extern "C" int adsr_swin_mlp_adjust_bf16(const void* y, int64_t ldy, int M, int C, const void* w1_packed, const void* w2_packed,
                                         const float* bias1, const float* colsum1, const float* bias2, const int32_t* plan,
                                         int plan_len, float ln_eps, const float* ln_stats_in, int stats_in_slots,
                                         int stats_in_stride, const void* wadj_packed, const float* bias_adj, float slope,
                                         void* out, int64_t ldo, int ocol0, float* stats_out, int stats_out_slot0,
                                         int stats_out_stride, int reverse_tiles, int num_sms, void* stream) {
    if (M <= 0) return ADSR_OK;
    if (plan_len < 24 || plan[23] != 1 || wadj_packed == nullptr || bias_adj == nullptr || out == nullptr || ldo < ocol0 + 32) return ADSR_ERR_BAD_SHAPE;
    SwinMlpParams p{};
    p.rev = reverse_tiles != 0;
    const int st = swin_mlp_common(p, y, ldy, M, C, w1_packed, w2_packed, bias1, colsum1, bias2, plan, plan_len, ln_eps, ln_stats_in,
                                   stats_in_slots, stats_in_stride);
    if (st != ADSR_OK) return st;
    p.fuse_adj = 1;
    p.wadj = static_cast<const uint8_t*>(wadj_packed);
    p.bias_adj = bias_adj;
    p.adj_out = static_cast<__nv_bfloat16*>(out);
    p.ld_adj = ldo;
    p.adj_col0 = ocol0;
    p.adj_slope = slope;
    p.adj_stats = reinterpret_cast<float2*>(stats_out);
    p.adj_stats_slot0 = stats_out_slot0;
    p.adj_stats_stride = stats_out_stride;
    return launch_swin_mlp(p, y, ldy, nullptr, 0, num_sms, static_cast<cudaStream_t>(stream));
}

extern "C" int adsr_swin_mlp_conv_res_bf16(const void* y, int64_t ldy, int M, int C, const void* w1_packed, const void* w2_packed,
                                           const float* bias1, const float* colsum1, const float* bias2, const int32_t* plan,
                                           int plan_len, float ln_eps, const float* ln_stats_in, int stats_in_slots,
                                           int stats_in_stride, const void* res, int64_t ldres, void* out, int64_t ldo, int c_out,
                                           float* stats_out, int stats_out_slot0, int stats_out_stride, int reverse_tiles, int num_sms,
                                           void* stream) {
    if (M <= 0) return ADSR_OK;
    if (plan_len < 24 || plan[23] != 2 || res == nullptr || out == nullptr) return ADSR_ERR_BAD_SHAPE;
    SwinMlpParams p{};
    p.rev = reverse_tiles != 0;
    const int st = swin_mlp_common(p, y, ldy, M, C, w1_packed, w2_packed, bias1, colsum1, bias2, plan, plan_len, ln_eps, ln_stats_in,
                                   stats_in_slots, stats_in_stride);
    if (st != ADSR_OK) return st;
    p.fold_res = 1;
    p.c_out = c_out;
    p.res = static_cast<const __nv_bfloat16*>(res);
    p.ld_res = ldres;
    p.adj_stats = reinterpret_cast<float2*>(stats_out);
    p.adj_stats_slot0 = stats_out_slot0;
    p.adj_stats_stride = stats_out_stride;
    return launch_swin_mlp(p, y, ldy, out, ldo, num_sms, static_cast<cudaStream_t>(stream));
}

static long long* g_attn_trace = nullptr;
extern "C" void adsr_debug_set_attn_trace(void* device_buffer) { g_attn_trace = static_cast<long long*>(device_buffer); }

extern "C" int adsr_swin_attn_mode(int C, int heads, int head_dim_padded, int allow_proj) {
    SwinAttnParams p{};
    return swin_attn_plan(p, C, heads, head_dim_padded, allow_proj);
}

extern "C" int adsr_swin_attn_bf16(const void* x, int64_t ldx, int B, int H, int W, int C, int shift, int heads, int head_dim,
                                   int head_dim_padded, const void* w1_packed, const void* w2_packed, const float* bias_qkv,
                                   const float* colsum_qkv, const float* bias_proj, const float* bias_table, float ln_eps,
                                   const float* ln_stats_in, int stats_in_slots, int stats_in_stride, int fuse_proj, void* out,
                                   int64_t ldo, float* stats_out, int stats_out_slot0, int stats_out_stride, int num_sms,
                                   void* stream) {
    if (B <= 0) return ADSR_OK;
    if (head_dim <= 0 || head_dim > head_dim_padded || ln_stats_in == nullptr || stats_in_slots <= 0 || x == nullptr || out == nullptr ||
        w1_packed == nullptr || bias_qkv == nullptr || colsum_qkv == nullptr || bias_table == nullptr)
        return ADSR_ERR_BAD_SHAPE;
    SwinAttnParams p{};
    const int mode = swin_attn_plan(p, C, heads, head_dim_padded, fuse_proj);
    if (mode == 0 || (fuse_proj != 0) != (mode == 2)) return ADSR_ERR_BAD_SHAPE;
    if (mode == 2 && (w2_packed == nullptr || bias_proj == nullptr)) return ADSR_ERR_BAD_SHAPE;
    if (stats_out != nullptr && (mode != 2 || stats_out_slot0 >= stats_out_stride)) return ADSR_ERR_BAD_SHAPE;
    p.x = static_cast<const __nv_bfloat16*>(x); p.ldx = ldx;
    p.out = static_cast<__nv_bfloat16*>(out); p.ldo = ldo;
    p.w1p = static_cast<const uint8_t*>(w1_packed); p.w2p = static_cast<const uint8_t*>(w2_packed);
    p.bias_qkv = bias_qkv; p.colsum_qkv = colsum_qkv; p.bias_p = bias_proj; p.table = bias_table;
    p.stats_in = reinterpret_cast<const float2*>(ln_stats_in);
    p.stats_in_slots = stats_in_slots; p.stats_in_stride = stats_in_stride;
    p.stats_out = reinterpret_cast<float2*>(stats_out);
    p.stats_out_slot0 = stats_out_slot0; p.stats_out_stride = stats_out_stride;
    p.ln_eps = ln_eps;
    p.scale_log2e = (1.0f / sqrtf(static_cast<float>(head_dim))) * 1.4426950408889634f;
    p.B = B; p.H = H; p.W = W; p.shift = shift;
    p.trace = g_attn_trace;
    return launch_swin_attn(p, num_sms, static_cast<cudaStream_t>(stream));
}

// ----------------------------------------------------------------------------- host-side weight packing + workspace sizes
// (SURVEY.md section 8b: `pack_weights_*` and `*_workspace_bytes`).  Pure host code: loading a model launches no device kernel.
static inline uint16_t bf16_bits_rn(float f) {
    const __nv_bfloat16 h = __float2bfloat16_rn(f);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
}

extern "C" int adsr_pack_slab_sw128(const float* host_src, int64_t ld, int rows, int cols, void* host_dst) {
    if (host_src == nullptr || host_dst == nullptr || rows <= 0 || cols < 0 || cols > 64 || ld < cols) return ADSR_ERR_BAD_SHAPE;
    uint16_t* dst = static_cast<uint16_t*>(host_dst);
    for (int r = 0; r < rows; ++r) {
        const float* src = host_src + static_cast<int64_t>(r) * ld;
        for (int pos = 0; pos < 8; ++pos) {                    // 16-byte chunk c of the row is stored at position c ^ (r % 8)
            const int c = pos ^ (r & 7);
            for (int e = 0; e < 8; ++e) {
                const int k = c * 8 + e;
                dst[(static_cast<int64_t>(r) * 8 + pos) * 8 + e] = k < cols ? bf16_bits_rn(src[k]) : uint16_t(0);
            }
        }
    }
    return ADSR_OK;
}

extern "C" int adsr_pack_tiles_sw128(const float* host_w, int64_t ld, int n, int k, int bn, int n_tiles, void* host_dst) {
    if (host_w == nullptr || host_dst == nullptr || n <= 0 || k <= 0 || bn <= 0 || n_tiles <= 0 || n > bn * n_tiles || ld < k) return ADSR_ERR_BAD_SHAPE;
    const int ks = (k + 63) / 64;
    uint8_t* dst = static_cast<uint8_t*>(host_dst);
    const size_t slab = static_cast<size_t>(bn) * 128;
    memset(dst, 0, slab * ks * n_tiles);
    for (int t = 0; t < n_tiles; ++t)
        for (int s = 0; s < ks; ++s) {
            const int row0 = t * bn, rows = n - row0 < bn ? n - row0 : bn;
            if (rows <= 0) continue;
            const int cols = k - 64 * s < 64 ? k - 64 * s : 64;
            const int st = adsr_pack_slab_sw128(host_w + static_cast<int64_t>(row0) * ld + 64 * s, ld, rows, cols, dst + (static_cast<size_t>(t) * ks + s) * slab);
            if (st != ADSR_OK) return st;
        }
    return ADSR_OK;
}

extern "C" int64_t adsr_drct_workspace_bytes(int B, int H, int W, int embed_dim, int gc, int upscale, int qkv_cols, int att_cols) {
    if (B <= 0 || H <= 0 || W <= 0 || embed_dim <= 0 || gc < 0 || upscale < 1 || (upscale & (upscale - 1))) return -1;
    const int64_t M = static_cast<int64_t>(B) * H * W;
    const int64_t pitch = (embed_dim + 4 * gc + 63) / 64 * 64, e16 = (embed_dim + 15) / 16 * 16;
    int64_t bytes = M * (3 * pitch + qkv_cols + att_cols + 2 * e16 + 64) * 2      // slab, y, z, qkv, att, x0, body, f   (bf16 rows)
                    + M * (12 + 8) * 2 * 4;                                       // per-row (sum, sumsq) slots of slab and y (fp32)
    int64_t m = M;
    for (int s = upscale; s > 1; s >>= 1) { m *= 4; bytes += m * 64 * 2; }        // PixelShuffle stages (64 channels)
    return bytes;
}

extern "C" int64_t adsr_score_workspace_bytes(int B, int H, int W, int C, int n_ws) {
    (void)B; (void)H; (void)W; (void)C; (void)n_ws;
    return 0;                                                                     // the scorer keeps everything on chip
}

