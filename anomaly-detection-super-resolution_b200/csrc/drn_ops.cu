// Bandwidth-bound kernels specific to the DRN path: bicubic up-sampling fused with the sub_mean MeanShift,
// the 1/3-channel head convolution, per-image channel means (global average pool) and the RCAB channel-
// attention epilogue  out = res * sigmoid(W2 relu(W1 mean + b1) + b2) + x.
#include "adsr_kernels.h"
#include "ptx.cuh"

namespace adsr {
namespace {

// ATen upsample_bicubic2d coefficients (A = -0.75), align_corners = False.
__device__ __forceinline__ float cubic1(float x) { return ((1.25f * x - 2.25f) * x) * x + 1.f; }             // |x| <= 1
__device__ __forceinline__ float cubic2(float x) { return ((-0.75f * x + 3.75f) * x - 6.f) * x + 3.f; }      // 1 < |x| < 2
__device__ __forceinline__ void cubic_coeffs(float t, float (&c)[4]) {
    c[0] = cubic2(t + 1.f);
    c[1] = cubic1(t);
    c[2] = cubic1(1.f - t);
    c[3] = cubic2(2.f - t);
}

// out[b, :, oy, ox] = Wm * bicubic(in)[b, :, oy, ox] + bm      (nn.Upsample(bicubic) + MeanShift, src/drn.py:243-246)
__global__ void __launch_bounds__(256) bicubic_affine_kernel(const float* __restrict__ in, int B, int nc, int h, int w,
                                                              int scale, const float* __restrict__ Wm,
                                                              const float* __restrict__ bm, float* __restrict__ out) {
    const int H = h * scale, W = w * scale;
    const long long total = static_cast<long long>(B) * H * W;
    const float inv = 1.0f / static_cast<float>(scale);
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int ox = static_cast<int>(i % W);
        const int oy = static_cast<int>((i / W) % H);
        const int b = static_cast<int>(i / (static_cast<long long>(W) * H));
        const float sy = (oy + 0.5f) * inv - 0.5f, sx = (ox + 0.5f) * inv - 0.5f;
        const float fy = floorf(sy), fx = floorf(sx);
        const int iy = static_cast<int>(fy), ix = static_cast<int>(fx);
        float cy[4], cx[4];
        cubic_coeffs(sy - fy, cy);
        cubic_coeffs(sx - fx, cx);
        float v[3] = {0.f, 0.f, 0.f};
        for (int c = 0; c < nc; ++c) {
            const float* plane = in + (static_cast<long long>(b) * nc + c) * h * w;
            float acc = 0.f;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int yy = min(max(iy - 1 + r, 0), h - 1);
                float row = 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int xx = min(max(ix - 1 + q, 0), w - 1);
                    row += __ldg(plane + yy * w + xx) * cx[q];
                }
                acc += row * cy[r];
            }
            v[c] = acc;
        }
        for (int c = 0; c < nc; ++c) {
            float o = __ldg(bm + c);
            for (int k = 0; k < nc; ++k) o += __ldg(Wm + c * nc + k) * v[k];
            out[((static_cast<long long>(b) * nc + c) * H + oy) * W + ox] = o;
        }
    }
}

// 3x3 conv, pad 1, stride 1, Cin <= 3 (fp32 NCHW in) -> Cout <= 64 channels, NHWC bf16, to one or two destinations
// (DRN head, src/drn.py:247; the second destination is the skip-connection slice of the concat buffer).
__global__ void __launch_bounds__(128) conv3x3_small_kernel(const float* __restrict__ x, int B, int nc, int H, int W,
                                                             const float* __restrict__ weight, const float* __restrict__ bias,
                                                             int C, __nv_bfloat16* __restrict__ out1, long long ld1,
                                                             int npad1, __nv_bfloat16* __restrict__ out2, long long ld2,
                                                             int col2) {
    extern __shared__ float sw[];                     // [nc*9][C] + bias[C]
    const int kk = nc * 9;
    for (int i = threadIdx.x; i < kk * C; i += blockDim.x) {
        const int k = i / C, c = i - k * C;
        sw[i] = weight[c * kk + k];
    }
    for (int i = threadIdx.x; i < C; i += blockDim.x) sw[kk * C + i] = bias ? bias[i] : 0.f;
    __syncthreads();
    const long long total = static_cast<long long>(B) * H * W;
    const long long pix = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pix >= total) return;
    const int b = static_cast<int>(pix / (H * W));
    const int rem = static_cast<int>(pix - static_cast<long long>(b) * H * W);
    const int y = rem / W, xx = rem - y * W;
    float taps[27];
#pragma unroll
    for (int k = 0; k < 27; ++k) taps[k] = 0.f;
    for (int c = 0; c < nc; ++c)
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const int iy = y + t / 3 - 1, ix = xx + t % 3 - 1;
            if (iy >= 0 && iy < H && ix >= 0 && ix < W)
                taps[c * 9 + t] = __ldg(x + ((static_cast<long long>(b) * nc + c) * H + iy) * W + ix);
        }
    for (int c0 = 0; c0 < C; c0 += 4) {                // C % 4 == 0
        float a[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) a[j] = sw[kk * C + c0 + j];
        for (int k = 0; k < kk; ++k) {
            const float4 wv = *reinterpret_cast<const float4*>(sw + k * C + c0);
            a[0] = fmaf(taps[k], wv.x, a[0]); a[1] = fmaf(taps[k], wv.y, a[1]);
            a[2] = fmaf(taps[k], wv.z, a[2]); a[3] = fmaf(taps[k], wv.w, a[3]);
        }
        const uint2 o = make_uint2(pack_bf16x2(a[0], a[1]), pack_bf16x2(a[2], a[3]));
        *reinterpret_cast<uint2*>(out1 + pix * ld1 + c0) = o;
        if (out2) *reinterpret_cast<uint2*>(out2 + pix * ld2 + col2 + c0) = o;
    }
    for (int c0 = C; c0 < npad1; c0 += 4) *reinterpret_cast<uint2*>(out1 + pix * ld1 + c0) = make_uint2(0, 0);
}

// Column sums of slice s of image b's HW pixels: x [B, HW, ld] bf16 -> part[(b * slices + s) * ld_part + c] fp32, the partial-row
// layout channel_mean_parts_kernel reduces in a fixed order (CALayer's AdaptiveAvgPool2d(1) where the halo conv does not run).
// grid = (slices, B), 16-byte loads (C % 8 == 0): thread = (pixel slot, 8-channel group), the slots meet in shared memory in order.
__global__ void __launch_bounds__(256) channel_sum8_kernel(const __nv_bfloat16* __restrict__ x, long long ld, int HW, int C,
                                                            float* __restrict__ part, int ld_part) {
    __shared__ float red[256 * 8];
    const int b = blockIdx.y;
    const int groups = C >> 3;
    const int ppi = 256 / groups;                           // pixels per iteration
    const int g = threadIdx.x % groups, slot = threadIdx.x / groups;
    const int per_slice = (HW + gridDim.x - 1) / gridDim.x;
    const int p0 = blockIdx.x * per_slice, p1 = min(HW, p0 + per_slice);
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (slot < ppi) {
        const __nv_bfloat16* base = x + static_cast<long long>(b) * HW * ld + 8 * g;
#pragma unroll 4
        for (int p = p0 + slot; p < p1; p += ppi) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(base + static_cast<long long>(p) * ld));
            s[0] += bf16_lo(v.x); s[1] += bf16_hi(v.x); s[2] += bf16_lo(v.y); s[3] += bf16_hi(v.y);
            s[4] += bf16_lo(v.z); s[5] += bf16_hi(v.z); s[6] += bf16_lo(v.w); s[7] += bf16_hi(v.w);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) red[slot * C + 8 * g + e] = s[e];
    }
    __syncthreads();
    if (threadIdx.x < C) {
        float t = 0.f;
        for (int sl = 0; sl < ppi; ++sl) t += red[sl * C + threadIdx.x];
        part[(static_cast<long long>(b) * gridDim.x + blockIdx.x) * ld_part + threadIdx.x] = t;
    }
}

// mean[b, c] from the per-(tile, row quadrant) column sums the halo conv's epilogue leaves behind (conv_halo.cu): fixed summation order
// With w1 != nullptr the block goes on to CALayer's squeeze-excite MLP and writes scale[b, c] = sigmoid(W2 relu(W1 mean + b1) + b2)
// instead of the mean: once per image, not once per block of the scaling pass.
__global__ void __launch_bounds__(1024) channel_mean_parts_kernel(const float* __restrict__ part, int parts, int ld, int C, float inv_hw,
                                                                   float* __restrict__ mean, const float* __restrict__ w1,
                                                                   const float* __restrict__ b1, const float* __restrict__ w2,
                                                                   const float* __restrict__ b2, int Cr) {
    __shared__ float red[8][128];
    __shared__ float hid[16];
    const int b = blockIdx.x, c = threadIdx.x & 127, g = threadIdx.x >> 7;      // 8 groups take every 8th partial row
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // the MLP weights do not depend on the sums: fetch them first so that the kernel is two L2 round trips, not seven
    float w1v[4] = {0.f, 0.f, 0.f, 0.f}, w2v[16], b1v = 0.f, b2v = 0.f;
    const bool mlp = w1 != nullptr;
    if (mlp && warp < Cr) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (lane + 32 * k < C) w1v[k] = w1[warp * C + lane + 32 * k];
        b1v = b1[warp];
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) w2v[j] = (mlp && g == 0 && c < C && j < Cr) ? w2[c * Cr + j] : 0.f;
    if (mlp && g == 0 && c < C) b2v = b2[c];
    pdl_launch_dependents();
    pdl_wait();                                                                 // the partial sums are the previous kernel's output
    float acc = 0.f;
    if (c < C) {
        const float* p = part + static_cast<long long>(b) * parts * ld + c;
        float v[24];
#pragma unroll
        for (int k = 0; k < 24; ++k) {                                          // up to 192 partial rows with every load in flight at once
            const int i = g + 8 * k;
            v[k] = i < parts ? p[static_cast<long long>(i) * ld] : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 24; ++k) acc += v[k];
        for (int i = g + 192; i < parts; i += 8) acc += p[static_cast<long long>(i) * ld];
    }
    red[g][c] = acc;
    __syncthreads();
    if (g == 0 && c < C) {
        float t = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) t += red[j][c];
        t *= inv_hw;
        if (!mlp) mean[static_cast<long long>(b) * C + c] = t;
        red[0][c] = t;
    }
    if (!mlp) return;
    __syncthreads();
    if (warp < Cr) {                                                            // one warp per hidden unit
        float a = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (lane + 32 * k < C) a = fmaf(w1v[k], red[0][lane + 32 * k], a);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (lane == 0) hid[warp] = fmaxf(a + b1v, 0.f);
    }
    __syncthreads();
    if (g == 0 && c < C) {
        float a = b2v;
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (j < Cr) a = fmaf(w2v[j], hid[j], a);
        mean[static_cast<long long>(b) * C + c] = 1.f / (1.f + __expf(-a));
    }
}

// out = res * scale[b] + x       (CALayer + RCAB residual, src/drn.py:123-158; the scales from channel_mean_parts with the MLP)
__global__ void __launch_bounds__(256) rcab_ca_scale_kernel(const __nv_bfloat16* __restrict__ res, long long ldr,
                                                             const __nv_bfloat16* __restrict__ x, long long ldx,
                                                             __nv_bfloat16* __restrict__ out, long long ldo,
                                                             const float* __restrict__ scale, int HW, int C) {
    __shared__ float sc[128];
    const int b = blockIdx.y;
    pdl_launch_dependents();
    pdl_wait();                                             // scale / res / x come from the previous kernels
    if (threadIdx.x < C) sc[threadIdx.x] = scale[static_cast<long long>(b) * C + threadIdx.x];
    __syncthreads();
    const uint32_t vec = static_cast<uint32_t>(C) / 8u;               // 16-byte vectors per pixel
    const uint32_t n = static_cast<uint32_t>(HW) * vec;                 // per image: < 2^31 (checked by the wrapper)
    const uint32_t step = gridDim.x * blockDim.x;
    const __nv_bfloat16* rb = res + static_cast<long long>(b) * HW * ldr;
    const __nv_bfloat16* xb = x + static_cast<long long>(b) * HW * ldx;
    __nv_bfloat16* ob = out + static_cast<long long>(b) * HW * ldo;
    // two vectors in flight per thread; 32-bit index arithmetic (a 64-bit division per vector used to dominate the issue slots)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += 2 * step) {
        const uint32_t i1 = i + step;
        const bool two = i1 < n;
        const uint32_t p0 = i / vec, c0 = (i - p0 * vec) * 8u;
        const uint32_t p1 = two ? i1 / vec : p0, c1 = two ? (i1 - p1 * vec) * 8u : c0;
        const uint4 r0 = __ldg(reinterpret_cast<const uint4*>(rb + static_cast<long long>(p0) * ldr + c0));
        const uint4 r1 = __ldg(reinterpret_cast<const uint4*>(rb + static_cast<long long>(p1) * ldr + c1));
        const uint4 x0 = *reinterpret_cast<const uint4*>(xb + static_cast<long long>(p0) * ldx + c0);
        const uint4 x1 = *reinterpret_cast<const uint4*>(xb + static_cast<long long>(p1) * ldx + c1);
        {
            const uint32_t rr[4] = {r0.x, r0.y, r0.z, r0.w}, xx[4] = {x0.x, x0.y, x0.z, x0.w};
            uint32_t o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                o[j] = pack_bf16x2(fmaf(bf16_lo(rr[j]), sc[c0 + 2 * j], bf16_lo(xx[j])), fmaf(bf16_hi(rr[j]), sc[c0 + 2 * j + 1], bf16_hi(xx[j])));
            *reinterpret_cast<uint4*>(ob + static_cast<long long>(p0) * ldo + c0) = make_uint4(o[0], o[1], o[2], o[3]);
        }
        if (two) {
            const uint32_t rr[4] = {r1.x, r1.y, r1.z, r1.w}, xx[4] = {x1.x, x1.y, x1.z, x1.w};
            uint32_t o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                o[j] = pack_bf16x2(fmaf(bf16_lo(rr[j]), sc[c1 + 2 * j], bf16_lo(xx[j])), fmaf(bf16_hi(rr[j]), sc[c1 + 2 * j + 1], bf16_hi(xx[j])));
            *reinterpret_cast<uint4*>(ob + static_cast<long long>(p1) * ldo + c1) = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
}

inline int check_launch() { return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH; }

}  // namespace
}  // namespace adsr

using namespace adsr;

extern "C" int adsr_bicubic_affine(const float* x_nchw, int B, int nc, int h, int w, int scale, const float* mat,
                                   const float* bias, float* out_nchw, void* stream) {
    if (B <= 0) return ADSR_OK;
    if (nc < 1 || nc > 3 || scale < 1 || h < 1 || w < 1) return ADSR_ERR_BAD_SHAPE;
    const long long total = static_cast<long long>(B) * h * scale * w * scale;
    const int grid = static_cast<int>(std::min<long long>((total + 255) / 256, 148 * 16));
    bicubic_affine_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x_nchw, B, nc, h, w, scale, mat, bias, out_nchw);
    return check_launch();
}

extern "C" int adsr_conv3x3_small(const float* x_nchw, int B, int nc, int H, int W, const float* weight, const float* bias,
                                  int C, void* out1, int64_t ld1, void* out2, int64_t ld2, int col2, void* stream) {
    if (B <= 0) return ADSR_OK;
    if (nc < 1 || nc > 3 || C < 4 || C > 64 || (C % 4) || (ld1 % 4) || (out2 && ((ld2 % 4) || (col2 % 4)))) return ADSR_ERR_BAD_SHAPE;
    const int npad1 = std::min<int64_t>(ld1, (C + 15) & ~15);
    const size_t smem = (static_cast<size_t>(nc) * 9 * C + C) * sizeof(float);
    const long long total = static_cast<long long>(B) * H * W;
    conv3x3_small_kernel<<<static_cast<int>((total + 127) / 128), 128, smem, static_cast<cudaStream_t>(stream)>>>(
        x_nchw, B, nc, H, W, weight, bias, C, static_cast<__nv_bfloat16*>(out1), ld1, npad1,
        static_cast<__nv_bfloat16*>(out2), ld2, col2);
    return check_launch();
}

extern "C" int adsr_channel_mean(const void* x, int64_t ld, int B, int HW, int C, int slices, float* part, int64_t ld_part,
                                 void* stream) {
    if (B <= 0) return ADSR_OK;
    if (C < 8 || C > 128 || (C % 8) || (ld % 8) || (reinterpret_cast<uintptr_t>(x) & 15) || slices < 1 || slices > HW || ld_part < C)
        return ADSR_ERR_BAD_SHAPE;
    channel_sum8_kernel<<<dim3(slices, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(x), ld, HW,
                                                                                         C, part, static_cast<int>(ld_part));
    return check_launch();
}

extern "C" int adsr_channel_mean_parts(const float* chan_part, int B, int parts, int ld_part, int C, int HW, float* mean, const float* w1,
                                       const float* b1, const float* w2, const float* b2, int Cr, void* stream) {
    if (B <= 0) return ADSR_OK;
    if (C < 1 || C > 128 || parts < 1 || ld_part < C || HW < 1) return ADSR_ERR_BAD_SHAPE;
    if (w1 != nullptr && (Cr < 1 || Cr > 16 || b1 == nullptr || w2 == nullptr || b2 == nullptr)) return ADSR_ERR_BAD_SHAPE;
    return launch_pdl(channel_mean_parts_kernel, dim3(B), dim3(1024), 0, static_cast<cudaStream_t>(stream), chan_part, parts, ld_part, C,
                      1.f / static_cast<float>(HW), mean, w1, b1, w2, b2, Cr) == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}

extern "C" int adsr_rcab_ca_scale(const void* res, int64_t ldr, const void* x, int64_t ldx, void* out, int64_t ldo,
                                  const float* scale, int B, int HW, int C, void* stream) {
    if (B <= 0) return ADSR_OK;
    if (C < 8 || C > 128 || (C % 8) || (ldr % 8) || (ldx % 8) || (ldo % 8)) return ADSR_ERR_BAD_SHAPE;
    if (static_cast<long long>(HW) * (C / 8) >= (1ll << 31)) return ADSR_ERR_BAD_SHAPE;
    const int slices = std::max(1, std::min(64, HW * (C / 8) / 1024));
    return launch_pdl(rcab_ca_scale_kernel, dim3(slices, B), dim3(256), 0, static_cast<cudaStream_t>(stream),
                      static_cast<const __nv_bfloat16*>(res), static_cast<long long>(ldr), static_cast<const __nv_bfloat16*>(x),
                      static_cast<long long>(ldx), static_cast<__nv_bfloat16*>(out), static_cast<long long>(ldo), scale, HW,
                      C) == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}
