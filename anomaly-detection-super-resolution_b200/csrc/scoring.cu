// Per-image anomaly scores: box-filter SSIM with reflect padding for every window size of the
// evaluator's sweep, MSE and PSNR, on uint8 HWC image pairs.
//
// Replaces the reference's per-pixel Python double loop `ssim_numpy` (src/metrics.py:26-67; 0.5-1.6 s
// per call, 14 calls per image), the MSE of src/evaluate.py:259-260 and psnr_numpy (src/metrics.py:15-23).
//
// Grid = (n_ws + 1, B): CTA (j, b) computes SSIM of image b for window size ws_j; the extra CTA
// computes MSE/PSNR.  Inside a CTA one thread owns one image column and walks down the rows keeping
// the five vertical window sums (x, y, x^2, y^2, xy) as fp64 running sums (add the entering row,
// subtract the leaving one, reflect indices at the borders); per row the five column sums are turned
// into prefix sums across the row (warp shuffles + one shared-memory hop), so each horizontal window
// sum is a difference of two prefix values (three differences when the window reflects at a border).
// Work per pixel is O(1) in the window size; the images are read straight from L2 as uint8 and no
// workspace is needed.  Sums are fp64 and the per-pixel term is ssim_term (adsr_kernels.h), so the result is
// within 1e-10 of the kernel-faithful oracle (oracle/scoring_oracle.py: the kernels' fmaf gray chain, exact
// window sums; MSE to 1e-14 relative) and within ~1e-6 of the reference's fp32 loop; an identical pair gives
// exactly 1.  The two kernels for images of up to 128 columns sum in the same order, so an image's row does
// not depend on the batch size that picks between them (tests/test_gpu_scoring_dispatch.py).
#include "adsr_kernels.h"
#include "ptx.cuh"

namespace adsr {
namespace {

constexpr int kMaxWs = 128;      // metrics.window_sizes_for(1024) gives 102 window sizes; W <= 1024 is the kernels' own limit
struct WsList { int32_t ws[kMaxWs]; };

__device__ __forceinline__ int reflect_idx(int i, int n) {        // np.pad(mode="reflect"), |overhang| < n
    if (i < 0) i = -i;
    if (i >= n) i = 2 * (n - 1) - i;
    return i;
}

// How a pixel is fetched.  Element strides let one kernel serve uint8 HWC (the evaluator), fp32 HWC
// (generic ssim_numpy / psnr_numpy callers) and cropped fp32 NCHW views (psnr_torch / ssim_torch).
struct PixelView {
    const void* base;
    long long sb, sr, sc, sch;   // element strides: image, row, column, channel
    int is_f32;                  // 0 = uint8, 1 = float
    float div;                   // value / div  (255 for uint8 -> [0,1]; rgb_range for ssim_torch; 1 otherwise)
    int clamp01;                 // clamp to [0,1] after the division (ssim_torch, src/metrics.py:86-87)
    float quant;                 // > 0: the validation loop's `quantize` (src/trainer.py:45-47) on the raw value first:
                                 // round_half_even(clamp(x * quant, 0, 255)) / quant with quant = 255 / rgb_range
};

__device__ __forceinline__ float fetch(const PixelView& v, long long off) {
    float x = v.is_f32 ? __ldg(static_cast<const float*>(v.base) + off)
                       : static_cast<float>(__ldg(static_cast<const uint8_t*>(v.base) + off));
    if (v.quant > 0.f) x = __fdiv_rn(rintf(fminf(fmaxf(x * v.quant, 0.f), 255.f)), v.quant);
    if (v.div != 1.0f) x = x / v.div;
    if (v.clamp01) x = fminf(fmaxf(x, 0.f), 1.f);
    return x;
}
// the MSE / PSNR terms of the validation loop are NOT clamped (psnr_torch, src/metrics.py:70-79), its SSIM terms are
__device__ __forceinline__ float fetch_mse(PixelView v, long long off, int noclamp) {
    if (noclamp) v.clamp01 = 0;
    return fetch(v, off);
}

// gray value exactly as the reference builds it: channels dotted with the fp32
// (65.738, 129.057, 25.064)/256 coefficients (src/metrics.py:37-39, :93-96); single channel: as is.
__device__ __forceinline__ float gray_at(const PixelView& v, long long off, int C) {
    if (C == 1) return fetch(v, off);
    const float c0 = 65.738f / 256.0f, c1 = 129.057f / 256.0f, c2 = 25.064f / 256.0f;
    const float r = fetch(v, off), g = fetch(v, off + v.sch), b = fetch(v, off + 2 * v.sch);
    return fmaf(b, c2, fmaf(g, c1, r * c0));
}

__device__ __forceinline__ double shfl_up_d(double v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }

struct ScoreParams {
    PixelView sr, hr;
    int H, W, C, n_ws;
    int zero_pad;               // 0 = np.pad(mode="reflect") (ssim_numpy), 1 = zero padding (F.conv2d, ssim_torch)
    int mse_noclamp;            // the MSE / PSNR terms ignore clamp01 (validation loop: psnr_torch does not clamp, ssim_torch does)
    double C1, C2, psnr_peak2;  // SSIM constants and data_range^2 of the PSNR
    double* scores;
    WsList wl;
};

__global__ void __launch_bounds__(1024) score_images_kernel(const ScoreParams p) {
    const int H = p.H, W = p.W, C = p.C, n_ws = p.n_ws;
    double* __restrict__ scores = p.scores;
    extern __shared__ double sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int b = blockIdx.y, j = blockIdx.x;
    const long long srb = static_cast<long long>(b) * p.sr.sb, hrb = static_cast<long long>(b) * p.hr.sb;
    double* red = sm;                                   // [32] block reduction scratch

    if (j == n_ws) {
        // ---------------- MSE / PSNR over all pixels and channels of u8/255 images ---------------
        const long long n = static_cast<long long>(H) * W * C;
        double acc = 0.0;
        for (long long i = tid; i < n; i += blockDim.x) {
            const int ch = static_cast<int>(i % C);
            const long long px = i / C;
            const int r = static_cast<int>(px / W), c = static_cast<int>(px - static_cast<long long>(r) * W);
            const float d = fetch_mse(p.sr, srb + r * p.sr.sr + c * p.sr.sc + ch * p.sr.sch, p.mse_noclamp) -
                            fetch_mse(p.hr, hrb + r * p.hr.sr + c * p.hr.sc + ch * p.hr.sch, p.mse_noclamp);
            acc += static_cast<double>(d * d);          // (ref - out) ** 2 on float32 arrays
        }
        double v = acc;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp] = v;
        __syncthreads();
        if (tid == 0) {
            double t = 0;
            for (int w = 0; w < nwarps; ++w) t += red[w];
            const double mse = t / static_cast<double>(n);
            scores[static_cast<long long>(b) * (n_ws + 2) + n_ws] = mse;
            scores[static_cast<long long>(b) * (n_ws + 2) + n_ws + 1] =
                mse == 0.0 ? __longlong_as_double(0x7ff0000000000000LL) : 10.0 * log10(p.psnr_peak2 / mse);
        }
        return;
    }

    // ---------------- SSIM for window size ws --------------------------------------------------
    const int ws = p.wl.ws[j], pad = ws / 2;
    const int col = tid;                                 // one column per thread (blockDim.x >= W)
    const bool active = col < W;
    double* wtot = sm + 32;                              // [2][5][32] per-warp totals (double buffered)
    double* pref = wtot + 2 * 5 * 32;                    // [2][5][W + 1] prefix sums (double buffered)
    const double inv_n = 1.0 / (static_cast<double>(ws) * ws);
    const double C1 = p.C1, C2 = p.C2;
    const bool zp = p.zero_pad != 0;

    double v[5] = {0, 0, 0, 0, 0};
    auto add_row = [&](int r, double sign) {
        const float x = gray_at(p.hr, hrb + r * p.hr.sr + col * p.hr.sc, C);   // x = reference (HR)
        const float y = gray_at(p.sr, srb + r * p.sr.sr + col * p.sr.sc, C);   // y = SR
        v[0] += sign * static_cast<double>(x);
        v[1] += sign * static_cast<double>(y);
        v[2] += sign * static_cast<double>(x * x);      // products are formed in fp32 like `ref * ref`
        v[3] += sign * static_cast<double>(y * y);
        v[4] += sign * static_cast<double>(x * y);
    };
    if (active)
        for (int r = -pad; r <= pad; ++r) {
            if (zp) { if (r >= 0 && r < H) add_row(r, 1.0); }
            else add_row(reflect_idx(r, H), 1.0);
        }

    double acc = 0.0;
    for (int i = 0; i < H; ++i) {
        const int bufi = i & 1;
        if (i > 0 && active) {
            if (zp) {
                if (i + pad < H) add_row(i + pad, 1.0);
                if (i - pad - 1 >= 0) add_row(i - pad - 1, -1.0);
            } else {
                add_row(reflect_idx(i + pad, H), 1.0);
                add_row(reflect_idx(i - pad - 1, H), -1.0);
            }
        }
        // inclusive scan of the 5 column sums across the row
        double s[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            double t = active ? v[q] : 0.0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double u = shfl_up_d(t, d);
                if (lane >= d) t += u;
            }
            s[q] = t;
            if (lane == 31) wtot[(bufi * 5 + q) * 32 + warp] = t;
        }
        __syncthreads();
        double* P = pref + bufi * 5 * (W + 1);
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            double base = 0.0;
            for (int w = 0; w < warp; ++w) base += wtot[(bufi * 5 + q) * 32 + w];
            if (active) P[q * (W + 1) + col + 1] = s[q] + base;
            if (tid == 0) P[q * (W + 1)] = 0.0;
        }
        __syncthreads();
        if (active) {
            const int lo = col - pad, hi = col + pad;
            const int a0 = lo < 0 ? 0 : lo, a1 = hi > W - 1 ? W - 1 : hi;
            double box[5];
#pragma unroll
            for (int q = 0; q < 5; ++q) {
                const double* Pq = P + q * (W + 1);
                double t = Pq[a1 + 1] - Pq[a0];
                if (!zp) {
                    if (lo < 0) t += Pq[-lo + 1] - Pq[1];                       // reflected columns 1 .. -lo
                    if (hi > W - 1) t += Pq[W - 1] - Pq[2 * (W - 1) - hi];      // reflected columns 2(W-1)-hi .. W-2
                }
                box[q] = t;
            }
            acc += ssim_term(box, inv_n, C1, C2);
        }
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __syncthreads();
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (tid == 0) {
        double t = 0;
        for (int w = 0; w < nwarps; ++w) t += red[w];
        scores[static_cast<long long>(b) * (n_ws + 2) + j] = t / (static_cast<double>(H) * W);
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// Fast path (images up to 128 columns whose two gray planes fit shared memory: the evaluator's 128 x 128 crops):
// ONE CTA of 512 threads per image.  The threads first turn the pair into fp32 gray planes in shared memory (and reduce the
// MSE on the way), then every WARP runs the running-sum / prefix-sum SSIM of one window size (w, w + 16, ...) on the shared
// planes: a lane owns 4 adjacent columns, so the row's prefix sums are a local 4-element prefix + ONE warp scan per quantity
// and the warp never leaves itself (no barriers; the round-1 layout -- 8 workers of 128 threads, one column per thread -- spent
// 73 % of the issue slots on 4x as many scan steps, two named barriers per row and the cross-warp bases, and 14 window sizes
// on 8 workers meant two rounds: 1.6 ms per 256 images).  The prefix rows carry one pad slot per 16 so that the stride-4 accesses
// of a warp are bank-conflict free.  Sums are fp64 in a fixed order (deterministic; same formulas as score_images_kernel).
constexpr int kFastWarps = 16;
constexpr int kFastThreads = kFastWarps * 32;

__device__ __forceinline__ int pidx(int i) { return i + (i >> 4); }      // prefix-array slot of logical index i

__global__ void __launch_bounds__(kFastThreads, 1) score_images_fast_kernel(const ScoreParams p) {
    const int H = p.H, W = p.W, C = p.C, n_ws = p.n_ws;
    extern __shared__ double sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.x;
    const int part = blockIdx.y, nparts = gridDim.y;                    // small batches: the window sizes of an image split over CTAs
    const long long srb = static_cast<long long>(b) * p.sr.sb, hrb = static_cast<long long>(b) * p.hr.sb;
    double* red = sm;                                                   // [32]
    const int prow = pidx(W) + 1;                                       // slots of one prefix row (logical indices 0 .. W)
    double* pref = sm + 32 + warp * 5 * prow;                           // per warp: [5][prow]
    float* gx = reinterpret_cast<float*>(sm + 32 + kFastWarps * 5 * prow);   // HR gray plane
    float* gy = gx + H * W;                                             // SR gray plane

    // ---- gray planes + MSE
    double acc_mse = 0.0;
    for (int idx = tid; idx < H * W; idx += kFastThreads) {
        const int r = idx / W, c = idx - r * W;
        const long long oh = hrb + r * p.hr.sr + c * p.hr.sc, os = srb + r * p.sr.sr + c * p.sr.sc;
        gx[idx] = gray_at(p.hr, oh, C);
        gy[idx] = gray_at(p.sr, os, C);
        for (int ch = 0; ch < C; ++ch) {
            const float d = fetch_mse(p.sr, os + ch * p.sr.sch, p.mse_noclamp) - fetch_mse(p.hr, oh + ch * p.hr.sch, p.mse_noclamp);
            acc_mse += static_cast<double>(d * d);
        }
    }
    for (int o = 16; o > 0; o >>= 1) acc_mse += __shfl_xor_sync(0xffffffffu, acc_mse, o);
    if (lane == 0) red[warp] = acc_mse;
    __syncthreads();
    if (tid == 0 && part == 0) {
        double t = 0;
        for (int w = 0; w < kFastWarps; ++w) t += red[w];
        const double mse = t / (static_cast<double>(H) * W * C);
        p.scores[static_cast<long long>(b) * (n_ws + 2) + n_ws] = mse;
        p.scores[static_cast<long long>(b) * (n_ws + 2) + n_ws + 1] =
            mse == 0.0 ? __longlong_as_double(0x7ff0000000000000LL) : 10.0 * log10(p.psnr_peak2 / mse);
    }

    // ---- SSIM sweep: warp = window size, lane = 4 adjacent columns
    const int c0 = 4 * lane;
    const bool w4 = (W & 3) == 0 && ((reinterpret_cast<uintptr_t>(gx) | reinterpret_cast<uintptr_t>(gy)) & 15) == 0;
    const bool zp = p.zero_pad != 0;
    const double C1 = p.C1, C2 = p.C2;
    for (int j = warp + kFastWarps * part; j < n_ws; j += kFastWarps * nparts) {
        const int ws = p.wl.ws[j], pad = ws / 2;
        const double inv_n = 1.0 / (static_cast<double>(ws) * ws);
        double v[4][5];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int q = 0; q < 5; ++q) v[k][q] = 0.0;
        auto add_row = [&](int r, double sign) {                       // columns >= W contribute nothing
            float xs[4] = {0.f, 0.f, 0.f, 0.f}, ys[4] = {0.f, 0.f, 0.f, 0.f};
            if (w4) {                                                  // one 16-byte load per plane (4 scalar loads at a 16-byte lane pitch are 4-way bank conflicted)
                if (c0 < W) {
                    const float4 a = *reinterpret_cast<const float4*>(gx + r * W + c0), c = *reinterpret_cast<const float4*>(gy + r * W + c0);
                    xs[0] = a.x; xs[1] = a.y; xs[2] = a.z; xs[3] = a.w;
                    ys[0] = c.x; ys[1] = c.y; ys[2] = c.z; ys[3] = c.w;
                }
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (c0 + k < W) { xs[k] = gx[r * W + c0 + k]; ys[k] = gy[r * W + c0 + k]; }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (c0 + k < W) {
                    const float x = xs[k], y = ys[k];
                    v[k][0] += sign * static_cast<double>(x);
                    v[k][1] += sign * static_cast<double>(y);
                    v[k][2] += sign * static_cast<double>(x * x);
                    v[k][3] += sign * static_cast<double>(y * y);
                    v[k][4] += sign * static_cast<double>(x * y);
                }
            }
        };
        for (int r = -pad; r <= pad; ++r) {
            if (zp) { if (r >= 0 && r < H) add_row(r, 1.0); }
            else add_row(reflect_idx(r, H), 1.0);
        }
        if (lane == 0)
            for (int q = 0; q < 5; ++q) pref[q * prow] = 0.0;          // P[0] = 0 (never overwritten)
        double acc = 0.0;
        for (int i = 0; i < H; ++i) {
            if (i > 0) {
                if (zp) {
                    if (i + pad < H) add_row(i + pad, 1.0);
                    if (i - pad - 1 >= 0) add_row(i - pad - 1, -1.0);
                } else {
                    add_row(reflect_idx(i + pad, H), 1.0);
                    add_row(reflect_idx(i - pad - 1, H), -1.0);
                }
            }
            // inclusive prefix sums of the 5 column-sum rows: local over my 4 columns, one warp scan of the lane totals
#pragma unroll
            for (int q = 0; q < 5; ++q) {
                const double l0 = v[0][q], l1 = l0 + v[1][q], l2 = l1 + v[2][q], l3 = l2 + v[3][q];
                double t = l3;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const double u = shfl_up_d(t, d);
                    if (lane >= d) t += u;
                }
                const double base = t - l3;                            // sum of the lanes to my left
                double* Pq = pref + q * prow;
                if (c0 + 0 < W) Pq[pidx(c0 + 1)] = base + l0;
                if (c0 + 1 < W) Pq[pidx(c0 + 2)] = base + l1;
                if (c0 + 2 < W) Pq[pidx(c0 + 3)] = base + l2;
                if (c0 + 3 < W) Pq[pidx(c0 + 4)] = base + l3;
            }
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int col = c0 + k;
                if (col < W) {
                    const int lo = col - pad, hi = col + pad;
                    const int a0 = lo < 0 ? 0 : lo, a1 = hi > W - 1 ? W - 1 : hi;
                    double box[5];
#pragma unroll
                    for (int q = 0; q < 5; ++q) {
                        const double* Pq = pref + q * prow;
                        double t = Pq[pidx(a1 + 1)] - Pq[pidx(a0)];
                        if (!zp) {
                            if (lo < 0) t += Pq[pidx(-lo + 1)] - Pq[pidx(1)];                       // reflected columns 1 .. -lo
                            if (hi > W - 1) t += Pq[pidx(W - 1)] - Pq[pidx(2 * (W - 1) - hi)];      // reflected columns 2(W-1)-hi .. W-2
                        }
                        box[q] = t;
                    }
                    acc += ssim_term(box, inv_n, C1, C2);
                }
            }
            __syncwarp();                                              // the next row overwrites the prefix rows
        }
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) p.scores[static_cast<long long>(b) * (n_ws + 2) + j] = acc / (static_cast<double>(H) * W);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Small-batch variant of the fast path: 8 workers of 128 threads per CTA, one column per thread, worker k runs window sizes
// k, k + 8, ... with a cross-warp prefix (two named barriers per row).  It issues more instructions than the warp-per-window kernel
// above but finishes ONE window size in about a quarter of the time, which is what counts when the batch leaves SMs idle.
// It produces the warp-per-window kernel's bits, so an image's score row does not depend on which of the two the batch size picks:
// the MSE is reduced by the first 16 warps in that kernel's order; a column's sums form a sequential prefix within its group of 4
// columns (the fast kernel's lane), the 32 group totals go through the same Hillis-Steele scan and P = (scan - total) + prefix;
// the group leader adds its 4 columns' SSIM terms in column order and the 32 group sums end in one xor butterfly.
constexpr int kFastWorkers = 8;

__global__ void __launch_bounds__(1024, 1) score_images_fast4_kernel(const ScoreParams p) {
    const int H = p.H, W = p.W, C = p.C, n_ws = p.n_ws;
    extern __shared__ double sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.x;
    const int part = blockIdx.y, nparts = gridDim.y;                    // small batches: the window sizes of an image split over CTAs
    const long long srb = static_cast<long long>(b) * p.sr.sb, hrb = static_cast<long long>(b) * p.hr.sb;
    double* red = sm;                                                   // [32]
    double* wbase = sm + 32;                                            // per worker: gtot [5][32], pref [5][W + 1]
    const int wstride = 5 * 32 + 5 * (W + 1);
    float* gx = reinterpret_cast<float*>(wbase + kFastWorkers * wstride);   // HR gray plane
    float* gy = gx + H * W;                                             // SR gray plane

    // ---- gray planes, then the MSE in score_images_fast_kernel's order (thread t < 512 takes pixels t, t + 512, ...)
    for (int idx = tid; idx < H * W; idx += 1024) {
        const int r = idx / W, c = idx - r * W;
        gx[idx] = gray_at(p.hr, hrb + r * p.hr.sr + c * p.hr.sc, C);
        gy[idx] = gray_at(p.sr, srb + r * p.sr.sr + c * p.sr.sc, C);
    }
    if (part == 0 && warp < kFastWarps) {
        double acc_mse = 0.0;
        for (int idx = tid; idx < H * W; idx += kFastThreads) {
            const int r = idx / W, c = idx - r * W;
            const long long oh = hrb + r * p.hr.sr + c * p.hr.sc, os = srb + r * p.sr.sr + c * p.sr.sc;
            for (int ch = 0; ch < C; ++ch) {
                const float d = fetch_mse(p.sr, os + ch * p.sr.sch, p.mse_noclamp) - fetch_mse(p.hr, oh + ch * p.hr.sch, p.mse_noclamp);
                acc_mse += static_cast<double>(d * d);
            }
        }
        for (int o = 16; o > 0; o >>= 1) acc_mse += __shfl_xor_sync(0xffffffffu, acc_mse, o);
        if (lane == 0) red[warp] = acc_mse;
    }
    __syncthreads();
    if (tid == 0 && part == 0) {
        double t = 0;
        for (int w = 0; w < kFastWarps; ++w) t += red[w];
        const double mse = t / (static_cast<double>(H) * W * C);
        p.scores[static_cast<long long>(b) * (n_ws + 2) + n_ws] = mse;
        p.scores[static_cast<long long>(b) * (n_ws + 2) + n_ws + 1] =
            mse == 0.0 ? __longlong_as_double(0x7ff0000000000000LL) : 10.0 * log10(p.psnr_peak2 / mse);
    }

    // ---- SSIM sweep: worker = 4 warps, thread = column, group g = the 4 columns a fast-kernel lane owns
    const int worker = tid >> 7, col = tid & 127, wwarp = warp & 3, k = col & 3, g = col >> 2;
    const bool active = col < W;
    // Single-buffered scratch: gtot is read only between a row's two barriers and written before the next row's first one; pref
    // is written after a row's first barrier and read after its second, before the next row's first one.
    double* gtot = wbase + worker * wstride;                            // [5][32] group totals, then the 32 group SSIM sums
    double* P = gtot + 5 * 32;                                          // [5][W + 1]
    const bool zp = p.zero_pad != 0;
    const double C1 = p.C1, C2 = p.C2;
    for (int j = worker + kFastWorkers * part; j < n_ws; j += kFastWorkers * nparts) {
        const int ws = p.wl.ws[j], pad = ws / 2;
        const double inv_n = 1.0 / (static_cast<double>(ws) * ws);
        double v[5] = {0, 0, 0, 0, 0};
        auto add_row = [&](int r, double sign) {
            const float x = gx[r * W + col], y = gy[r * W + col];
            v[0] += sign * static_cast<double>(x);
            v[1] += sign * static_cast<double>(y);
            v[2] += sign * static_cast<double>(x * x);
            v[3] += sign * static_cast<double>(y * y);
            v[4] += sign * static_cast<double>(x * y);
        };
        if (active)
            for (int r = -pad; r <= pad; ++r) {
                if (zp) { if (r >= 0 && r < H) add_row(r, 1.0); }
                else add_row(reflect_idx(r, H), 1.0);
            }
        double acc = 0.0;                                               // group leader: SSIM sum of its 4 columns
        for (int i = 0; i < H; ++i) {
            if (i > 0 && active) {
                if (zp) {
                    if (i + pad < H) add_row(i + pad, 1.0);
                    if (i - pad - 1 >= 0) add_row(i - pad - 1, -1.0);
                } else {
                    add_row(reflect_idx(i + pad, H), 1.0);
                    add_row(reflect_idx(i - pad - 1, H), -1.0);
                }
            }
            double l[5];                                                // prefix of my column within its group, left to right
#pragma unroll
            for (int q = 0; q < 5; ++q) {
                double t = v[q];
#pragma unroll
                for (int s = 1; s < 4; ++s) {
                    const double u = shfl_up_d(t, 1);
                    if (k == s) t = u + t;
                }
                l[q] = t;
                if (k == 3) gtot[q * 32 + g] = t;
            }
            named_bar_sync(1 + worker, 128);
#pragma unroll
            for (int q = 0; q < 5; ++q) {
                double t = gtot[q * 32 + lane];                         // every warp scans all 32 group totals
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const double u = shfl_up_d(t, d);
                    if (lane >= d) t += u;
                }
                const double base = __shfl_sync(0xffffffffu, t, g) - gtot[q * 32 + g];   // sum of the groups to my left
                if (active) P[q * (W + 1) + col + 1] = base + l[q];
                if (col == 0) P[q * (W + 1)] = 0.0;
            }
            named_bar_sync(1 + worker, 128);
            double term = 0.0;
            if (active) {
                const int lo = col - pad, hi = col + pad;
                const int a0 = lo < 0 ? 0 : lo, a1 = hi > W - 1 ? W - 1 : hi;
                double box[5];
#pragma unroll
                for (int q = 0; q < 5; ++q) {
                    const double* Pq = P + q * (W + 1);
                    double t = Pq[a1 + 1] - Pq[a0];
                    if (!zp) {
                        if (lo < 0) t += Pq[-lo + 1] - Pq[1];
                        if (hi > W - 1) t += Pq[W - 1] - Pq[2 * (W - 1) - hi];
                    }
                    box[q] = t;
                }
                term = ssim_term(box, inv_n, C1, C2);
            }
            const double t1 = __shfl_down_sync(0xffffffffu, term, 1), t2 = __shfl_down_sync(0xffffffffu, term, 2),
                         t3 = __shfl_down_sync(0xffffffffu, term, 3);
            if (k == 0) {
                if (col < W) acc += term;
                if (col + 1 < W) acc += t1;
                if (col + 2 < W) acc += t2;
                if (col + 3 < W) acc += t3;
            }
        }
        if (k == 0) gtot[g] = acc;                                      // the last row's scan reads of gtot are behind its 2nd barrier
        named_bar_sync(1 + worker, 128);
        if (wwarp == 0) {
            double t = gtot[lane];
            for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
            if (lane == 0) p.scores[static_cast<long long>(b) * (n_ws + 2) + j] = t / (static_cast<double>(H) * W);
        }
        named_bar_sync(1 + worker, 128);                                // gtot is rewritten by the next window size
    }
}

}  // namespace
}  // namespace adsr

namespace {
int launch_score(adsr::ScoreParams& p, int B, const int32_t* host_ws_list, int n_ws, cudaStream_t st) {
    using namespace adsr;
    if (B <= 0) return ADSR_OK;
    if (n_ws < 0 || n_ws > kMaxWs || (p.C != 1 && p.C != 3) || p.W > 1024 || p.W < 2 || p.H < 2) return ADSR_ERR_BAD_SHAPE;
    for (int i = 0; i < kMaxWs; ++i) p.wl.ws[i] = 1;
    for (int i = 0; i < n_ws; ++i) {
        const int ws = host_ws_list[i];
        if (ws < 1 || (ws % 2) == 0 || ws / 2 >= p.H || ws / 2 >= p.W) return ADSR_ERR_BAD_SHAPE;
        p.wl.ws[i] = ws;
    }
    p.n_ws = n_ws;
    // one CTA per image when the gray planes fit shared memory (the evaluator's 128 x 128 crops)
    const size_t fast_smem = (32 + kFastWarps * 5 * static_cast<size_t>(p.W + (p.W >> 4) + 1)) * sizeof(double) +
                             2 * static_cast<size_t>(p.H) * p.W * sizeof(float);
    if (p.W <= 128 && fast_smem <= 227 * 1024 && n_ws > 0) {
        if (ensure_dynamic_smem(score_images_fast_kernel, static_cast<int>(fast_smem)) != cudaSuccess)
            return ADSR_ERR_CUDA;
        // a CTA costs ~0.3 units (gray planes + MSE) + one unit per window size of its busiest warp; with few images and more
        // window sizes than warps two CTAs per image halve the sweep, with many images the extra waves would cost more
        static int sms = 0;
        if (sms == 0) {
            int dev = 0;
            if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
                sms = 148;
        }
        auto cost = [&](int parts) {
            const int waves = (B * parts + sms - 1) / sms;
            const int per_worker = (n_ws + kFastWarps * parts - 1) / (kFastWarps * parts);
            return waves * (0.3 + per_worker);
        };
        const size_t fast4_smem = (32 + kFastWorkers * (5 * 32 + 5 * static_cast<size_t>(p.W + 1))) * sizeof(double) +
                                  2 * static_cast<size_t>(p.H) * p.W * sizeof(float);
        if (2 * B <= sms && n_ws > kFastWorkers && fast4_smem <= 227 * 1024) {
            // the batch leaves more than half of the SMs idle: latency per window size counts, not instructions per SM
            if (ensure_dynamic_smem(score_images_fast4_kernel, static_cast<int>(fast4_smem)) != cudaSuccess) return ADSR_ERR_CUDA;
            score_images_fast4_kernel<<<dim3(B, 2), 1024, fast4_smem, st>>>(p);
            return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
        }
        const int parts = (n_ws > kFastWarps && cost(2) < cost(1)) ? 2 : 1;
        score_images_fast_kernel<<<dim3(B, parts), kFastThreads, fast_smem, st>>>(p);
        return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
    }
    const int threads = ((p.W + 31) / 32) * 32;
    const size_t smem = (32 + 2 * 5 * 32 + 2 * 5 * static_cast<size_t>(p.W + 1)) * sizeof(double);
    if (smem > 48 * 1024) {
        if (ensure_dynamic_smem(score_images_kernel, static_cast<int>(smem)) != cudaSuccess)
            return ADSR_ERR_CUDA;
    }
    dim3 grid(n_ws + 1, B);
    score_images_kernel<<<grid, threads, smem, st>>>(p);
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}
}  // namespace

extern "C" int adsr_score_images(const uint8_t* sr_u8_hwc, const uint8_t* hr_u8_hwc, int B, int H, int W, int C,
                                 const int32_t* host_ws_list, int n_ws, double* scores, void* stream) {
    adsr::ScoreParams p{};
    const long long sb = static_cast<long long>(H) * W * C;
    p.sr = {sr_u8_hwc, sb, static_cast<long long>(W) * C, C, 1, 0, 255.0f, 0};
    p.hr = {hr_u8_hwc, sb, static_cast<long long>(W) * C, C, 1, 0, 255.0f, 0};
    p.H = H; p.W = W; p.C = C;
    p.zero_pad = 0;
    p.C1 = 0.01 * 0.01; p.C2 = 0.03 * 0.03; p.psnr_peak2 = 1.0;
    p.scores = scores;
    return launch_score(p, B, host_ws_list, n_ws, static_cast<cudaStream_t>(stream));
}

extern "C" int adsr_score_images_strided(const void* sr, const void* hr, int is_f32, int B, int H, int W, int C,
                                         const int64_t* host_strides_sr, const int64_t* host_strides_hr, float div,
                                         int clamp01, int zero_pad, double c1, double c2, double psnr_peak,
                                         const int32_t* host_ws_list, int n_ws, double* scores, void* stream) {
    adsr::ScoreParams p{};
    p.sr = {sr, host_strides_sr[0], host_strides_sr[1], host_strides_sr[2], host_strides_sr[3], is_f32, div, clamp01};
    p.hr = {hr, host_strides_hr[0], host_strides_hr[1], host_strides_hr[2], host_strides_hr[3], is_f32, div, clamp01};
    p.H = H; p.W = W; p.C = C;
    p.zero_pad = zero_pad;
    p.C1 = c1; p.C2 = c2; p.psnr_peak2 = psnr_peak * psnr_peak;
    p.scores = scores;
    return launch_score(p, B, host_ws_list, n_ws, static_cast<cudaStream_t>(stream));
}

extern "C" int adsr_validate_images(const void* sr, const void* hr, int B, int H, int W, int C, const int64_t* host_strides_sr,
                                    const int64_t* host_strides_hr, float rgb_range, int win_size, double* scores, void* stream) {
    if (rgb_range <= 0.f) return ADSR_ERR_BAD_SHAPE;
    adsr::ScoreParams p{};
    p.sr = {sr, host_strides_sr[0], host_strides_sr[1], host_strides_sr[2], host_strides_sr[3], 1, rgb_range, 1, 255.0f / rgb_range};
    p.hr = {hr, host_strides_hr[0], host_strides_hr[1], host_strides_hr[2], host_strides_hr[3], 1, rgb_range, 1, 0.f};
    p.H = H; p.W = W; p.C = C;
    p.zero_pad = 1;
    p.mse_noclamp = 1;
    p.C1 = 0.01 * 0.01 * 255.0 * 255.0; p.C2 = 0.03 * 0.03 * 255.0 * 255.0; p.psnr_peak2 = 1.0;
    p.scores = scores;
    const int32_t ws = win_size;
    return launch_score(p, B, &ws, 1, static_cast<cudaStream_t>(stream));
}
