// Per-pixel anomaly maps of uint8 HWC SR / HR pairs: the 1 - SSIM map of ONE window size and the squared-error map, optionally
// smoothed by a Gaussian, plus the per-image maximum of each map.  The scorer (scoring.cu) computes the same per-pixel SSIM values
// and averages them away; here they are stored.
//
// Kernel A (anomaly_maps_raw_kernel): grid = (row bands, B).  One thread owns one image column and walks down the band's rows keeping
// the five vertical window sums (x, y, x^2, y^2, xy) as fp64 running sums (np.pad(mode="reflect") rows at the image borders); per row
// the column sums become prefix sums across the row (warp shuffles + one shared-memory hop) and each horizontal window sum is a
// difference of two prefix values -- the formulas of score_images_kernel: gray via gray_at, values / 255, products in fp32, sums in
// fp64, C1 = 1e-4, C2 = 9e-4.  1 - SSIM is formed in fp64 and stored as fp32, so the map's mean is 1 - the scorer's SSIM.  Then the
// same thread writes the band's squared-error pixels mean_c (sr/255 - hr/255)^2, with d formed in fp32 like the MSE term.
// Kernels B / C (gauss_rows_kernel, gauss_cols_kernel): the separable Gaussian of scipy.ndimage.gaussian_filter(map, sigma,
// mode="reflect", truncate=4.0): radius r = int(4 sigma + 0.5), taps exp(-x^2 / 2 sigma^2) / sum computed in double on the host,
// half-sample reflection (d c b a | a b c d), fp64 accumulation and an fp32 result after each pass (as scipy does for float32 input).
// Each map goes map -> scratch (rows) -> map (columns).
// Kernel D (map_max_kernel): one CTA per image, max of both final maps.
// Everything is a pure function of the image's own pixels with fixed summation orders: deterministic and batch independent.
#include "adsr_kernels.h"

namespace adsr {
namespace {

constexpr int kMaxGaussRadius = 64;        // taps table in the kernel parameters: (r + 1) doubles
constexpr int kBandRows = 16;              // output rows per CTA of the raw-map kernel

__device__ __forceinline__ int reflect_np(int i, int n) {        // np.pad(mode="reflect"), |overhang| < n
    if (i < 0) i = -i;
    if (i >= n) i = 2 * (n - 1) - i;
    return i;
}

__device__ __forceinline__ int reflect_scipy(int i, int n) {     // scipy.ndimage mode="reflect" (half-sample), |overhang| <= n
    if (i < 0) i = -i - 1;
    if (i >= n) i = 2 * n - 1 - i;
    return i;
}

__device__ __forceinline__ float u8_01(const uint8_t* p) { return static_cast<float>(__ldg(p)) / 255.0f; }

// gray value as score_images builds it: channels dotted with the fp32 (65.738, 129.057, 25.064)/256 coefficients; one channel: as is
__device__ __forceinline__ float gray01(const uint8_t* p, int C) {
    if (C == 1) return u8_01(p);
    const float c0 = 65.738f / 256.0f, c1 = 129.057f / 256.0f, c2 = 25.064f / 256.0f;
    return fmaf(u8_01(p + 2), c2, fmaf(u8_01(p + 1), c1, u8_01(p) * c0));
}

struct RawParams {
    const uint8_t* sr;
    const uint8_t* hr;
    int H, W, C, ws;
    float* ssim_map;
    float* se_map;
};

__global__ void __launch_bounds__(1024) anomaly_maps_raw_kernel(const RawParams p) {
    const int H = p.H, W = p.W, C = p.C, ws = p.ws, pad = ws / 2;
    extern __shared__ double sm[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.y, r0 = blockIdx.x * kBandRows, r1 = min(H, r0 + kBandRows);
    const long long img = static_cast<long long>(b) * H * W;
    const uint8_t* sr = p.sr + img * C;
    const uint8_t* hr = p.hr + img * C;
    const int col = tid;                                 // one column per thread (blockDim.x >= W)
    const bool active = col < W;
    double* wtot = sm;                                   // [2][5][32] per-warp totals (double buffered)
    double* pref = wtot + 2 * 5 * 32;                    // [2][5][W + 1] prefix sums (double buffered)
    const double inv_n = 1.0 / (static_cast<double>(ws) * ws);
    const double C1 = 1e-4, C2 = 9e-4;

    double v[5] = {0, 0, 0, 0, 0};
    auto add_row = [&](int r, double sign) {
        const long long off = (static_cast<long long>(r) * W + col) * C;
        const float x = gray01(hr + off, C);             // x = reference (HR)
        const float y = gray01(sr + off, C);             // y = SR
        v[0] += sign * static_cast<double>(x);
        v[1] += sign * static_cast<double>(y);
        v[2] += sign * static_cast<double>(x * x);      // products are formed in fp32 like `ref * ref`
        v[3] += sign * static_cast<double>(y * y);
        v[4] += sign * static_cast<double>(x * y);
    };
    if (active)
        for (int r = r0 - pad; r <= r0 + pad; ++r) add_row(reflect_np(r, H), 1.0);

    for (int i = r0; i < r1; ++i) {
        const int bufi = i & 1;
        if (i > r0 && active) {
            add_row(reflect_np(i + pad, H), 1.0);
            add_row(reflect_np(i - pad - 1, H), -1.0);
        }
        // inclusive scan of the 5 column sums across the row
        double s[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            double t = active ? v[q] : 0.0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double u = __shfl_up_sync(0xffffffffu, t, d);
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
                if (lo < 0) t += Pq[-lo + 1] - Pq[1];                       // reflected columns 1 .. -lo
                if (hi > W - 1) t += Pq[W - 1] - Pq[2 * (W - 1) - hi];      // reflected columns 2(W-1)-hi .. W-2
                box[q] = t * inv_n;
            }
            // products rounded on their own (no FMA contraction): for an identical pair m11 = m22 = m12 and s1 = s2 = s12, so the
            // numerator and the denominator are the same double and the map is exactly 0
            const double mu1 = box[0], mu2 = box[1];
            const double m11 = __dmul_rn(mu1, mu1), m22 = __dmul_rn(mu2, mu2), m12 = __dmul_rn(mu1, mu2);
            const double s1 = box[2] - m11, s2 = box[3] - m22, s12 = box[4] - m12;
            const double ssim = __dmul_rn(__dmul_rn(2.0, m12) + C1, __dmul_rn(2.0, s12) + C2) / __dmul_rn(m11 + m22 + C1, s1 + s2 + C2);
            const long long o = img + static_cast<long long>(i) * W + col;
            p.ssim_map[o] = static_cast<float>(1.0 - ssim);
        }
    }
    // squared-error map of the band
    if (active)
        for (int i = r0; i < r1; ++i) {
            const long long off = (static_cast<long long>(i) * W + col) * C;
            double se = 0.0;
            for (int ch = 0; ch < C; ++ch) {
                const float d = u8_01(sr + off + ch) - u8_01(hr + off + ch);
                se += static_cast<double>(d * d);       // (ref - out) ** 2 on float32 arrays
            }
            p.se_map[img + static_cast<long long>(i) * W + col] = static_cast<float>(se / C);
        }
}

struct GaussTaps { double w[kMaxGaussRadius + 1]; };   // w[j] = weight of offset +-j

// scipy's correlate1d order for a symmetric kernel: w0 x[i] + sum_{j = r .. 1} w_j (x[i - j] + x[i + j]), in double
__global__ void __launch_bounds__(256) gauss_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, long long n, int W,
                                                         int r, const GaussTaps t) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const long long row = idx / W;
    const int c = static_cast<int>(idx - row * W);
    const float* s = src + row * W;
    double acc = t.w[0] * static_cast<double>(s[c]);
    for (int j = r; j >= 1; --j)
        acc += (static_cast<double>(s[reflect_scipy(c - j, W)]) + static_cast<double>(s[reflect_scipy(c + j, W)])) * t.w[j];
    dst[idx] = static_cast<float>(acc);
}

__global__ void __launch_bounds__(256) gauss_cols_kernel(const float* __restrict__ src, float* __restrict__ dst, long long n, int H,
                                                         int W, int r, const GaussTaps t) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const long long hw = static_cast<long long>(H) * W;
    const long long b = idx / hw;
    const int rem = static_cast<int>(idx - b * hw);
    const int i = rem / W, c = rem - i * W;
    const float* s = src + b * hw + c;
    double acc = t.w[0] * static_cast<double>(s[static_cast<long long>(i) * W]);
    for (int j = r; j >= 1; --j)
        acc += (static_cast<double>(s[static_cast<long long>(reflect_scipy(i - j, H)) * W]) +
                static_cast<double>(s[static_cast<long long>(reflect_scipy(i + j, H)) * W])) * t.w[j];
    dst[idx] = static_cast<float>(acc);
}

constexpr int kMaxThreads = 512;

__global__ void __launch_bounds__(kMaxThreads) map_max_kernel(const float* __restrict__ ssim_map, const float* __restrict__ se_map,
                                                              int HW, double* __restrict__ map_max) {
    __shared__ float red[2][kMaxThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* a = ssim_map + static_cast<long long>(b) * HW;
    const float* e = se_map + static_cast<long long>(b) * HW;
    float ma = -INFINITY, me = -INFINITY;
    for (int k = tid; k < HW; k += kMaxThreads) {
        ma = fmaxf(ma, a[k]);
        me = fmaxf(me, e[k]);
    }
    for (int o = 16; o > 0; o >>= 1) {
        ma = fmaxf(ma, __shfl_xor_sync(0xffffffffu, ma, o));
        me = fmaxf(me, __shfl_xor_sync(0xffffffffu, me, o));
    }
    if (lane == 0) { red[0][warp] = ma; red[1][warp] = me; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < kMaxThreads / 32; ++w) { ma = fmaxf(ma, red[0][w]); me = fmaxf(me, red[1][w]); }
        map_max[2 * b] = static_cast<double>(ma);
        map_max[2 * b + 1] = static_cast<double>(me);
    }
}

}  // namespace
}  // namespace adsr

extern "C" int adsr_anomaly_maps(const uint8_t* sr_u8_hwc, const uint8_t* hr_u8_hwc, int B, int H, int W, int C, int win_size,
                                 float sigma, float* ssim_map, float* se_map, float* scratch, double* map_max, void* stream) {
    using namespace adsr;
    if ((C != 1 && C != 3) || H < 2 || W < 2 || W > 1024 || B < 0) return ADSR_ERR_BAD_SHAPE;
    const int min_hw = H < W ? H : W;
    if (win_size < 1 || (win_size % 2) == 0 || win_size / 2 >= min_hw) return ADSR_ERR_BAD_SHAPE;
    if (!(sigma >= 0.0f) || sigma > static_cast<float>(kMaxGaussRadius)) return ADSR_ERR_BAD_SHAPE;   // also rejects NaN
    const int r = sigma > 0.0f ? static_cast<int>(4.0 * static_cast<double>(sigma) + 0.5) : 0;
    if (sigma > 0.0f && (r > kMaxGaussRadius || r >= min_hw || scratch == nullptr)) return ADSR_ERR_BAD_SHAPE;
    if (B == 0) return ADSR_OK;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);

    RawParams p{sr_u8_hwc, hr_u8_hwc, H, W, C, win_size, ssim_map, se_map};
    const int threads = ((W + 31) / 32) * 32;
    const size_t smem = (2 * 5 * 32 + 2 * 5 * static_cast<size_t>(W + 1)) * sizeof(double);
    if (smem > 48 * 1024 && ensure_dynamic_smem(anomaly_maps_raw_kernel, static_cast<int>(smem)) != cudaSuccess) return ADSR_ERR_CUDA;
    anomaly_maps_raw_kernel<<<dim3((H + kBandRows - 1) / kBandRows, B), threads, smem, st>>>(p);
    if (cudaGetLastError() != cudaSuccess) return ADSR_ERR_LAUNCH;

    if (sigma > 0.0f) {
        // scipy.ndimage._gaussian_kernel1d(sigma, 0, r): exp(-0.5 x^2 / sigma^2) over x = -r .. r, normalised to sum 1
        GaussTaps t{};
        const double s2 = static_cast<double>(sigma) * static_cast<double>(sigma);
        double sum = 0.0;
        for (int x = -r; x <= r; ++x) sum += exp(-0.5 / s2 * static_cast<double>(x * x));
        for (int j = 0; j <= r; ++j) t.w[j] = exp(-0.5 / s2 * static_cast<double>(j * j)) / sum;
        const long long n = static_cast<long long>(B) * H * W;
        const unsigned blocks = static_cast<unsigned>((n + 255) / 256);
        float* const maps[2] = {ssim_map, se_map};
        for (float* m : maps) {
            gauss_rows_kernel<<<blocks, 256, 0, st>>>(m, scratch, n, W, r, t);
            gauss_cols_kernel<<<blocks, 256, 0, st>>>(scratch, m, n, H, W, r, t);
        }
        if (cudaGetLastError() != cudaSuccess) return ADSR_ERR_LAUNCH;
    }
    map_max_kernel<<<B, kMaxThreads, 0, st>>>(ssim_map, se_map, H * W, map_max);
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}
