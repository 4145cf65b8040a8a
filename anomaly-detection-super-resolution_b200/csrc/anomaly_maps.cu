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
// Kernel D (map_max_kernel): one CTA per image, max of each final map.
//
// adsr_gms_map: the multi-scale gradient-magnitude-similarity (MSGMS) map of RIAD (Zavrtanik et al., Pattern Recognition 2021), built
// on GMSD (Xue et al., IEEE TIP 2014), on the gray plane of the 1 - SSIM map:
//   gms_pyramid_kernel: one CTA per (image, 16 x 64 tile); gray planes of both images (level 0) and the three 2x2-mean levels
//     (avg_pool2d(2, 2), odd sizes floored) of both images to the workspace, each level from the one below it in shared memory.
//   gms_levels_kernel: thread per pixel of levels 1-3: 1 - GMS of the zero-padded Prewitt gradient magnitudes.
//   gms_combine_kernel: thread per output pixel: level-0 1 - GMS from the 3 x 3 gray neighbourhoods plus the bilinear
//     (align_corners=False) samples of levels 1-3, accumulated in level order, times 1/4.
//   then the shared Gaussian passes (sigma > 0; the scratch aliases the level-0 gray planes, dead by then) and map_max_kernel.
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

template <int NM>
struct MapPtrs { const float* m[NM]; };

// map_max[NM * b + q] = max of map q of image b
template <int NM>
__global__ void __launch_bounds__(kMaxThreads) map_max_kernel(const MapPtrs<NM> maps, int HW, double* __restrict__ map_max) {
    __shared__ float red[NM][kMaxThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float mx[NM];
#pragma unroll
    for (int q = 0; q < NM; ++q) mx[q] = -INFINITY;
    for (int k = tid; k < HW; k += kMaxThreads)
#pragma unroll
        for (int q = 0; q < NM; ++q) mx[q] = fmaxf(mx[q], maps.m[q][static_cast<long long>(b) * HW + k]);
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int q = 0; q < NM; ++q) mx[q] = fmaxf(mx[q], __shfl_xor_sync(0xffffffffu, mx[q], o));
    if (lane == 0)
#pragma unroll
        for (int q = 0; q < NM; ++q) red[q][warp] = mx[q];
    __syncthreads();
    if (tid == 0)
#pragma unroll
        for (int q = 0; q < NM; ++q) {
            for (int w = 1; w < kMaxThreads / 32; ++w) mx[q] = fmaxf(mx[q], red[q][w]);
            map_max[NM * b + q] = static_cast<double>(mx[q]);
        }
}

// Radius int(4 sigma + 0.5) of the Gaussian of sigma (0 = no smoothing), or -1 when sigma is NaN or negative, or its radius is over
// kMaxGaussRadius or >= min_hw (the half-sample reflection covers one image length)
int gauss_radius(float sigma, int min_hw) {
    if (!(sigma >= 0.0f) || sigma > static_cast<float>(kMaxGaussRadius)) return -1;      // also rejects NaN
    const int r = sigma > 0.0f ? static_cast<int>(4.0 * static_cast<double>(sigma) + 0.5) : 0;
    if (sigma > 0.0f && (r > kMaxGaussRadius || r >= min_hw)) return -1;
    return r;
}

// scipy.ndimage._gaussian_kernel1d(sigma, 0, r): exp(-0.5 x^2 / sigma^2) over x = -r .. r, normalised to sum 1
GaussTaps gauss_taps(float sigma, int r) {
    GaussTaps t{};
    const double s2 = static_cast<double>(sigma) * static_cast<double>(sigma);
    double sum = 0.0;
    for (int x = -r; x <= r; ++x) sum += exp(-0.5 / s2 * static_cast<double>(x * x));
    for (int j = 0; j <= r; ++j) t.w[j] = exp(-0.5 / s2 * static_cast<double>(j * j)) / sum;
    return t;
}

// map [B, H, W] (n = B H W values) -> scratch (rows) -> map (columns)
void gauss_smooth(float* map, float* scratch, long long n, int H, int W, int r, const GaussTaps& t, cudaStream_t st) {
    const unsigned blocks = static_cast<unsigned>((n + 255) / 256);
    gauss_rows_kernel<<<blocks, 256, 0, st>>>(map, scratch, n, W, r, t);
    gauss_cols_kernel<<<blocks, 256, 0, st>>>(scratch, map, n, H, W, r, t);
}

// ---- MSGMS map
constexpr int kGmsLevels = 4;                       // scales 1, 1/2, 1/4, 1/8 (RIAD)
constexpr int kGmsTileRows = 16, kGmsTileCols = 64;  // level-0 tile of the pyramid kernel: multiples of 2^(kGmsLevels - 1)
constexpr int kGmsThreads = 256;
constexpr float kGmsC = 0.0026f;                    // GMSD's T = 170 on the 0-255 scale: 170 / 255^2

struct GmsPlanes {                                  // carved from the caller's workspace by gms_planes()
    int h[kGmsLevels], w[kGmsLevels];               // level k is (H >> k) x (W >> k)
    float* hr[kGmsLevels];                          // gray pyramid of the HR images, fp32 [B, h_k, w_k]
    float* sr[kGmsLevels];                          // gray pyramid of the SR images
    float* d[kGmsLevels];                           // 1 - GMS at levels 1 .. 3 (d[0] unused: the combine pass forms it)
};

// floats of the workspace: both gray pyramids plus the 1 - GMS planes of levels 1 .. 3; also fits the Gaussian scratch (B H W)
long long gms_workspace_floats(long long B, int H, int W) {
    long long n = 2 * B * H * W;
    for (int k = 1; k < kGmsLevels; ++k) n += 3 * B * (H >> k) * (W >> k);
    return n;
}

GmsPlanes gms_planes(float* ws, long long B, int H, int W) {
    GmsPlanes p{};
    for (int k = 0; k < kGmsLevels; ++k) {
        p.h[k] = H >> k;
        p.w[k] = W >> k;
        const long long n = B * p.h[k] * p.w[k];
        p.hr[k] = ws;
        p.sr[k] = ws + n;
        ws += 2 * n;
        if (k > 0) {
            p.d[k] = ws;
            ws += n;
        }
    }
    return p;
}

// dst tile (rows x cols of level k, origin (i0, j0)) = 2 x 2 means of the src tile of level k - 1 (pitch 2 cols), both images
// (src / dst: [2][tile]); a level-k pixel exists only when its whole 2 x 2 block does (avg_pool2d floors odd sizes)
__device__ __forceinline__ void gms_pool_tile(const float* src, float* dst, int rows, int cols, int k, long long b, int i0, int j0,
                                              const GmsPlanes& P) {
    const int h = P.h[k], w = P.w[k];
    float* const hr_k = P.hr[k];
    float* const sr_k = P.sr[k];
    for (int e = threadIdx.x; e < 2 * rows * cols; e += kGmsThreads) {
        const int img = e / (rows * cols), rem = e - img * rows * cols, r = rem / cols, c = rem - r * cols;
        const int i = i0 + r, j = j0 + c;
        if (i >= h || j >= w) continue;
        const float* s = src + img * 4 * rows * cols + 2 * r * 2 * cols + 2 * c;
        const float v = (((s[0] + s[1]) + s[2 * cols]) + s[2 * cols + 1]) * 0.25f;
        if (dst != nullptr) dst[img * rows * cols + r * cols + c] = v;
        (img ? sr_k : hr_k)[(b * h + i) * w + j] = v;
    }
}

// min 4 CTAs / SM: without it ptxas holds this kernel to 32 registers and spills
__global__ void __launch_bounds__(kGmsThreads, 4) gms_pyramid_kernel(const uint8_t* __restrict__ sr, const uint8_t* __restrict__ hr, int C,
                                                                 int tiles_x, int tiles_per_image, const GmsPlanes P) {
    __shared__ float t0[2 * kGmsTileRows * kGmsTileCols];
    __shared__ float t1[2 * (kGmsTileRows / 2) * (kGmsTileCols / 2)];
    __shared__ float t2[2 * (kGmsTileRows / 4) * (kGmsTileCols / 4)];
    const long long b = blockIdx.x / tiles_per_image;
    const int t = blockIdx.x - static_cast<int>(b) * tiles_per_image;
    const int i0 = (t / tiles_x) * kGmsTileRows, j0 = (t % tiles_x) * kGmsTileCols;
    const int H = P.h[0], W = P.w[0];
    constexpr int n0 = kGmsTileRows * kGmsTileCols;
    for (int e = threadIdx.x; e < n0; e += kGmsThreads) {           // a warp reads 32 consecutive pixels of one row
        const int r = e / kGmsTileCols, c = e - r * kGmsTileCols, i = i0 + r, j = j0 + c;
        if (i >= H || j >= W) continue;
        const long long px = (b * H + i) * W + j;
        const float x = gray01(hr + px * C, C), y = gray01(sr + px * C, C);
        P.hr[0][px] = x;
        P.sr[0][px] = y;
        t0[e] = x;
        t0[n0 + e] = y;
    }
    __syncthreads();
    gms_pool_tile(t0, t1, kGmsTileRows / 2, kGmsTileCols / 2, 1, b, i0 / 2, j0 / 2, P);
    __syncthreads();
    gms_pool_tile(t1, t2, kGmsTileRows / 4, kGmsTileCols / 4, 2, b, i0 / 4, j0 / 4, P);
    __syncthreads();
    gms_pool_tile(t2, nullptr, kGmsTileRows / 8, kGmsTileCols / 8, 3, b, i0 / 8, j0 / 8, P);
}

// Prewitt gradient magnitude of plane p (h x w) at (i, j): F.conv2d(p, [[1/3, 0, -1/3]] * 3 and its transpose, padding=1), then
// sqrt(gx^2 + gy^2 + 1e-12)
__device__ __forceinline__ float prewitt_mag(const float* __restrict__ p, int h, int w, int i, int j) {
    float v[3][3];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const int y = i + a - 1, x = j + c - 1;
            v[a][c] = (y >= 0 && y < h && x >= 0 && x < w) ? __ldg(p + static_cast<long long>(y) * w + x) : 0.0f;
        }
    const float gx = ((v[0][0] - v[0][2]) + (v[1][0] - v[1][2]) + (v[2][0] - v[2][2])) / 3.0f;
    const float gy = ((v[0][0] - v[2][0]) + (v[0][1] - v[2][1]) + (v[0][2] - v[2][2])) / 3.0f;
    return sqrtf(gx * gx + gy * gy + 1e-12f);
}

// 1 - (2 a b + c) / (a^2 + b^2 + c); products and sums rounded one by one (no FMA contraction): for a == b the numerator and the
// denominator are the same float (2 a * b = 2 (a * a) exactly), so an identical pair gives exactly 0
__device__ __forceinline__ float one_minus_gms(float a, float b) {
    const float num = __fadd_rn(__fmul_rn(__fmul_rn(2.0f, a), b), kGmsC);
    const float den = __fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)), kGmsC);
    return 1.0f - num / den;
}

template <int K>
__device__ __forceinline__ void gms_level_pixel(const GmsPlanes& P, int idx) {
    const int h = P.h[K], w = P.w[K];
    const int b = idx / (h * w), rem = idx - b * h * w, i = rem / w, j = rem - i * w;
    const long long img = static_cast<long long>(b) * h * w;
    P.d[K][idx] = one_minus_gms(prewitt_mag(P.hr[K] + img, h, w, i, j), prewitt_mag(P.sr[K] + img, h, w, i, j));
}

// thread per pixel of levels 1, 2, 3 (in that order)
__global__ void __launch_bounds__(256) gms_levels_kernel(const GmsPlanes P, int B) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int n1 = B * P.h[1] * P.w[1], n2 = B * P.h[2] * P.w[2], n3 = B * P.h[3] * P.w[3];
    if (idx < n1) gms_level_pixel<1>(P, idx);
    else if (idx < n1 + n2) gms_level_pixel<2>(P, idx - n1);
    else if (idx < n1 + n2 + n3) gms_level_pixel<3>(P, idx - n1 - n2);
}

// F.interpolate(bilinear, align_corners=False) source position of output index o on an axis of n_in -> n_out: i0, i1, weight of i1
__device__ __forceinline__ void bilinear_axis(int o, int n_in, int n_out, int& i0, int& i1, float& l1) {
    const float scale = static_cast<float>(n_in) / static_cast<float>(n_out);
    const float src = fmaxf(scale * (static_cast<float>(o) + 0.5f) - 0.5f, 0.0f);
    i0 = static_cast<int>(src);
    i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
    l1 = src - static_cast<float>(i0);
}

__global__ void __launch_bounds__(256) gms_combine_kernel(const GmsPlanes P, int n, float* __restrict__ out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const int H = P.h[0], W = P.w[0], hw = H * W;
    const int b = idx / hw, rem = idx - b * hw, i = rem / W, j = rem - i * W;
    const long long img = static_cast<long long>(b) * hw;
    float acc = one_minus_gms(prewitt_mag(P.hr[0] + img, H, W, i, j), prewitt_mag(P.sr[0] + img, H, W, i, j));
#pragma unroll
    for (int k = 1; k < kGmsLevels; ++k) {
        const int h = P.h[k], w = P.w[k];
        int y0, y1, x0, x1;
        float ly, lx;
        bilinear_axis(i, h, H, y0, y1, ly);
        bilinear_axis(j, w, W, x0, x1, lx);
        const float* d = P.d[k] + static_cast<long long>(b) * h * w;
        const float top = (1.0f - lx) * __ldg(d + y0 * w + x0) + lx * __ldg(d + y0 * w + x1);
        const float bot = (1.0f - lx) * __ldg(d + y1 * w + x0) + lx * __ldg(d + y1 * w + x1);
        acc += (1.0f - ly) * top + ly * bot;
    }
    out[idx] = acc * 0.25f;
}

}  // namespace
}  // namespace adsr

extern "C" int adsr_anomaly_maps(const uint8_t* sr_u8_hwc, const uint8_t* hr_u8_hwc, int B, int H, int W, int C, int win_size,
                                 float sigma, float* ssim_map, float* se_map, float* scratch, double* map_max, void* stream) {
    using namespace adsr;
    if ((C != 1 && C != 3) || H < 2 || W < 2 || W > 1024 || B < 0) return ADSR_ERR_BAD_SHAPE;
    const int min_hw = H < W ? H : W;
    if (win_size < 1 || (win_size % 2) == 0 || win_size / 2 >= min_hw) return ADSR_ERR_BAD_SHAPE;
    const int r = gauss_radius(sigma, min_hw);
    if (r < 0 || (sigma > 0.0f && scratch == nullptr)) return ADSR_ERR_BAD_SHAPE;
    if (B == 0) return ADSR_OK;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);

    RawParams p{sr_u8_hwc, hr_u8_hwc, H, W, C, win_size, ssim_map, se_map};
    const int threads = ((W + 31) / 32) * 32;
    const size_t smem = (2 * 5 * 32 + 2 * 5 * static_cast<size_t>(W + 1)) * sizeof(double);
    if (smem > 48 * 1024 && ensure_dynamic_smem(anomaly_maps_raw_kernel, static_cast<int>(smem)) != cudaSuccess) return ADSR_ERR_CUDA;
    anomaly_maps_raw_kernel<<<dim3((H + kBandRows - 1) / kBandRows, B), threads, smem, st>>>(p);
    if (cudaGetLastError() != cudaSuccess) return ADSR_ERR_LAUNCH;

    if (sigma > 0.0f) {
        const GaussTaps t = gauss_taps(sigma, r);
        const long long n = static_cast<long long>(B) * H * W;
        gauss_smooth(ssim_map, scratch, n, H, W, r, t, st);
        gauss_smooth(se_map, scratch, n, H, W, r, t, st);
        if (cudaGetLastError() != cudaSuccess) return ADSR_ERR_LAUNCH;
    }
    map_max_kernel<2><<<B, kMaxThreads, 0, st>>>(MapPtrs<2>{{ssim_map, se_map}}, H * W, map_max);
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}

extern "C" int64_t adsr_gms_workspace_bytes(int B, int H, int W) {
    if (B < 0 || H < 0 || W < 0) return -1;
    return adsr::gms_workspace_floats(B, H, W) * static_cast<int64_t>(sizeof(float));
}

extern "C" int adsr_gms_map(const uint8_t* sr_u8_hwc, const uint8_t* hr_u8_hwc, int B, int H, int W, int C, float sigma, float* gms_map,
                            double* map_max, void* workspace, void* stream) {
    using namespace adsr;
    if ((C != 1 && C != 3) || H < 8 || W < 8 || B < 0 || static_cast<long long>(B) * H * W >= (1LL << 31)) return ADSR_ERR_BAD_SHAPE;
    const int r = gauss_radius(sigma, H < W ? H : W);
    if (r < 0) return ADSR_ERR_BAD_SHAPE;
    if (B == 0) return ADSR_OK;
    if (workspace == nullptr || gms_map == nullptr || map_max == nullptr) return ADSR_ERR_BAD_SHAPE;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const GmsPlanes P = gms_planes(static_cast<float*>(workspace), B, H, W);

    const int tiles_x = (W + kGmsTileCols - 1) / kGmsTileCols;
    const int tiles_per_image = tiles_x * ((H + kGmsTileRows - 1) / kGmsTileRows);
    gms_pyramid_kernel<<<static_cast<unsigned>(static_cast<long long>(B) * tiles_per_image), kGmsThreads, 0, st>>>(
        sr_u8_hwc, hr_u8_hwc, C, tiles_x, tiles_per_image, P);
    int n_coarse = 0;
    for (int k = 1; k < kGmsLevels; ++k) n_coarse += B * P.h[k] * P.w[k];
    gms_levels_kernel<<<(n_coarse + 255) / 256, 256, 0, st>>>(P, B);
    const int n = B * H * W;
    gms_combine_kernel<<<(n + 255) / 256, 256, 0, st>>>(P, n, gms_map);
    if (cudaGetLastError() != cudaSuccess) return ADSR_ERR_LAUNCH;
    if (sigma > 0.0f) {
        gauss_smooth(gms_map, P.hr[0], n, H, W, r, gauss_taps(sigma, r), st);   // the level-0 gray planes are dead after the combine
        if (cudaGetLastError() != cudaSuccess) return ADSR_ERR_LAUNCH;
    }
    map_max_kernel<1><<<B, kMaxThreads, 0, st>>>(MapPtrs<1>{{gms_map}}, H * W, map_max);
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}
