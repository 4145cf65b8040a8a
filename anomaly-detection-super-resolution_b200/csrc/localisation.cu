// Localisation metrics of one anomaly map over a whole test set: pixel AUROC, AU-PRO@alpha, pixel AP and F1-max with its threshold,
// exact (no threshold binning) and deterministic.  All of them come from ONE descending order of all pixels by score.
//
// Sort: a stable LSD radix sort of (key, region index) pairs, 4 passes of 8 bits.  The key is the fp32 score made order-preserving and
// complemented (descending order = ascending keys; -0.0 canonicalised to +0.0), formed on the fly by the first pass, which also counts
// NaN scores, defect-free pixels and out-of-range region indices.  A pass = radix_hist_kernel (per-tile digit histogram, tile = 4096
// pixels) + radix_scan_kernel (one CTA per digit: exclusive scan of that digit's tile counts) + radix_scatter_kernel (the tile again,
// in 16 chunks of 256: stable rank inside a chunk by __match_any_sync + per-warp digit counts, then a direct scatter).  Integer counts
// only, so the order is unique: ties keep the order in which the pixels were appended.
//
// Curve: the sorted sequence is cut into tiles of 2048 pixels; a segmented scan carries, per position, the running number of
// defect-free (ok) and defect pixels and the running PRO weight (fixed point: a region's pixels add up to 2^63, one pixel of region r
// adds floor(2^63 / |r|), summed in 128 bits), plus the same three values just before the current run of equal keys began.  At the
// last pixel of a run (the next key differs) that gives the curve point (FPR, PRO) of the run's score and the point before it, so the
// run adds its trapezoid (cut at alpha) and its exact AUROC term n_def * (2 (N_ok - ok_seen) + n_ok_run) (128-bit integer).  Kernels:
// seg_tile_kernel (tile aggregates) -> seg_scan_kernel (one CTA: exclusive scan over the tiles) -> seg_curve_kernel (per-tile
// contributions) -> finish_kernel (one CTA, fixed order).  Everything is integer except the per-run area terms, which are fp64 values
// of integer prefixes added in a fixed order: bitwise the same on every run, and for the same pixel sequence however it was batched.
//
// Precision-recall, from the same run ends.  With d_k / o_k = cumulative defect / defect-free pixels at the end of run k and
// N_def = n - n_ok:
//   pixel AP  = sum_k (d_k - d_{k-1}) / N_def * d_k / (d_k + o_k)   (= sklearn.metrics.average_precision_score, ties included);
//   F1-max    = max_k 2 d_k / (d_k + o_k + N_def), the fractions compared exactly (128-bit cross products), a tie going to the
//               earlier run (higher score): a unique answer whatever the reduction order;
//   threshold = the fp32 score of that run (decoded from its key, -0.0 reported as +0.0): `score >= threshold` selects exactly the
//               pixels that reach F1-max.
// Only runs holding a defect pixel are evaluated: a run without one adds 0 to AP, and its F1 is at most that of the run before it
// (same d, larger o), equal only when both are 0, which the tie rule and the final run (d = N_def >= 1) already settle.  The AP
// terms are fp64 sums in a fixed order like the area; the F1 candidates are reduced by the exact max.
//
// Two more entry points read the scores without sorting them, for thresholds calibrated on defect-free images:
//   adsr_score_quantile: the exact k-th smallest score, by an MSD radix select over ascending keys (~desc_key), 4 passes of 8 bits.
//     A pass = select_hist_kernel (digit histogram of the pixels whose higher digits equal the running prefix: per-warp shared
//     histograms, integer atomics into one global histogram) + select_pick_kernel (one CTA: the digit that holds rank k, the new
//     prefix and the rank left inside it, kept in device memory).  No scatter: ~16 B read per pixel over the 4 passes.
//   adsr_threshold_metrics: one pass, `score >= threshold`, TP / FP / FN counts and the fixed-point PRO weight of the detected
//     defect pixels (the AU-PRO curve's quantity at one threshold), per-CTA partials added by one CTA in a fixed order.
// Both are integer-exact, deterministic and free of host synchronisation.
#include "adsr_kernels.h"

namespace adsr {
namespace {

typedef unsigned __int128 u128;
typedef unsigned long long u64;

constexpr int kThreads = 256;
constexpr int kBins = 256;                           // 8-bit digits
constexpr int kSortItems = 16;
constexpr int kSortTile = kThreads * kSortItems;     // pixels per CTA of the radix passes
constexpr int kScanItems = 8;
constexpr int kScanTile = kThreads * kScanItems;     // pixels per CTA of the curve kernels
constexpr u64 kProOne = 1ull << 63;                  // fixed-point PRO weight of one whole region
static_assert(kThreads == kBins, "one thread per digit in the scatter kernel");

// order-preserving, complemented: a larger score gives a smaller key
__device__ __forceinline__ uint32_t desc_key(float f) {
    const uint32_t u = __float_as_uint(f == 0.0f ? 0.0f : f);   // -0.0 -> +0.0
    return (u & 0x80000000u) ? u : (~u & 0x7fffffffu);
}

__device__ __forceinline__ u64 warp_sum(u64 v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// inverse of desc_key (the map is its own inverse on non-NaN keys): the fp32 score of a key, +0.0 for a zero
__device__ __forceinline__ float key_score(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? k : (~k & 0x7fffffffu));
}

// ---------------------------------------------------------------------------------------------------------- radix sort
// counters: [0] NaN scores, [1] defect-free pixels, [2] region indices outside [-1, n_regions) or of a region with size < 1
template <bool kFirst>
__global__ void __launch_bounds__(kThreads) radix_hist_kernel(const uint32_t* __restrict__ keys, const float* __restrict__ scores,
                                                              const int32_t* __restrict__ regions, const int64_t* __restrict__ sizes,
                                                              int n_regions, long long n, int shift, int n_tiles,
                                                              long long* __restrict__ hist, u64* __restrict__ counters) {
    __shared__ unsigned int h[kBins];
    __shared__ u64 cnt[3];
    const int tid = threadIdx.x;
    h[tid] = 0;
    if (kFirst && tid < 3) cnt[tid] = 0;
    __syncthreads();
    const long long base = static_cast<long long>(blockIdx.x) * kSortTile;
    u64 nan_c = 0, ok_c = 0, bad_c = 0;
#pragma unroll 4
    for (int j = 0; j < kSortItems; ++j) {
        const long long i = base + j * kThreads + tid;
        if (i >= n) break;
        uint32_t k;
        if (kFirst) {
            const float f = scores[i];
            const int r = regions[i];
            k = desc_key(f);
            nan_c += f != f;
            ok_c += r < 0;
            bad_c += r < -1 || r >= n_regions || (r >= 0 && sizes[r] < 1);
        } else {
            k = keys[i];
        }
        atomicAdd(&h[(k >> shift) & (kBins - 1)], 1u);
    }
    if (kFirst) {
        nan_c = warp_sum(nan_c), ok_c = warp_sum(ok_c), bad_c = warp_sum(bad_c);
        if ((tid & 31) == 0) {
            if (nan_c) atomicAdd(&cnt[0], nan_c);
            if (ok_c) atomicAdd(&cnt[1], ok_c);
            if (bad_c) atomicAdd(&cnt[2], bad_c);
        }
    }
    __syncthreads();
    hist[static_cast<long long>(tid) * n_tiles + blockIdx.x] = h[tid];
    if (kFirst && tid < 3 && cnt[tid]) atomicAdd(&counters[tid], cnt[tid]);
}

// CTA d: exclusive scan of hist[d][0 .. n_tiles) in place, digit total -> digit_tot[d]
__global__ void __launch_bounds__(1024) radix_scan_kernel(long long* __restrict__ hist, int n_tiles, long long* __restrict__ digit_tot) {
    __shared__ long long wsum[32];
    long long* row = hist + static_cast<long long>(blockIdx.x) * n_tiles;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    long long carry = 0;
    for (int b0 = 0; b0 < n_tiles; b0 += 1024) {
        const int i = b0 + tid;
        const long long v = i < n_tiles ? row[i] : 0;
        long long x = v;
        for (int d = 1; d < 32; d <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += u;
        }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            long long s = wsum[lane];
            for (int d = 1; d < 32; d <<= 1) {
                const long long u = __shfl_up_sync(0xffffffffu, s, d);
                if (lane >= d) s += u;
            }
            wsum[lane] = s;
        }
        __syncthreads();
        if (i < n_tiles) row[i] = carry + (warp ? wsum[warp - 1] : 0) + x - v;
        carry += wsum[31];
        __syncthreads();
    }
    if (tid == 0) digit_tot[blockIdx.x] = carry;
}

template <bool kFirst>
__global__ void __launch_bounds__(kThreads) radix_scatter_kernel(const uint32_t* __restrict__ keys_in, const int32_t* __restrict__ vals_in,
                                                                 const float* __restrict__ scores, long long n, int shift, int n_tiles,
                                                                 const long long* __restrict__ hist, const long long* __restrict__ digit_tot,
                                                                 uint32_t* __restrict__ keys_out, int32_t* __restrict__ vals_out) {
    __shared__ long long next[kBins];                   // global position of the next pixel of each digit
    __shared__ unsigned int wcnt[kThreads / 32][kBins]; // per-warp digit counts of the current chunk
    __shared__ long long wsum[kThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // digit bases = exclusive scan of the digit totals, plus this tile's offset inside each digit
    {
        const long long v = digit_tot[tid];
        long long x = v;
        for (int d = 1; d < 32; d <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += u;
        }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        long long b = 0;
        for (int w = 0; w < warp; ++w) b += wsum[w];
        next[tid] = b + x - v + hist[static_cast<long long>(tid) * n_tiles + blockIdx.x];
    }
    const unsigned lt_mask = (1u << lane) - 1u;
    const long long base = static_cast<long long>(blockIdx.x) * kSortTile;
    for (int j = 0; j < kSortItems; ++j) {
        const long long i = base + j * kThreads + tid;
        const bool valid = i < n;
        uint32_t k = 0;
        int32_t v = 0;
        if (valid) {
            k = kFirst ? desc_key(scores[i]) : keys_in[i];
            v = vals_in[i];
        }
        const int d = valid ? static_cast<int>((k >> shift) & (kBins - 1)) : kBins;   // invalid lanes only match each other
#pragma unroll
        for (int q = 0; q < kBins / 32; ++q) wcnt[warp][lane * (kBins / 32) + q] = 0;
        __syncwarp();
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(peers & lt_mask);
        if (valid && rank == 0) wcnt[warp][d] = __popc(peers);
        __syncthreads();
        if (valid) {
            long long pos = next[d] + rank;
            for (int w = 0; w < warp; ++w) pos += wcnt[w][d];
            keys_out[pos] = k;
            vals_out[pos] = v;
        }
        __syncthreads();
        unsigned int tot = 0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) tot += wcnt[w][tid];
        next[tid] += tot;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------- curve
// Segmented running sums: (ok, def, pro) over a stretch of the sorted pixels, and (sok, sdef, spro) = their values just before the last
// run start inside the stretch (relative to the stretch's beginning; meaningful when has != 0).
struct Seg {
    u128 pro, spro;
    u64 ok, def, sok, sdef;
    int has;
};

__device__ __forceinline__ Seg seg_identity() {
    Seg s;
    s.pro = s.spro = 0;
    s.ok = s.def = s.sok = s.sdef = 0;
    s.has = 0;
    return s;
}

__device__ __forceinline__ Seg combine(const Seg& a, const Seg& b) {
    Seg r;
    r.ok = a.ok + b.ok;
    r.def = a.def + b.def;
    r.pro = a.pro + b.pro;
    if (b.has) {
        r.sok = a.ok + b.sok;
        r.sdef = a.def + b.sdef;
        r.spro = a.pro + b.spro;
        r.has = 1;
    } else {
        r.sok = a.sok;
        r.sdef = a.sdef;
        r.spro = a.spro;
        r.has = a.has;
    }
    return r;
}

// one sorted pixel; `start`: the first pixel of its run of equal keys
// (an out-of-range index counts as a defect pixel of weight 0; the first radix pass has counted it for the caller)
__device__ __forceinline__ Seg seg_pixel(int32_t region, const int64_t* __restrict__ sizes, int n_regions, bool start) {
    Seg s = seg_identity();
    if (region < 0) {
        s.ok = 1;
    } else {
        s.def = 1;
        const long long sz = region < n_regions ? sizes[region] : 0;
        s.pro = sz > 0 ? static_cast<u128>(kProOne / static_cast<u64>(sz)) : 0;
    }
    s.has = start;
    return s;
}

// exclusive scan of one Seg per thread over the CTA (fixed Hillis-Steele order); *total = the CTA's aggregate
__device__ Seg block_exclusive_scan(const Seg& v, Seg* sh, Seg* total) {
    const int t = threadIdx.x;
    sh[t] = v;
    __syncthreads();
    for (int d = 1; d < kThreads; d <<= 1) {
        Seg x = sh[t];
        if (t >= d) x = combine(sh[t - d], x);
        __syncthreads();
        sh[t] = x;
        __syncthreads();
    }
    const Seg ex = t ? sh[t - 1] : seg_identity();
    *total = sh[kThreads - 1];
    __syncthreads();
    return ex;
}

// stages a tile's keys (with the key before and after it) and region indices in shared memory
struct ScanStage {
    uint32_t key[kScanTile + 2];    // key[0] = key before the tile, key[1 + j] = pixel j, key[kScanTile + 1] = key after the tile
    int32_t reg[kScanTile];
};

__device__ __forceinline__ void stage_tile(ScanStage& st, const uint32_t* __restrict__ keys, const int32_t* __restrict__ regs,
                                           long long n, long long base) {
    const int tid = threadIdx.x;
    for (int j = tid; j < kScanTile; j += kThreads) {
        const long long i = base + j;
        st.key[1 + j] = i < n ? keys[i] : 0u;
        st.reg[j] = i < n ? regs[i] : -1;
    }
    if (tid == 0) st.key[0] = base > 0 ? keys[base - 1] : 0u;
    if (tid == 1) st.key[kScanTile + 1] = base + kScanTile < n ? keys[base + kScanTile] : 0u;
    __syncthreads();
}

__device__ __forceinline__ Seg thread_aggregate(const ScanStage& st, const int64_t* __restrict__ sizes, int n_regions, long long n,
                                                long long base) {
    Seg acc = seg_identity();
    for (int q = 0; q < kScanItems; ++q) {
        const int j = threadIdx.x * kScanItems + q;
        const long long i = base + j;
        if (i >= n) break;
        acc = combine(acc, seg_pixel(st.reg[j], sizes, n_regions, i == 0 || st.key[j] != st.key[1 + j]));
    }
    return acc;
}

__global__ void __launch_bounds__(kThreads) seg_tile_kernel(const uint32_t* __restrict__ keys, const int32_t* __restrict__ regs,
                                                            const int64_t* __restrict__ sizes, int n_regions, long long n,
                                                            Seg* __restrict__ agg) {
    __shared__ ScanStage st;
    __shared__ Seg sh[kThreads];
    const long long base = static_cast<long long>(blockIdx.x) * kScanTile;
    stage_tile(st, keys, regs, n, base);
    Seg total;
    block_exclusive_scan(thread_aggregate(st, sizes, n_regions, n, base), sh, &total);
    if (threadIdx.x == 0) agg[blockIdx.x] = total;
}

// one CTA: agg[t] <- exclusive prefix of the tile aggregates
__global__ void __launch_bounds__(kThreads) seg_scan_kernel(Seg* __restrict__ agg, int n_tiles) {
    __shared__ Seg sh[kThreads];
    Seg carry = seg_identity();
    for (int b0 = 0; b0 < n_tiles; b0 += kThreads) {
        const int t = b0 + threadIdx.x;
        Seg total;
        const Seg ex = block_exclusive_scan(t < n_tiles ? agg[t] : seg_identity(), sh, &total);
        if (t < n_tiles) agg[t] = combine(carry, ex);
        carry = combine(carry, total);
    }
}

__device__ __forceinline__ double u128_to_double(u128 v) {
    return static_cast<double>(static_cast<u64>(v >> 64)) * 18446744073709551616.0 + static_cast<double>(static_cast<u64>(v));
}

struct CurveParams {
    long long n;
    long long n_ok;        // defect-free pixels (FPR denominator)
    int n_regions;
    double inv_n_ok;
    double inv_pro;        // 1 / (n_regions * 2^63)
    double alpha;
    u64 n_def;             // defect pixels, n - n_ok
};

// F1 of a run end as an exact fraction: F1 = 2 num / den, num = d_k, den = d_k + o_k + N_def (< 2^64: the products below fit 128 bits)
struct F1Cand {
    u64 num, den;
    uint32_t key;          // the run's key
};

__device__ __forceinline__ F1Cand f1_identity() {
    F1Cand c;
    c.num = 0, c.den = 1, c.key = 0xffffffffu;
    return c;
}

// a beats b: a larger fraction, or the same one at a smaller key (an earlier run, a higher score).  A total order on distinct keys,
// and every key ends one run only, so the max does not depend on the order of the reduction.
__device__ __forceinline__ bool f1_better(const F1Cand& a, const F1Cand& b) {
    const u128 l = static_cast<u128>(a.num) * b.den, r = static_cast<u128>(b.num) * a.den;
    return l > r || (l == r && a.key < b.key);
}

// lane 0 gets the warp's sum, added in a fixed order
__device__ __forceinline__ double warp_sum_fixed(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ F1Cand warp_f1_max(F1Cand c) {
    for (int o = 16; o > 0; o >>= 1) {
        F1Cand x;
        x.num = __shfl_xor_sync(0xffffffffu, c.num, o);
        x.den = __shfl_xor_sync(0xffffffffu, c.den, o);
        x.key = __shfl_xor_sync(0xffffffffu, c.key, o);
        if (f1_better(x, c)) c = x;
    }
    return c;
}

__global__ void __launch_bounds__(kThreads) seg_curve_kernel(const uint32_t* __restrict__ keys, const int32_t* __restrict__ regs,
                                                             const int64_t* __restrict__ sizes, const Seg* __restrict__ tile_prefix,
                                                             const CurveParams p, u128* __restrict__ part_num, double* __restrict__ part_area,
                                                             double* __restrict__ part_ap, F1Cand* __restrict__ part_f1) {
    __shared__ ScanStage st;
    __shared__ Seg sh[kThreads];
    __shared__ double red_a[kThreads];
    __shared__ u128 red_n[kThreads];
    __shared__ double warp_ap[kThreads / 32];
    __shared__ F1Cand warp_f1[kThreads / 32];
    const int tid = threadIdx.x;
    const long long base = static_cast<long long>(blockIdx.x) * kScanTile;
    stage_tile(st, keys, regs, p.n, base);
    Seg total;
    const Seg ex = block_exclusive_scan(thread_aggregate(st, sizes, p.n_regions, p.n, base), sh, &total);
    Seg run = combine(tile_prefix[blockIdx.x], ex);
    double area = 0.0, ap = 0.0;
    u128 num = 0;
    F1Cand f1 = f1_identity();
    for (int q = 0; q < kScanItems; ++q) {
        const int j = tid * kScanItems + q;
        const long long i = base + j;
        if (i >= p.n) break;
        run = combine(run, seg_pixel(st.reg[j], sizes, p.n_regions, i == 0 || st.key[j] != st.key[1 + j]));
        if (i + 1 < p.n && st.key[1 + j] == st.key[2 + j]) continue;     // not the last pixel of its run
        const u64 ok_run = run.ok - run.sok, def_run = run.def - run.sdef;
        num += static_cast<u128>(def_run) * static_cast<u128>(2ull * (static_cast<u64>(p.n_ok) - run.ok) + ok_run);
        if (def_run) {                                                  // precision-recall: runs with a defect pixel only
            const u64 seen = run.def + run.ok;
            ap += static_cast<double>(def_run) * (static_cast<double>(run.def) / static_cast<double>(seen));
            F1Cand c;
            c.num = run.def, c.den = seen + p.n_def, c.key = st.key[1 + j];
            if (f1_better(c, f1)) f1 = c;
        }
        const double x0 = static_cast<double>(run.sok) * p.inv_n_ok;
        if (x0 < p.alpha) {
            double x1 = static_cast<double>(run.ok) * p.inv_n_ok;
            const double y0 = u128_to_double(run.spro) * p.inv_pro;
            double y1 = u128_to_double(run.pro) * p.inv_pro;
            if (x1 > p.alpha) {
                y1 = y0 + (y1 - y0) * (p.alpha - x0) / (x1 - x0);
                x1 = p.alpha;
            }
            area += (x1 - x0) * (y0 + y1) * 0.5;
        }
    }
    ap = warp_sum_fixed(ap);
    f1 = warp_f1_max(f1);
    if ((tid & 31) == 0) {
        warp_ap[tid >> 5] = ap;
        warp_f1[tid >> 5] = f1;
    }
    red_a[tid] = area;
    red_n[tid] = num;
    __syncthreads();
    for (int s = kThreads / 2; s > 0; s >>= 1) {
        if (tid < s) {
            red_a[tid] += red_a[tid + s];
            red_n[tid] += red_n[tid + s];
        }
        __syncthreads();
    }
    if (tid == 0) {
        part_area[blockIdx.x] = red_a[0];
        part_num[blockIdx.x] = red_n[0];
        double a = 0.0;
        F1Cand best = f1_identity();
        for (int w = 0; w < kThreads / 32; ++w) {
            a += warp_ap[w];
            if (f1_better(warp_f1[w], best)) best = warp_f1[w];
        }
        part_ap[blockIdx.x] = a;
        part_f1[blockIdx.x] = best;
    }
}

// one CTA: out = {pixel AUROC, AU-PRO@alpha, NaN scores, defect-free pixels seen, bad region indices, pixel AP, F1-max, F1 threshold}
__global__ void __launch_bounds__(kThreads) finish_kernel(const u128* __restrict__ part_num, const double* __restrict__ part_area,
                                                          const double* __restrict__ part_ap, const F1Cand* __restrict__ part_f1,
                                                          int n_tiles, const u64* __restrict__ counters, long long n, long long n_ok,
                                                          double alpha, double* __restrict__ out) {
    __shared__ double red_a[kThreads];
    __shared__ u128 red_n[kThreads];
    __shared__ double red_p[kThreads];
    __shared__ F1Cand red_f[kThreads];
    const int tid = threadIdx.x;
    double a = 0.0, ap = 0.0;
    u128 s = 0;
    F1Cand f1 = f1_identity();
    for (int t = tid; t < n_tiles; t += kThreads) {
        a += part_area[t];
        s += part_num[t];
        ap += part_ap[t];
        if (f1_better(part_f1[t], f1)) f1 = part_f1[t];
    }
    red_a[tid] = a;
    red_n[tid] = s;
    red_p[tid] = ap;
    red_f[tid] = f1;
    __syncthreads();
    for (int k = kThreads / 2; k > 0; k >>= 1) {
        if (tid < k) {
            red_a[tid] += red_a[tid + k];
            red_n[tid] += red_n[tid + k];
            red_p[tid] += red_p[tid + k];
            if (f1_better(red_f[tid + k], red_f[tid])) red_f[tid] = red_f[tid + k];
        }
        __syncthreads();
    }
    if (tid == 0) {
        const double n_def = static_cast<double>(n - n_ok);
        out[0] = u128_to_double(red_n[0]) / (2.0 * static_cast<double>(n_ok) * n_def);
        out[1] = red_a[0] / alpha;
        out[2] = static_cast<double>(counters[0]);
        out[3] = static_cast<double>(counters[1]);
        out[4] = static_cast<double>(counters[2]);
        out[5] = red_p[0] / n_def;
        out[6] = 2.0 * static_cast<double>(red_f[0].num) / static_cast<double>(red_f[0].den);
        out[7] = static_cast<double>(key_score(red_f[0].key));
    }
}

// ---------------------------------------------------------------------------------------------------------- radix select
// The streaming kernels below (select_hist_kernel, threshold_kernel) read the pixels in a grid-stride loop, with 16-byte loads when
// the arrays are 16-byte aligned (kVec) and the < 4 pixels of the tail read by the first CTA.
// Running state of the select, in device memory between the kernels: the rank still to find inside the pixels that match the prefix.
struct SelectState {
    u64 rank;              // 1-based rank inside the current prefix
    u64 nan;               // NaN scores (excluded from the ranking)
    uint32_t prefix;       // ascending key bits fixed so far
    uint32_t empty;        // 1: fewer non-NaN scores than the rank asked for
};
static_assert(sizeof(SelectState) == 3 * sizeof(u64), "the select state lives in the 3 counters of the layout");

// ascending key: order-preserving, so the k-th smallest key is the k-th smallest score
__device__ __forceinline__ uint32_t asc_key(float f) { return ~desc_key(f); }

template <bool kVec>
__global__ void __launch_bounds__(kThreads) select_hist_kernel(const float* __restrict__ scores, long long n, int shift,
                                                               u64* __restrict__ hist, SelectState* __restrict__ st) {
    __shared__ unsigned int h[kThreads / 32][kBins];
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int j = tid; j < (kThreads / 32) * kBins; j += kThreads) (&h[0][0])[j] = 0;
    __syncthreads();
    const uint32_t hi_mask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));   // the digits above this pass
    const uint32_t prefix = st->prefix & hi_mask;
    u64 nan_c = 0;
    auto one = [&](float f) {
        if (f != f) {
            ++nan_c;
            return;
        }
        const uint32_t a = asc_key(f);
        if (((a ^ prefix) & hi_mask) == 0) atomicAdd(&h[warp][(a >> shift) & (kBins - 1)], 1u);
    };
    const long long stride = static_cast<long long>(gridDim.x) * kThreads;
    const long long first = static_cast<long long>(blockIdx.x) * kThreads + tid;
    if (kVec) {
        const long long n4 = n >> 2;
        const float4* s4 = reinterpret_cast<const float4*>(scores);
        for (long long v = first; v < n4; v += stride) {
            const float4 f = s4[v];
            one(f.x), one(f.y), one(f.z), one(f.w);
        }
        if (blockIdx.x == 0 && tid < (n & 3)) one(scores[(n4 << 2) + tid]);
    } else {
        for (long long i = first; i < n; i += stride) one(scores[i]);
    }
    __syncthreads();
    unsigned int c = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) c += h[w][tid];
    if (c) atomicAdd(&hist[tid], static_cast<u64>(c));
    if (shift == 24) {
        nan_c = warp_sum(nan_c);
        if ((tid & 31) == 0 && nan_c) atomicAdd(&st->nan, nan_c);
    }
}

// one CTA: the digit holding the rank (first pass: rank k), the new prefix and the rank left inside it; clears the histogram for the
// next pass.  The last pass writes out = {score, NaN count}.
__global__ void __launch_bounds__(kThreads) select_pick_kernel(int shift, u64 k, u64* __restrict__ hist, SelectState* __restrict__ st,
                                                               double* __restrict__ out) {
    __shared__ u64 s[kBins];
    const int tid = threadIdx.x;
    const u64 c = hist[tid];
    hist[tid] = 0;
    s[tid] = c;
    const bool first = shift == 24;
    const u64 rank = first ? k : st->rank;
    const uint32_t prefix = first ? 0u : st->prefix;
    const bool empty = first ? false : st->empty != 0;
    __syncthreads();
    for (int d = 1; d < kBins; d <<= 1) {                       // inclusive scan of the digit counts
        const u64 x = tid >= d ? s[tid - d] : 0;
        __syncthreads();
        s[tid] += x;
        __syncthreads();
    }
    const u64 total = s[kBins - 1], before = s[tid] - c;
    const bool none = empty || rank > total;                    // only NaNs can leave fewer scores than k <= n
    if (!none && c && before < rank && rank <= s[tid]) {        // exactly one digit
        const uint32_t p = prefix | (static_cast<uint32_t>(tid) << shift);
        st->rank = rank - before;
        st->prefix = p;
        if (shift == 0) out[0] = static_cast<double>(key_score(~p));
    }
    if (tid == 0) {
        if (first) st->empty = none;
        if (shift == 0) {
            if (none) out[0] = __longlong_as_double(0x7ff8000000000000LL);
            out[1] = static_cast<double>(st->nan);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------- metrics at a threshold
struct ThrCounts {
    u128 pro;              // fixed-point PRO weight of the detected defect pixels
    u64 tp, fp, fn, nan, bad;
};

__device__ __forceinline__ u128 warp_sum_u128(u128 v) {
    for (int o = 16; o > 0; o >>= 1) {
        const u64 lo = __shfl_xor_sync(0xffffffffu, static_cast<u64>(v), o);
        const u64 hi = __shfl_xor_sync(0xffffffffu, static_cast<u64>(v >> 64), o);
        v += (static_cast<u128>(hi) << 64) | lo;
    }
    return v;
}

template <bool kVec>
__global__ void __launch_bounds__(kThreads) threshold_kernel(const float* __restrict__ scores, const int32_t* __restrict__ regions,
                                                             const int64_t* __restrict__ sizes, int n_regions, long long n,
                                                             float threshold, ThrCounts* __restrict__ part) {
    __shared__ ThrCounts wsum[kThreads / 32];
    const int tid = threadIdx.x;
    u64 tp = 0, fp = 0, fn = 0, nan_c = 0, bad = 0;
    u128 pro = 0;
    auto one = [&](float f, int32_t r) {
        const bool pred = f >= threshold, def = r >= 0;
        nan_c += f != f;
        bad += r < -1 || r >= n_regions || (def && sizes[r] < 1);
        tp += pred && def;
        fp += pred && !def;
        fn += !pred && def;
        if (pred && def && r < n_regions) {
            const long long sz = sizes[r];
            if (sz > 0) pro += kProOne / static_cast<u64>(sz);
        }
    };
    const long long stride = static_cast<long long>(gridDim.x) * kThreads;
    const long long first = static_cast<long long>(blockIdx.x) * kThreads + tid;
    if (kVec) {
        const long long n4 = n >> 2;
        const float4* s4 = reinterpret_cast<const float4*>(scores);
        const int4* r4 = reinterpret_cast<const int4*>(regions);
        for (long long v = first; v < n4; v += stride) {
            const float4 f = s4[v];
            const int4 r = r4[v];
            one(f.x, r.x), one(f.y, r.y), one(f.z, r.z), one(f.w, r.w);
        }
        if (blockIdx.x == 0 && tid < (n & 3)) one(scores[(n4 << 2) + tid], regions[(n4 << 2) + tid]);
    } else {
        for (long long i = first; i < n; i += stride) one(scores[i], regions[i]);
    }
    tp = warp_sum(tp), fp = warp_sum(fp), fn = warp_sum(fn), nan_c = warp_sum(nan_c), bad = warp_sum(bad);
    pro = warp_sum_u128(pro);
    if ((tid & 31) == 0) {
        ThrCounts& w = wsum[tid >> 5];
        w.pro = pro, w.tp = tp, w.fp = fp, w.fn = fn, w.nan = nan_c, w.bad = bad;
    }
    __syncthreads();
    if (tid == 0) {
        ThrCounts t = wsum[0];
        for (int w = 1; w < kThreads / 32; ++w) {
            t.pro += wsum[w].pro, t.tp += wsum[w].tp, t.fp += wsum[w].fp, t.fn += wsum[w].fn;
            t.nan += wsum[w].nan, t.bad += wsum[w].bad;
        }
        part[blockIdx.x] = t;
    }
}

// one CTA: out = {TP, FP, FN, TN, PRO@threshold, NaN scores, bad region indices}
__global__ void __launch_bounds__(kThreads) threshold_finish_kernel(const ThrCounts* __restrict__ part, int n_parts, long long n,
                                                                    int n_regions, double* __restrict__ out) {
    __shared__ ThrCounts red[kThreads];
    const int tid = threadIdx.x;
    ThrCounts t = {};
    for (int b = tid; b < n_parts; b += kThreads) {
        t.pro += part[b].pro, t.tp += part[b].tp, t.fp += part[b].fp, t.fn += part[b].fn;
        t.nan += part[b].nan, t.bad += part[b].bad;
    }
    red[tid] = t;
    __syncthreads();
    for (int s = kThreads / 2; s > 0; s >>= 1) {
        if (tid < s) {
            ThrCounts& a = red[tid];
            const ThrCounts& b = red[tid + s];
            a.pro += b.pro, a.tp += b.tp, a.fp += b.fp, a.fn += b.fn, a.nan += b.nan, a.bad += b.bad;
        }
        __syncthreads();
    }
    if (tid == 0) {
        const ThrCounts& r = red[0];
        out[0] = static_cast<double>(r.tp);
        out[1] = static_cast<double>(r.fp);
        out[2] = static_cast<double>(r.fn);
        out[3] = static_cast<double>(static_cast<u64>(n) - r.tp - r.fp - r.fn);
        out[4] = n_regions > 0 ? u128_to_double(r.pro) / (static_cast<double>(n_regions) * static_cast<double>(kProOne))
                               : __longlong_as_double(0x7ff8000000000000LL);
        out[5] = static_cast<double>(r.nan);
        out[6] = static_cast<double>(r.bad);
    }
}

// ---------------------------------------------------------------------------------------------------------- workspace
struct Layout {
    size_t keys_a, keys_b, vals_a, vals_b, hist, digit_tot, counters, agg, part_num, part_area, part_ap, part_f1, total;
    int sort_tiles, scan_tiles;
};

inline size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

bool make_layout(long long n, Layout& L) {
    if (n <= 0) return false;
    const long long st = (n + kSortTile - 1) / kSortTile, ct = (n + kScanTile - 1) / kScanTile;
    if (st > 0x7fffffffLL || ct > 0x7fffffffLL) return false;
    L.sort_tiles = static_cast<int>(st);
    L.scan_tiles = static_cast<int>(ct);
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align256(off + bytes); return o; };
    const size_t un = static_cast<size_t>(n);
    L.keys_a = take(un * 4);
    L.keys_b = take(un * 4);
    L.vals_a = take(un * 4);
    L.vals_b = take(un * 4);
    L.hist = take(static_cast<size_t>(kBins) * st * 8);
    L.digit_tot = take(kBins * 8);
    L.counters = take(3 * 8);
    L.agg = take(static_cast<size_t>(ct) * sizeof(Seg));
    L.part_num = take(static_cast<size_t>(ct) * sizeof(u128));
    L.part_area = take(static_cast<size_t>(ct) * sizeof(double));
    L.part_ap = take(static_cast<size_t>(ct) * sizeof(double));
    L.part_f1 = take(static_cast<size_t>(ct) * sizeof(F1Cand));
    L.total = off;
    return true;
}

// CTAs of the streaming kernels: 4 per SM (threshold_kernel's 60 registers allow 4 x 256 threads), never more than the sort tiles
// (the threshold partials live in the histogram area of the layout, 2 KB per sort tile).
int stream_grid(const Layout& L) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        sms = 148;
    return L.sort_tiles < 4 * sms ? L.sort_tiles : 4 * sms;
}

}  // namespace
}  // namespace adsr

extern "C" int64_t adsr_localisation_workspace_bytes(int64_t n) {
    adsr::Layout L;
    return adsr::make_layout(n, L) ? static_cast<int64_t>(L.total) : -1;
}

extern "C" int adsr_localisation_metrics(const float* scores, const int32_t* regions, int64_t n, const int64_t* region_sizes,
                                         int n_regions, int64_t n_ok, double fpr_limit, void* workspace, int64_t workspace_bytes,
                                         double* out, void* stream) {
    using namespace adsr;
    Layout L;
    if (!make_layout(n, L) || n_regions < 1 || n_ok < 1 || n_ok >= n || !(fpr_limit > 0.0 && fpr_limit <= 1.0)) return ADSR_ERR_BAD_SHAPE;
    if (scores == nullptr || regions == nullptr || region_sizes == nullptr || workspace == nullptr || out == nullptr ||
        workspace_bytes < static_cast<int64_t>(L.total))
        return ADSR_ERR_BAD_SHAPE;
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return ADSR_ERR_BAD_ALIGN;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(workspace);
    uint32_t* keys[2] = {reinterpret_cast<uint32_t*>(ws + L.keys_a), reinterpret_cast<uint32_t*>(ws + L.keys_b)};
    int32_t* vals[2] = {reinterpret_cast<int32_t*>(ws + L.vals_a), reinterpret_cast<int32_t*>(ws + L.vals_b)};
    long long* hist = reinterpret_cast<long long*>(ws + L.hist);
    long long* digit_tot = reinterpret_cast<long long*>(ws + L.digit_tot);
    u64* counters = reinterpret_cast<u64*>(ws + L.counters);
    Seg* agg = reinterpret_cast<Seg*>(ws + L.agg);
    u128* part_num = reinterpret_cast<u128*>(ws + L.part_num);
    double* part_area = reinterpret_cast<double*>(ws + L.part_area);
    double* part_ap = reinterpret_cast<double*>(ws + L.part_ap);
    F1Cand* part_f1 = reinterpret_cast<F1Cand*>(ws + L.part_f1);

    if (cudaMemsetAsync(counters, 0, 3 * sizeof(u64), s) != cudaSuccess) return ADSR_ERR_CUDA;
    // pass 0 reads the scores and region indices and writes buffer 1; passes alternate 1 -> 0 -> 1 -> 0: the sorted pairs end in buffer 0
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 8 * pass, src = pass & 1, dst = src ^ 1;
        if (pass == 0)
            radix_hist_kernel<true><<<L.sort_tiles, kThreads, 0, s>>>(nullptr, scores, regions, region_sizes, n_regions, n, shift,
                                                                      L.sort_tiles, hist, counters);
        else
            radix_hist_kernel<false><<<L.sort_tiles, kThreads, 0, s>>>(keys[src], nullptr, nullptr, nullptr, 0, n, shift, L.sort_tiles,
                                                                       hist, nullptr);
        radix_scan_kernel<<<kBins, 1024, 0, s>>>(hist, L.sort_tiles, digit_tot);
        if (pass == 0)
            radix_scatter_kernel<true><<<L.sort_tiles, kThreads, 0, s>>>(nullptr, regions, scores, n, shift, L.sort_tiles, hist, digit_tot,
                                                                         keys[dst], vals[dst]);
        else
            radix_scatter_kernel<false><<<L.sort_tiles, kThreads, 0, s>>>(keys[src], vals[src], nullptr, n, shift, L.sort_tiles, hist,
                                                                          digit_tot, keys[dst], vals[dst]);
    }
    if (cudaGetLastError() != cudaSuccess) return ADSR_ERR_LAUNCH;

    seg_tile_kernel<<<L.scan_tiles, kThreads, 0, s>>>(keys[0], vals[0], region_sizes, n_regions, n, agg);
    seg_scan_kernel<<<1, kThreads, 0, s>>>(agg, L.scan_tiles);
    CurveParams p;
    p.n = n;
    p.n_ok = n_ok;
    p.n_regions = n_regions;
    p.inv_n_ok = 1.0 / static_cast<double>(n_ok);
    p.inv_pro = 1.0 / (static_cast<double>(n_regions) * static_cast<double>(kProOne));
    p.alpha = fpr_limit;
    p.n_def = static_cast<u64>(n - n_ok);
    seg_curve_kernel<<<L.scan_tiles, kThreads, 0, s>>>(keys[0], vals[0], region_sizes, agg, p, part_num, part_area, part_ap, part_f1);
    finish_kernel<<<1, kThreads, 0, s>>>(part_num, part_area, part_ap, part_f1, L.scan_tiles, counters, n, n_ok, fpr_limit, out);
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}

extern "C" int adsr_score_quantile(const float* scores, int64_t n, int64_t k, void* workspace, int64_t workspace_bytes, double* out,
                                   void* stream) {
    using namespace adsr;
    Layout L;
    if (!make_layout(n, L) || k < 1 || k > n) return ADSR_ERR_BAD_SHAPE;
    if (scores == nullptr || workspace == nullptr || out == nullptr || workspace_bytes < static_cast<int64_t>(L.total))
        return ADSR_ERR_BAD_SHAPE;
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return ADSR_ERR_BAD_ALIGN;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(workspace);
    u64* hist = reinterpret_cast<u64*>(ws + L.digit_tot);
    SelectState* st = reinterpret_cast<SelectState*>(ws + L.counters);
    if (cudaMemsetAsync(hist, 0, kBins * sizeof(u64), s) != cudaSuccess || cudaMemsetAsync(st, 0, sizeof(SelectState), s) != cudaSuccess)
        return ADSR_ERR_CUDA;
    const int grid = stream_grid(L);
    const bool vec = (reinterpret_cast<uintptr_t>(scores) & 15) == 0;
    for (int shift = 24; shift >= 0; shift -= 8) {             // most significant digit first
        if (vec)
            select_hist_kernel<true><<<grid, kThreads, 0, s>>>(scores, n, shift, hist, st);
        else
            select_hist_kernel<false><<<grid, kThreads, 0, s>>>(scores, n, shift, hist, st);
        select_pick_kernel<<<1, kThreads, 0, s>>>(shift, static_cast<u64>(k), hist, st, out);
    }
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}

extern "C" int adsr_threshold_metrics(const float* scores, const int32_t* regions, int64_t n, const int64_t* region_sizes,
                                      int n_regions, float threshold, void* workspace, int64_t workspace_bytes, double* out,
                                      void* stream) {
    using namespace adsr;
    Layout L;
    if (!make_layout(n, L) || n_regions < 0 || threshold != threshold) return ADSR_ERR_BAD_SHAPE;
    if (scores == nullptr || regions == nullptr || (n_regions > 0 && region_sizes == nullptr) || workspace == nullptr ||
        out == nullptr || workspace_bytes < static_cast<int64_t>(L.total))
        return ADSR_ERR_BAD_SHAPE;
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return ADSR_ERR_BAD_ALIGN;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    ThrCounts* part = reinterpret_cast<ThrCounts*>(static_cast<char*>(workspace) + L.hist);
    static_assert(sizeof(ThrCounts) <= kBins * sizeof(long long), "one partial per sort tile fits the tile's histogram slice");
    const int grid = stream_grid(L);
    const bool vec = ((reinterpret_cast<uintptr_t>(scores) | reinterpret_cast<uintptr_t>(regions)) & 15) == 0;
    if (vec)
        threshold_kernel<true><<<grid, kThreads, 0, s>>>(scores, regions, region_sizes, n_regions, n, threshold, part);
    else
        threshold_kernel<false><<<grid, kThreads, 0, s>>>(scores, regions, region_sizes, n_regions, n, threshold, part);
    threshold_finish_kernel<<<1, kThreads, 0, s>>>(part, grid, n, n_regions, out);
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}
