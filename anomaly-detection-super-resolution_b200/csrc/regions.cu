// Defect regions: the 8-connected components of a thresholded anomaly map (or of a mask), a minimum-area filter, and per-region
// statistics, exact and deterministic.
//
// Labelling (adsr_label_regions) is a block-based union-find in the style of Playne & Hawick (IEEE TPDS 2018).  Every foreground pixel
// holds a parent index inside its image (linear index y W + x), background holds -1, and parent[i] <= i always, so a tree's root is the
// smallest index of its component whatever order the unions ran in: the result is canonical.
//   local_label_kernel   one CTA per 32 x 32 tile: union-find over the tile in shared memory, roots written as image indices;
//   border_kernel        the top row, left and right columns of every tile unite with their W / NW / N / NE neighbours in other tiles
//                        (global atomicMin unions);
//   compress_kernel      every foreground pixel points straight at its root, and the root's area is counted (warp-aggregated atomics);
//   keep_count_kernel    per 1024-pixel chunk of an image: roots with area >= min_area;
//   keep_scan_kernel     per image: exclusive scan of the chunk counts in raster order, the image's region count;
//   keep_assign_kernel   each kept root gets label chunk offset + rank + 1 (written over its area), a dropped or non-root entry 0;
//   relabel_kernel       every pixel takes its root's label.
// A union retry strictly lowers the larger of the two roots and a find step strictly lowers the index, so both loops end; they still
// carry a cap (the pixel count of the tile / image) that adds to an error counter at the start of the workspace instead of spinning.
//
// Statistics (adsr_region_stats) are one pass over the labels with integer atomics only: area, min / max of y and x, sums of y and x,
// the peak as the 64-bit max of (order-preserving fp32 key << 32 | ~index) -- the highest score wins, a tie goes to the first raster
// pixel -- the ground-truth pixels of each region and a hit flag per ground-truth region.  A warp whose foreground pixels all share one
// region reduces them in registers and issues one atomic per field.
#include "adsr_kernels.h"

namespace adsr {
namespace {

typedef unsigned long long u64;
constexpr int kTile = 32;              // local labelling tile: 32 x 32 pixels, one thread each
constexpr int kChunk = 1024;           // pixels per CTA of the per-pixel passes: one raster range of one image
constexpr int kFields = 9;             // area, y min, x min, y max, x max, sum y, sum x, peak key, ground-truth pixels
constexpr unsigned kFull = 0xffffffffu;

// ---------------------------------------------------------------------------------------------------------- union-find
__device__ __forceinline__ int find_shared(volatile int* s, int x, unsigned int* err) {
    for (int it = 0; it < kTile * kTile; ++it) {
        const int q = s[x];
        if (q == x) return x;
        x = q;
    }
    atomicAdd(err, 1u);
    return x;
}

__device__ __forceinline__ void unite_shared(volatile int* s, int a, int b, unsigned int* err) {
    for (int it = 0; it < kTile * kTile; ++it) {
        a = find_shared(s, a, err);
        b = find_shared(s, b, err);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(const_cast<int*>(s + b), a);   // link the larger root under the smaller one
        if (old == b) return;
        b = old;                                                   // b was linked meanwhile: unite a with its new parent
    }
    atomicAdd(err, 1u);
}

__device__ __forceinline__ int find_global(const int32_t* p, int x, int cap, unsigned int* err) {
    for (int it = 0; it < cap; ++it) {
        const int q = __ldcg(p + x);
        if (q == x) return x;
        x = q;
    }
    atomicAdd(err, 1u);
    return x;
}

__device__ __forceinline__ void unite_global(int32_t* p, int a, int b, int cap, unsigned int* err) {
    for (int it = 0; it < cap; ++it) {
        a = find_global(p, a, cap, err);
        b = find_global(p, b, cap, err);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(p + b, a);
        if (old == b) return;
        b = old;
    }
    atomicAdd(err, 1u);
}

// ---------------------------------------------------------------------------------------------------------- labelling
__global__ void __launch_bounds__(kTile * kTile) local_label_kernel(const float* __restrict__ scores, float thr,
                                                                    const uint8_t* __restrict__ mask, int H, int W, int tiles_x,
                                                                    int tiles_per_img, int32_t* __restrict__ parent,
                                                                    unsigned int* __restrict__ err) {
    __shared__ int s[kTile * kTile];
    const int b = blockIdx.x / tiles_per_img, t = blockIdx.x - b * tiles_per_img;
    const int ty0 = (t / tiles_x) * kTile, tx0 = (t % tiles_x) * kTile;
    const int lx = threadIdx.x, ly = threadIdx.y, lid = ly * kTile + lx;
    const int y = ty0 + ly, x = tx0 + lx;
    const bool inside = y < H && x < W;
    const long long g = static_cast<long long>(b) * H * W + static_cast<long long>(y) * W + x;
    bool fg = false;
    if (inside) fg = scores != nullptr ? scores[g] >= thr : mask[g] != 0;   // a NaN score is never foreground
    s[lid] = fg ? lid : -1;
    __syncthreads();
    volatile int* vs = s;
    if (fg) {                                                     // W, NW, N, NE inside the tile (a foreground entry stays >= 0)
        if (lx > 0 && vs[lid - 1] >= 0) unite_shared(vs, lid, lid - 1, err);
        if (ly > 0) {
            if (lx > 0 && vs[lid - kTile - 1] >= 0) unite_shared(vs, lid, lid - kTile - 1, err);
            if (vs[lid - kTile] >= 0) unite_shared(vs, lid, lid - kTile, err);
            if (lx < kTile - 1 && vs[lid - kTile + 1] >= 0) unite_shared(vs, lid, lid - kTile + 1, err);
        }
    }
    __syncthreads();
    if (inside) {
        int out = -1;
        if (fg) {                                                  // tile raster order is image raster order: the root stays the minimum
            const int r = find_shared(vs, lid, err);
            out = (ty0 + r / kTile) * W + tx0 + r % kTile;
        }
        parent[g] = out;
    }
}

// threads 0..31: the tile's top row; 32..62: its left column, rows 1..31; 64..94: its right column, rows 1..31
__global__ void __launch_bounds__(96) border_kernel(int H, int W, int tiles_x, int tiles_per_img, int32_t* __restrict__ parent,
                                                    unsigned int* __restrict__ err) {
    const int b = blockIdx.x / tiles_per_img, t = blockIdx.x - b * tiles_per_img;
    const int ty0 = (t / tiles_x) * kTile, tx0 = (t % tiles_x) * kTile;
    const int k = threadIdx.x;
    int ly, lx;
    if (k < kTile) ly = 0, lx = k;
    else if (k < 2 * kTile - 1) ly = k - (kTile - 1), lx = 0;
    else if (k >= 2 * kTile && k < 3 * kTile - 1) ly = k - (2 * kTile - 1), lx = kTile - 1;
    else return;
    const int y = ty0 + ly, x = tx0 + lx;
    if (y >= H || x >= W) return;
    const int hw = H * W;
    int32_t* p = parent + static_cast<long long>(b) * hw;
    const int i = y * W + x;
    if (__ldcg(p + i) < 0) return;
    for (int d = 0; d < 4; ++d) {                                  // W, NW, N, NE
        const int dy = d == 0 ? 0 : -1, dx = d == 0 ? -1 : d - 2;
        if (ly + dy >= 0 && lx + dx >= 0 && lx + dx < kTile) continue;   // same tile: already united
        const int gy = y + dy, gx = x + dx;
        if (gy < 0 || gx < 0 || gx >= W) continue;
        const int j = gy * W + gx;
        if (__ldcg(p + j) >= 0) unite_global(p, i, j, hw, err);
    }
}

__global__ void __launch_bounds__(kChunk) compress_kernel(int hw, int chunks, int32_t* __restrict__ parent, int32_t* __restrict__ area,
                                                          unsigned int* __restrict__ err) {
    const int b = blockIdx.x / chunks, c = blockIdx.x - b * chunks;
    const int local = c * kChunk + threadIdx.x;
    const long long base = static_cast<long long>(b) * hw;
    int32_t* p = parent + base;
    int root = -1;
    if (local < hw && __ldcg(p + local) >= 0) {
        root = find_global(p, local, hw, err);
        p[local] = root;
    }
    const unsigned m = __ballot_sync(kFull, root >= 0);
    if (m == 0) return;
    const int lead = __ffs(m) - 1;
    const int r0 = __shfl_sync(kFull, root, lead);
    if (__all_sync(kFull, root < 0 || root == r0)) {
        if ((threadIdx.x & 31) == lead) atomicAdd(area + base + r0, __popc(m));
    } else if (root >= 0) {
        atomicAdd(area + base + root, 1);
    }
}

// exclusive rank of this thread's flag among the CTA's flags in thread order; *total = the CTA's count.  sh: 33 ints.
__device__ __forceinline__ int cta_rank(bool f, int* sh, int* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const unsigned bal = __ballot_sync(kFull, f);
    if (lane == 0) sh[w] = __popc(bal);
    __syncthreads();
    if (w == 0) {
        const int v = lane < nw ? sh[lane] : 0;
        int incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += n;
        }
        if (lane < nw) sh[lane] = incl - v;
        if (lane == 31) sh[32] = incl;
    }
    __syncthreads();
    *total = sh[32];
    return sh[w] + __popc(bal & ((1u << lane) - 1u));
}

__device__ __forceinline__ bool kept_root(const int32_t* p, const int32_t* a, int local, int hw, int min_area) {
    return local < hw && p[local] == local && a[local] >= min_area;
}

__global__ void __launch_bounds__(kChunk) keep_count_kernel(int hw, int chunks, int min_area, const int32_t* __restrict__ parent,
                                                            const int32_t* __restrict__ area, int32_t* __restrict__ chunk_cnt) {
    __shared__ int sh[33];
    const int b = blockIdx.x / chunks, c = blockIdx.x - b * chunks;
    const long long base = static_cast<long long>(b) * hw;
    int total;
    cta_rank(kept_root(parent + base, area + base, c * kChunk + threadIdx.x, hw, min_area), sh, &total);
    if (threadIdx.x == 0) chunk_cnt[blockIdx.x] = total;
}

// one CTA per image: exclusive scan of its chunk counts -> chunk offsets, and the image's region count
__global__ void __launch_bounds__(kChunk) keep_scan_kernel(int chunks, const int32_t* __restrict__ chunk_cnt, int32_t* __restrict__ chunk_off,
                                                           int32_t* __restrict__ counts) {
    __shared__ int sh[33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long base = static_cast<long long>(blockIdx.x) * chunks;
    int carry = 0;
    for (int c0 = 0; c0 < chunks; c0 += kChunk) {
        const int c = c0 + threadIdx.x;
        const int v = c < chunks ? chunk_cnt[base + c] : 0;
        int incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += n;
        }
        if (lane == 31) sh[w] = incl;
        __syncthreads();
        if (w == 0) {
            const int s = sh[lane];
            int si = s;
            for (int o = 1; o < 32; o <<= 1) {
                const int n = __shfl_up_sync(kFull, si, o);
                if (lane >= o) si += n;
            }
            sh[lane] = si - s;
            if (lane == 31) sh[32] = si;
        }
        __syncthreads();
        if (c < chunks) chunk_off[base + c] = carry + sh[w] + incl - v;
        carry += sh[32];
        __syncthreads();                                          // sh is rewritten by the next round
    }
    if (threadIdx.x == 0) counts[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(kChunk) keep_assign_kernel(int hw, int chunks, int min_area, const int32_t* __restrict__ parent,
                                                             int32_t* __restrict__ area, const int32_t* __restrict__ chunk_off) {
    __shared__ int sh[33];
    const int b = blockIdx.x / chunks, c = blockIdx.x - b * chunks;
    const long long base = static_cast<long long>(b) * hw;
    const int local = c * kChunk + threadIdx.x;
    const bool kept = kept_root(parent + base, area + base, local, hw, min_area);
    int total;
    const int rank = cta_rank(kept, sh, &total);
    if (local < hw) area[base + local] = kept ? chunk_off[blockIdx.x] + rank + 1 : 0;   // each thread rewrites only its own entry
}

__global__ void __launch_bounds__(kChunk) relabel_kernel(int hw, int chunks, const int32_t* __restrict__ parent,
                                                         const int32_t* __restrict__ root_label, int32_t* __restrict__ labels) {
    const int b = blockIdx.x / chunks, c = blockIdx.x - b * chunks;
    const long long base = static_cast<long long>(b) * hw;
    const int local = c * kChunk + threadIdx.x;
    if (local >= hw) return;
    const int q = parent[base + local];
    labels[base + local] = q < 0 ? 0 : root_label[base + q];
}

// ---------------------------------------------------------------------------------------------------------- statistics
__device__ __forceinline__ u64 warp_sum64(u64 v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

__device__ __forceinline__ u64 warp_max64(u64 v) {
    for (int o = 16; o > 0; o >>= 1) {
        const u64 n = __shfl_xor_sync(kFull, v, o);
        v = n > v ? n : v;
    }
    return v;
}

// ascending order-preserving key of an fp32 score, -0.0 ranked as +0.0
__device__ __forceinline__ uint32_t asc_key(float f) {
    const uint32_t u = __float_as_uint(f == 0.0f ? 0.0f : f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void stats_init_kernel(u64* __restrict__ table, long long n_rows, int32_t* __restrict__ hit, long long n_gt) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_rows * kFields; i += stride) {
        const int f = static_cast<int>(i % kFields);
        table[i] = (f == 1 || f == 2) ? ~0ull : 0ull;
    }
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_gt; i += stride) hit[i] = 0;
}

__global__ void __launch_bounds__(kChunk) stats_kernel(const int32_t* __restrict__ labels, const float* __restrict__ scores,
                                                       const int32_t* __restrict__ gt, int W, int hw, int chunks,
                                                       const long long* __restrict__ row_off, const long long* __restrict__ gt_off,
                                                       u64* __restrict__ table, int32_t* __restrict__ hit, unsigned int* __restrict__ err) {
    const int b = blockIdx.x / chunks, c = blockIdx.x - b * chunks;
    const long long base = static_cast<long long>(b) * hw;
    const int local = c * kChunk + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int l = 0, g = 0;
    if (local < hw) {
        l = labels[base + local];
        if (gt != nullptr) g = gt[base + local];
    }
    long long row = -1;
    if (l > 0) {
        row = row_off[b] + l - 1;
        if (row >= row_off[b + 1]) row = -1;
    }
    bool bad = l < 0 || (l > 0 && row < 0) || g < 0;
    const bool in = row >= 0, on_gt = g > 0;
    if (in && on_gt) {
        const long long gr = gt_off[b] + g - 1;
        if (gr < gt_off[b + 1]) hit[gr] = 1;
        else bad = true;
    }
    if (bad) atomicAdd(err, 1u);
    const unsigned y = local < hw ? static_cast<unsigned>(local / W) : 0u, x = local < hw ? static_cast<unsigned>(local % W) : 0u;
    u64 key = 0;
    if (in && scores != nullptr) key = (static_cast<u64>(asc_key(scores[base + local])) << 32) | static_cast<uint32_t>(~local);
    const unsigned m = __ballot_sync(kFull, in);
    if (m == 0) return;
    const int lead = __ffs(m) - 1;
    const long long row0 = __shfl_sync(kFull, row, lead);
    if (__all_sync(kFull, !in || row == row0)) {                  // one region in this warp: reduce in registers
        const unsigned n_gt_px = __popc(__ballot_sync(kFull, in && on_gt));
        const unsigned ymin = __reduce_min_sync(kFull, in ? y : 0xffffffffu), xmin = __reduce_min_sync(kFull, in ? x : 0xffffffffu);
        const unsigned ymax = __reduce_max_sync(kFull, in ? y : 0u), xmax = __reduce_max_sync(kFull, in ? x : 0u);
        const u64 sy = warp_sum64(in ? y : 0u), sx = warp_sum64(in ? x : 0u), pk = warp_max64(key);
        if (lane == lead) {
            u64* r = table + row0 * kFields;
            atomicAdd(r + 0, static_cast<u64>(__popc(m)));
            atomicMin(r + 1, static_cast<u64>(ymin));
            atomicMin(r + 2, static_cast<u64>(xmin));
            atomicMax(r + 3, static_cast<u64>(ymax));
            atomicMax(r + 4, static_cast<u64>(xmax));
            atomicAdd(r + 5, sy);
            atomicAdd(r + 6, sx);
            if (scores != nullptr) atomicMax(r + 7, pk);
            if (n_gt_px) atomicAdd(r + 8, static_cast<u64>(n_gt_px));
        }
    } else if (in) {
        u64* r = table + row * kFields;
        atomicAdd(r + 0, 1ull);
        atomicMin(r + 1, static_cast<u64>(y));
        atomicMin(r + 2, static_cast<u64>(x));
        atomicMax(r + 3, static_cast<u64>(y));
        atomicMax(r + 4, static_cast<u64>(x));
        atomicAdd(r + 5, static_cast<u64>(y));
        atomicAdd(r + 6, static_cast<u64>(x));
        if (scores != nullptr) atomicMax(r + 7, key);
        if (on_gt) atomicAdd(r + 8, 1ull);
    }
}

// ---------------------------------------------------------------------------------------------------------- workspace
struct RegionLayout {
    size_t err, parent, area, chunk_cnt, chunk_off, total;
    int hw, tiles_x, tiles_per_img, chunks;
};

inline size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

bool make_region_layout(int B, int H, int W, RegionLayout& L) {
    if (B < 1 || H < 1 || W < 1) return false;
    const long long hw = static_cast<long long>(H) * W;
    if (hw >= (1LL << 31)) return false;
    const long long tx = (W + kTile - 1) / kTile, ty = (H + kTile - 1) / kTile, ch = (hw + kChunk - 1) / kChunk;
    if (B * tx * ty >= (1LL << 31) || B * ch >= (1LL << 31)) return false;   // 1-D grids
    L.hw = static_cast<int>(hw);
    L.tiles_x = static_cast<int>(tx);
    L.tiles_per_img = static_cast<int>(tx * ty);
    L.chunks = static_cast<int>(ch);
    const size_t n = static_cast<size_t>(B) * hw;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align256(off + bytes); return o; };
    L.err = take(sizeof(unsigned int));
    L.parent = take(n * 4);
    L.area = take(n * 4);
    L.chunk_cnt = take(static_cast<size_t>(B) * ch * 4);
    L.chunk_off = take(static_cast<size_t>(B) * ch * 4);
    L.total = off;
    return true;
}

}  // namespace
}  // namespace adsr

extern "C" int64_t adsr_regions_workspace_bytes(int B, int H, int W) {
    adsr::RegionLayout L;
    return adsr::make_region_layout(B, H, W, L) ? static_cast<int64_t>(L.total) : -1;
}

extern "C" int adsr_label_regions(const float* scores, float threshold, const uint8_t* mask, int B, int H, int W, int min_area,
                                  int32_t* labels, int32_t* counts, void* workspace, int64_t workspace_bytes, void* stream) {
    using namespace adsr;
    RegionLayout L;
    if (!make_region_layout(B, H, W, L) || min_area < 1 || (scores == nullptr) == (mask == nullptr) ||
        (scores != nullptr && threshold != threshold))
        return ADSR_ERR_BAD_SHAPE;
    if (labels == nullptr || counts == nullptr || workspace == nullptr || workspace_bytes < static_cast<int64_t>(L.total))
        return ADSR_ERR_BAD_SHAPE;
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return ADSR_ERR_BAD_ALIGN;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(workspace);
    unsigned int* err = reinterpret_cast<unsigned int*>(ws + L.err);
    int32_t* parent = reinterpret_cast<int32_t*>(ws + L.parent);
    int32_t* area = reinterpret_cast<int32_t*>(ws + L.area);
    int32_t* chunk_cnt = reinterpret_cast<int32_t*>(ws + L.chunk_cnt);
    int32_t* chunk_off = reinterpret_cast<int32_t*>(ws + L.chunk_off);
    if (cudaMemsetAsync(err, 0, sizeof(unsigned int), s) != cudaSuccess ||
        cudaMemsetAsync(area, 0, static_cast<size_t>(B) * L.hw * 4, s) != cudaSuccess)
        return ADSR_ERR_CUDA;
    const int tiles = B * L.tiles_per_img, chunks = B * L.chunks;
    local_label_kernel<<<tiles, dim3(kTile, kTile), 0, s>>>(scores, threshold, mask, H, W, L.tiles_x, L.tiles_per_img, parent, err);
    border_kernel<<<tiles, 96, 0, s>>>(H, W, L.tiles_x, L.tiles_per_img, parent, err);
    compress_kernel<<<chunks, kChunk, 0, s>>>(L.hw, L.chunks, parent, area, err);
    keep_count_kernel<<<chunks, kChunk, 0, s>>>(L.hw, L.chunks, min_area, parent, area, chunk_cnt);
    keep_scan_kernel<<<B, kChunk, 0, s>>>(L.chunks, chunk_cnt, chunk_off, counts);
    keep_assign_kernel<<<chunks, kChunk, 0, s>>>(L.hw, L.chunks, min_area, parent, area, chunk_off);
    relabel_kernel<<<chunks, kChunk, 0, s>>>(L.hw, L.chunks, parent, area, labels);
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}

extern "C" int adsr_region_stats(const int32_t* labels, const float* scores, const int32_t* gt_labels, int B, int H, int W,
                                 const int64_t* row_offsets, int64_t n_rows, const int64_t* gt_offsets, int64_t n_gt, int64_t* table,
                                 int32_t* gt_hit, void* workspace, int64_t workspace_bytes, void* stream) {
    using namespace adsr;
    RegionLayout L;
    if (!make_region_layout(B, H, W, L) || n_rows < 0 || n_gt < 0) return ADSR_ERR_BAD_SHAPE;
    if (labels == nullptr || row_offsets == nullptr || (n_rows > 0 && table == nullptr) || workspace == nullptr ||
        workspace_bytes < static_cast<int64_t>(L.total) || (gt_labels != nullptr && (gt_offsets == nullptr || (n_gt > 0 && gt_hit == nullptr))))
        return ADSR_ERR_BAD_SHAPE;
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return ADSR_ERR_BAD_ALIGN;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    unsigned int* err = reinterpret_cast<unsigned int*>(static_cast<char*>(workspace) + L.err);
    if (cudaMemsetAsync(err, 0, sizeof(unsigned int), s) != cudaSuccess) return ADSR_ERR_CUDA;
    const long long init_items = n_rows * kFields > n_gt ? n_rows * kFields : n_gt;
    const long long blocks = (init_items + 255) / 256;
    stats_init_kernel<<<static_cast<int>(blocks < 1 ? 1 : blocks < 4096 ? blocks : 4096), 256, 0, s>>>(
        reinterpret_cast<u64*>(table), n_rows, gt_labels != nullptr ? gt_hit : nullptr, gt_labels != nullptr ? n_gt : 0);
    stats_kernel<<<B * L.chunks, kChunk, 0, s>>>(labels, scores, gt_labels, W, L.hw, L.chunks, reinterpret_cast<const long long*>(row_offsets),
                                                 reinterpret_cast<const long long*>(gt_offsets), reinterpret_cast<u64*>(table), gt_hit, err);
    return cudaGetLastError() == cudaSuccess ? ADSR_OK : ADSR_ERR_LAUNCH;
}
