// scene_blocks.cu -- whole-scene block tiling, sampling and per-point votes on the device.
//
// The whole-scene evaluation loader of PointNet++ ScanNet segmentation cuts a scan into 1.5 m columns padded by 0.2 m,
// samples `npoints` points of each with replacement and weights them by "inside the column's core"; labelling a whole
// scan covers every padded column with forwards and takes a per-point majority vote.  Both run here without per-block
// host work: oracle/whole_scene_ref.py states the protocol in numpy and is the definition the tests pin.
//
//   pn2_scene_index   bounds (two-pass reduction), grid dims, <= 4 (block, point) pairs per point, stable segment sort
//   pn2_scene_keep    sampled core counts per block, kept-block compaction           -> grid->count = kept blocks
//   pn2_scene_sample  sampled index map, targets, weights and [xyz | feats] rows of the kept blocks
//   pn2_scene_chunks  chunk count per non-empty block, exclusive scan                -> grid->count = chunks
//   pn2_scene_chunk_rows  chunk sizes, index map and rows
//   pn2_scene_votes   integer-atomic votes (exact, order independent), optional first-maximum labels
//
// Membership tests run in fp64 on the widened fp32 values, in the loader's operation order.
#include <cub/cub.cuh>

#include "common.cuh"

namespace pn2 {
namespace {

constexpr double BLOCK = 1.5;  // column edge (m)
constexpr double PAD = 0.2;    // padding of the sampled column
constexpr double CORE = 0.001; // margin of the column's core (the points that are scored)
constexpr double MIN_CORE = 0.01;
constexpr int MAX_BLOCKS = PN2_SCENE_MAX_BLOCKS;
constexpr uint32_t SENTINEL = MAX_BLOCKS;  // key of unused pair slots: sorts after every block
constexpr int SEG_KEYS = MAX_BLOCKS + 1;   // blocks + the sentinel bucket
constexpr int BOUNDS_CTAS = 256;
constexpr int THREADS = 256;

static_assert(sizeof(pn2_scene_grid) == 40, "the Python layer reads the record as 10 words");
static_assert(2 * PAD < BLOCK, "a point must lie in at most two padded blocks per axis");

__device__ __forceinline__ bool grid_ok(const pn2_scene_grid &g) {
    return g.nx > 0 && g.ny > 0 && (long long)g.nx * g.ny <= MAX_BLOCKS;
}

// p in [(cmin + i*BLOCK) - margin, (cmin + (i+1)*BLOCK) + margin], fp64, the loader's order of operations.
// z sets no condition: the loader's z range is [cmin_z, cmin_z + fl32(cmax_z - cmin_z)] and the rounding error of that
// fp32 difference (half an ulp, < 0.001 m for extents below 8 km) is far below both margins, so every point passes.
__device__ __forceinline__ bool in_range(float p, float cmin, int i, double margin) {
    const double c = (double)cmin;
    const double lo = __dsub_rn(__dadd_rn(c, __dmul_rn((double)i, BLOCK)), margin);
    const double hi = __dadd_rn(__dadd_rn(c, __dmul_rn((double)(i + 1), BLOCK)), margin);
    const double v = (double)p;
    return v >= lo && v <= hi;
}

__device__ __forceinline__ bool in_block(const float *xyz, int p, const pn2_scene_grid &g, int block, double margin) {
    const int i = block / g.ny, j = block % g.ny;
    return in_range(xyz[3 * (size_t)p], g.cmin[0], i, margin) && in_range(xyz[3 * (size_t)p + 1], g.cmin[1], j, margin);
}

// splitmix64 finaliser
__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 30;
    x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27;
    x *= 0x94D049BB133111EBull;
    x ^= x >> 31;
    return x;
}

// segment position read by slot s of block b (count points): with-replacement draw of the loader's np.random.choice
__device__ __forceinline__ int sample_pos(uint64_t seed, int b, int s, int count) {
    const uint64_t h = mix64(seed * 0x9E3779B97F4A7C15ull + (((uint64_t)b << 32) | (uint32_t)s));
    return (int)(((h >> 32) * (uint64_t)count) >> 32);
}

__device__ __forceinline__ int cap_dim(double v) {  // ceil(extent / BLOCK); NaN -> 0, huge -> above MAX_BLOCKS
    const double c = ceil(v);
    return c >= 0.0 ? (int)fmin(c, (double)(4 * MAX_BLOCKS)) : 0;
}

__global__ void __launch_bounds__(THREADS) bounds_partial_kernel(int n, const float *__restrict__ xyz, float *__restrict__ partial) {
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int p = blockIdx.x * THREADS + threadIdx.x; p < n; p += gridDim.x * THREADS)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = xyz[3 * (size_t)p + a];
            lo[a] = fminf(lo[a], v);
            hi[a] = fmaxf(hi[a], v);
        }
    using Reduce = cub::BlockReduce<float, THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float l = Reduce(tmp).Reduce(lo[a], cub::Min());
        __syncthreads();
        const float h = Reduce(tmp).Reduce(hi[a], cub::Max());
        __syncthreads();
        if (threadIdx.x == 0) partial[blockIdx.x * 6 + a] = l, partial[blockIdx.x * 6 + 3 + a] = h;
    }
}

// one CTA: min / max over the partials (exact in any order), then the grid dims of step 1
__global__ void __launch_bounds__(THREADS) grid_kernel(int parts, const float *__restrict__ partial, pn2_scene_grid *__restrict__ grid) {
    using Reduce = cub::BlockReduce<float, THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
    __shared__ float res[6];
    for (int q = 0; q < 6; ++q) {
        float v = q < 3 ? INFINITY : -INFINITY;
        for (int t = threadIdx.x; t < parts; t += THREADS) v = q < 3 ? fminf(v, partial[t * 6 + q]) : fmaxf(v, partial[t * 6 + q]);
        const float r = q < 3 ? Reduce(tmp).Reduce(v, cub::Min()) : Reduce(tmp).Reduce(v, cub::Max());
        if (threadIdx.x == 0) res[q] = r;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        pn2_scene_grid g;
        for (int a = 0; a < 3; ++a) g.cmin[a] = res[a], g.cmax[a] = res[3 + a];
        g.nx = cap_dim(__ddiv_rn((double)__fsub_rn(g.cmax[0], g.cmin[0]), BLOCK));
        g.ny = cap_dim(__ddiv_rn((double)__fsub_rn(g.cmax[1], g.cmin[1]), BLOCK));
        g.count = 0;
        g.reserved = 0;
        *grid = g;
    }
}

// Per point its <= 4 (block, point) pairs in ascending block id; unused slots (and every slot when the grid is empty or
// too large) get the sentinel key.  A padded block along one axis is one of floor(d / BLOCK) - 1 .. + 1, d = p - cmin:
// the interval test admits (d - BLOCK - PAD) / BLOCK <= i <= (d + PAD) / BLOCK, which lies within 0.14 of that range.
__global__ void __launch_bounds__(THREADS) pairs_kernel(int n, const float *__restrict__ xyz, const pn2_scene_grid *__restrict__ grid,
                                                         uint32_t *__restrict__ keys, int32_t *__restrict__ payload) {
    const int p = blockIdx.x * THREADS + threadIdx.x;
    if (p >= n) return;
    const pn2_scene_grid g = *grid;
    int i1 = 0, j1 = 0, ni = 0, nj = 0;  // the matching blocks along an axis are consecutive: i1 .. i1 + ni - 1
    if (grid_ok(g)) {
        const float px = xyz[3 * (size_t)p], py = xyz[3 * (size_t)p + 1];
        const int i0 = (int)floor(((double)px - (double)g.cmin[0]) / BLOCK), j0 = (int)floor(((double)py - (double)g.cmin[1]) / BLOCK);
        for (int i = max(i0 - 1, 0); i <= min(i0 + 1, g.nx - 1); ++i)
            if (in_range(px, g.cmin[0], i, PAD)) i1 = ni++ ? i1 : i;
        for (int j = max(j0 - 1, 0); j <= min(j0 + 1, g.ny - 1); ++j)
            if (in_range(py, g.cmin[1], j, PAD)) j1 = nj++ ? j1 : j;
    }
    int q = 0;
    for (int a = 0; a < ni; ++a)
        for (int c = 0; c < nj; ++c, ++q) keys[4 * (size_t)p + q] = (uint32_t)((i1 + a) * g.ny + j1 + c);
    for (; q < 4; ++q) keys[4 * (size_t)p + q] = SENTINEL;
#pragma unroll
    for (int q2 = 0; q2 < 4; ++q2) payload[4 * (size_t)p + q2] = p;
}

// Sampled core slots of every block (CTA-strided over blocks); keep = non-empty and core / npoints >= MIN_CORE in fp64
__global__ void __launch_bounds__(THREADS) keep_kernel(int npoints, uint64_t seed, const float *__restrict__ xyz,
                                                        const pn2_scene_grid *__restrict__ grid, const int32_t *__restrict__ seg_start,
                                                        const int32_t *__restrict__ pos, int32_t *__restrict__ keep) {
    const pn2_scene_grid g = *grid;
    const int nblocks = grid_ok(g) ? g.nx * g.ny : 0;
    using Reduce = cub::BlockReduce<int, THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
    for (int b = blockIdx.x; b < nblocks; b += gridDim.x) {
        const int s0 = seg_start[b], count = seg_start[b + 1] - s0;
        if (count == 0) {
            if (threadIdx.x == 0) keep[b] = 0;
            continue;
        }
        int core = 0;
        for (int s = threadIdx.x; s < npoints; s += THREADS) core += in_block(xyz, pos[s0 + sample_pos(seed, b, s, count)], g, b, CORE);
        const int total = Reduce(tmp).Sum(core);
        if (threadIdx.x == 0) keep[b] = !(__ddiv_rn((double)total, (double)npoints) < MIN_CORE);
        __syncthreads();
    }
}

// One CTA: exclusive scan of per-block values over the grid's blocks.  keep mode: val = keep flag, writes the ids of the
// flagged blocks in ascending order to out[]; chunk mode: val = ceil(count / npoints), writes out[b] = first chunk of b
// (b <= nblocks).  The total goes to grid->count.
template <bool CHUNKS>
__global__ void __launch_bounds__(1024) scan_kernel(int npoints, const int32_t *__restrict__ val, const int32_t *__restrict__ seg_start,
                                                     pn2_scene_grid *__restrict__ grid, int32_t *__restrict__ out) {
    const pn2_scene_grid g = *grid;
    const int nblocks = grid_ok(g) ? g.nx * g.ny : 0;
    using Scan = cub::BlockScan<int, 1024>;
    __shared__ typename Scan::TempStorage tmp;
    int base = 0;
    for (int b0 = 0; b0 < nblocks; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        int v = 0;
        if (b < nblocks) {
            if (CHUNKS) {
                const int count = seg_start[b + 1] - seg_start[b];
                v = (int)(((long long)count + npoints - 1) / npoints);
            } else {
                v = val[b];
            }
        }
        int off, sum;
        Scan(tmp).ExclusiveSum(v, off, sum);
        if (b < nblocks) {
            if (CHUNKS) out[b] = base + off;
            else if (v) out[base + off] = b;
        }
        base += sum;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (CHUNKS) out[nblocks] = base;
        grid->count = base;
    }
}

// slot (k, s) of kept block kept[k]: scene index, target and weight = labelweights[label] * core
__global__ void __launch_bounds__(THREADS) sample_kernel(long long total, int npoints, uint64_t seed, const float *__restrict__ xyz,
                                                          const long long *__restrict__ labels, const float *__restrict__ labelweights,
                                                          int num_classes, const pn2_scene_grid *__restrict__ grid,
                                                          const int32_t *__restrict__ seg_start, const int32_t *__restrict__ pos,
                                                          const int32_t *__restrict__ kept, int32_t *__restrict__ point_index,
                                                          long long *__restrict__ target, float *__restrict__ weights) {
    const long long e = (long long)blockIdx.x * THREADS + threadIdx.x;
    if (e >= total) return;
    const pn2_scene_grid g = *grid;
    const int k = (int)(e / npoints), s = (int)(e - (long long)k * npoints);
    const int b = kept[k];
    const int s0 = seg_start[b], count = seg_start[b + 1] - s0;
    const int p = pos[s0 + sample_pos(seed, b, s, count)];
    point_index[e] = p;
    const bool core = in_block(xyz, p, g, b, CORE);
    float w = core ? 1.f : 0.f;
    if (labels) {
        const long long l = labels[p];
        target[e] = l;
        if (labelweights) w = (l >= 0 && l < num_classes) ? __fmul_rn(labelweights[l], w) : 0.f;
    }
    weights[e] = w;
}

// chunk ch: its block (last b with first[b] <= ch, so empty blocks are skipped) and size
__device__ __forceinline__ int chunk_block(int ch, int nblocks, const int32_t *__restrict__ first) {
    int lo = 0, hi = nblocks;  // first[lo] <= ch < first[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (first[mid] <= ch) lo = mid;
        else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(THREADS) chunk_table_kernel(int n_chunks, const pn2_scene_grid *__restrict__ grid,
                                                               const int32_t *__restrict__ seg_start, const int32_t *__restrict__ first,
                                                               int32_t *__restrict__ block_of, int32_t *__restrict__ sizes) {
    const int ch = blockIdx.x * THREADS + threadIdx.x;
    if (ch >= n_chunks) return;
    const pn2_scene_grid g = *grid;
    const int b = chunk_block(ch, g.nx * g.ny, first);
    const int count = seg_start[b + 1] - seg_start[b];
    const int k = first[b + 1] - first[b], c = ch - first[b];
    block_of[ch] = b;
    sizes[ch] = (count - c + k - 1) / k;
}

// slot s of chunk c of block b reads segment position c + k * (s mod size)
__global__ void __launch_bounds__(THREADS) chunk_index_kernel(long long total, int npoints, const int32_t *__restrict__ seg_start,
                                                               const int32_t *__restrict__ pos, const int32_t *__restrict__ first,
                                                               const int32_t *__restrict__ block_of, const int32_t *__restrict__ sizes,
                                                               int32_t *__restrict__ point_index) {
    const long long e = (long long)blockIdx.x * THREADS + threadIdx.x;
    if (e >= total) return;
    const int ch = (int)(e / npoints), s = (int)(e - (long long)ch * npoints);
    const int b = block_of[ch];
    const int k = first[b + 1] - first[b], c = ch - first[b];
    point_index[e] = pos[seg_start[b] + c + k * (s % sizes[ch])];
}

// out (rows, 3 + C) = [xyz | feats] of point_index, exact copies
__global__ void __launch_bounds__(THREADS) rows_kernel(long long total, int c, const int32_t *__restrict__ point_index,
                                                        const float *__restrict__ xyz, const float *__restrict__ feats,
                                                        float *__restrict__ out) {
    const int w = 3 + c;
    for (long long e = (long long)blockIdx.x * THREADS + threadIdx.x; e < total; e += (long long)gridDim.x * THREADS) {
        const long long r = e / w;
        const int col = (int)(e - r * w);
        const size_t p = (size_t)__ldg(point_index + r);
        out[e] = col < 3 ? __ldg(xyz + 3 * p + col) : __ldg(feats + p * c + (col - 3));
    }
}

__global__ void __launch_bounds__(THREADS) votes_kernel(long long total, int npoints, int n, int num_classes, const int32_t *__restrict__ point_index,
                                                         const int32_t *__restrict__ sizes, const uint8_t *__restrict__ pred,
                                                         int32_t *__restrict__ votes) {
    const long long e = (long long)blockIdx.x * THREADS + threadIdx.x;
    if (e >= total) return;
    const long long ch = e / npoints;
    const int s = (int)(e - ch * npoints);
    const int cls = pred[e], p = point_index[e];
    if (s < sizes[ch] && cls < num_classes && p >= 0 && p < n) atomicAdd(votes + (size_t)p * num_classes + cls, 1);
}

// first maximum, as numpy.argmax
__global__ void __launch_bounds__(THREADS) vote_labels_kernel(int n, int num_classes, const int32_t *__restrict__ votes,
                                                               uint8_t *__restrict__ labels) {
    const int p = blockIdx.x * THREADS + threadIdx.x;
    if (p >= n) return;
    const int32_t *v = votes + (size_t)p * num_classes;
    int best = 0, bv = v[0];
    for (int c = 1; c < num_classes; ++c)
        if (v[c] > bv) best = c, bv = v[c];
    labels[p] = (uint8_t)best;
}

inline unsigned blocks_for(long long total) { return (unsigned)((total + THREADS - 1) / THREADS); }
inline unsigned strided_blocks(long long total) {  // grid-stride kernels: at most 16 CTAs per SM
    const long long cap = 16ll * sm_count(), want = (total + THREADS - 1) / THREADS;
    return (unsigned)(want < cap ? want : cap);
}

}  // namespace
}  // namespace pn2

extern "C" int pn2_scene_index(int n, const float *xyz, pn2_scene_grid *grid, int32_t *seg_start, int32_t *pos, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(n >= 1, "scene_index: need n >= 1 points (n=%d)", n);
    PN2_REQUIRE(4ll * n < (1ll << 31), "scene_index: 4n must be < 2^31 (n=%d)", n);
    PN2_REQUIRE(xyz && grid && seg_start && pos, "scene_index: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    const long long pairs = 4ll * n;
    const int parts = min(BOUNDS_CTAS, ceil_div(n, THREADS));
    const size_t key_bytes = ((size_t)pairs * sizeof(uint32_t) + 255) / 256 * 256;
    const size_t part_bytes = (size_t)BOUNDS_CTAS * 6 * sizeof(float);
    Scratch scratch_mem(s);  // [keys | payloads | partial bounds | segment_sort scratch]
    PN2_CUDA(scratch_mem.alloc(2 * key_bytes + part_bytes + segment_sort_scratch_bytes(pairs, SEG_KEYS)));
    unsigned char *scratch = (unsigned char *)scratch_mem.ptr;
    uint32_t *keys = (uint32_t *)scratch;
    int32_t *payload = (int32_t *)(scratch + key_bytes);
    float *partial = (float *)(scratch + 2 * key_bytes);
    bounds_partial_kernel<<<parts, THREADS, 0, s>>>(n, xyz, partial);
    PN2_LAUNCH_OK("bounds_partial_kernel");
    grid_kernel<<<1, THREADS, 0, s>>>(parts, partial, grid);
    PN2_LAUNCH_OK("grid_kernel");
    pairs_kernel<<<blocks_for(n), THREADS, 0, s>>>(n, xyz, grid, keys, payload);
    PN2_LAUNCH_OK("pairs_kernel");
    return segment_sort(pairs, SEG_KEYS, keys, payload, scratch + 2 * key_bytes + part_bytes, seg_start, pos, s);
}

extern "C" int pn2_scene_keep(int npoints, unsigned long long seed, const float *xyz, pn2_scene_grid *grid, const int32_t *seg_start,
                              const int32_t *pos, int32_t *kept, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(npoints >= 1, "scene_keep: need npoints >= 1 (npoints=%d)", npoints);
    PN2_REQUIRE(xyz && grid && seg_start && pos && kept, "scene_keep: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    Scratch flags(s);
    PN2_CUDA(flags.alloc((size_t)MAX_BLOCKS * sizeof(int32_t)));
    keep_kernel<<<4 * sm_count(), THREADS, 0, s>>>(npoints, (uint64_t)seed, xyz, grid, seg_start, pos, (int32_t *)flags.ptr);
    PN2_LAUNCH_OK("keep_kernel");
    scan_kernel<false><<<1, 1024, 0, s>>>(npoints, (const int32_t *)flags.ptr, seg_start, grid, kept);
    PN2_LAUNCH_OK("scan_kernel<keep>");
    return PN2_OK;
}

static int check_grid_dims(const char *who, int nx, int ny) {
    PN2_REQUIRE(nx >= 1 && ny >= 1, "%s: empty grid nx=%d ny=%d", who, nx, ny);
    PN2_REQUIRE((long long)nx * ny <= pn2::MAX_BLOCKS, "%s: %lld blocks, at most %d are supported", who, (long long)nx * ny, pn2::MAX_BLOCKS);
    return PN2_OK;
}

extern "C" int pn2_scene_sample(int nx, int ny, int nb, int npoints, unsigned long long seed, int c, const float *xyz, const float *feats,
                                const long long *labels, const float *labelweights, int num_classes, const pn2_scene_grid *grid,
                                const int32_t *seg_start, const int32_t *pos, const int32_t *kept, int32_t *point_index, float *points,
                                long long *target, float *weights, void *stream) {
    using namespace pn2;
    if (int st = check_grid_dims("scene_sample", nx, ny)) return st;
    PN2_REQUIRE(npoints >= 1 && c >= 0 && nb >= 0 && nb <= nx * ny, "scene_sample: bad dims nb=%d npoints=%d c=%d", nb, npoints, c);
    PN2_REQUIRE((long long)nb * npoints < (1ll << 31), "scene_sample: nb * npoints must be < 2^31");
    PN2_REQUIRE(!labelweights || (labels && num_classes >= 1), "scene_sample: labelweights need labels and num_classes >= 1");
    if (nb == 0) return PN2_OK;
    PN2_REQUIRE(xyz && (c == 0 || feats) && grid && seg_start && pos && kept && point_index && points && weights && (!labels || target),
                "scene_sample: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    const long long slots = (long long)nb * npoints, elems = slots * (3 + c);
    sample_kernel<<<blocks_for(slots), THREADS, 0, s>>>(slots, npoints, (uint64_t)seed, xyz, labels, labelweights, num_classes, grid,
                                                        seg_start, pos, kept, point_index, target, weights);
    PN2_LAUNCH_OK("sample_kernel");
    rows_kernel<<<strided_blocks(elems), THREADS, 0, s>>>(elems, c, point_index, xyz, feats, points);
    PN2_LAUNCH_OK("rows_kernel");
    return PN2_OK;
}

extern "C" int pn2_scene_chunks(int npoints, pn2_scene_grid *grid, const int32_t *seg_start, int32_t *first, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(npoints >= 1, "scene_chunks: need npoints >= 1 (npoints=%d)", npoints);
    PN2_REQUIRE(grid && seg_start && first, "scene_chunks: null pointer");
    scan_kernel<true><<<1, 1024, 0, (cudaStream_t)stream>>>(npoints, nullptr, seg_start, grid, first);
    PN2_LAUNCH_OK("scan_kernel<chunks>");
    return PN2_OK;
}

extern "C" int pn2_scene_chunk_rows(int nx, int ny, int n_chunks, int npoints, int c, const float *xyz, const float *feats,
                                    const pn2_scene_grid *grid, const int32_t *seg_start, const int32_t *pos, const int32_t *first,
                                    int32_t *point_index, int32_t *sizes, float *points, void *stream) {
    using namespace pn2;
    if (int st = check_grid_dims("scene_chunk_rows", nx, ny)) return st;
    PN2_REQUIRE(npoints >= 1 && c >= 0 && n_chunks >= 0, "scene_chunk_rows: bad dims n_chunks=%d npoints=%d c=%d", n_chunks, npoints, c);
    PN2_REQUIRE((long long)n_chunks * npoints < (1ll << 31), "scene_chunk_rows: n_chunks * npoints must be < 2^31");
    if (n_chunks == 0) return PN2_OK;
    PN2_REQUIRE(xyz && (c == 0 || feats) && grid && seg_start && pos && first && point_index && sizes && points,
                "scene_chunk_rows: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    Scratch block_of(s);
    PN2_CUDA(block_of.alloc((size_t)n_chunks * sizeof(int32_t)));
    chunk_table_kernel<<<blocks_for(n_chunks), THREADS, 0, s>>>(n_chunks, grid, seg_start, first, (int32_t *)block_of.ptr, sizes);
    PN2_LAUNCH_OK("chunk_table_kernel");
    const long long slots = (long long)n_chunks * npoints, elems = slots * (3 + c);
    chunk_index_kernel<<<blocks_for(slots), THREADS, 0, s>>>(slots, npoints, seg_start, pos, first, (const int32_t *)block_of.ptr, sizes,
                                                             point_index);
    PN2_LAUNCH_OK("chunk_index_kernel");
    rows_kernel<<<strided_blocks(elems), THREADS, 0, s>>>(elems, c, point_index, xyz, feats, points);
    PN2_LAUNCH_OK("rows_kernel");
    return PN2_OK;
}

extern "C" int pn2_scene_votes(int n_chunks, int npoints, const int32_t *point_index, const int32_t *sizes, const uint8_t *pred, int n,
                               int num_classes, int32_t *votes, uint8_t *labels, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(n_chunks >= 0 && npoints >= 1 && n >= 1 && num_classes >= 1 && num_classes <= 256,
                "scene_votes: bad dims n_chunks=%d npoints=%d n=%d num_classes=%d", n_chunks, npoints, n, num_classes);
    PN2_REQUIRE((long long)n * num_classes < (1ll << 31) && (long long)n_chunks * npoints < (1ll << 31), "scene_votes: more than 2^31 entries");
    PN2_REQUIRE(votes && (n_chunks == 0 || (point_index && sizes && pred)), "scene_votes: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    PN2_CUDA(cudaMemsetAsync(votes, 0, (size_t)n * num_classes * sizeof(int32_t), s));
    const long long slots = (long long)n_chunks * npoints;
    if (slots) {
        votes_kernel<<<blocks_for(slots), THREADS, 0, s>>>(slots, npoints, n, num_classes, point_index, sizes, pred, votes);
        PN2_LAUNCH_OK("votes_kernel");
    }
    if (labels) {
        vote_labels_kernel<<<blocks_for(n), THREADS, 0, s>>>(n, num_classes, votes, labels);
        PN2_LAUNCH_OK("vote_labels_kernel");
    }
    return PN2_OK;
}
