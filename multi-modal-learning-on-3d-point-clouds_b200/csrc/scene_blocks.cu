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
// The training loader's crops (oracle/scene_crops_ref.py) draw up to ten random 1.5 m columns per crop from a bank of
// scenes resident on the device, with no host read, so a batch can be graph-captured:
//   pn2_scene_bank_bounds  per-scene min / max, once per bank
//   pn2_scene_crops   try 0 of every crop, then tries 1-9 where it failed (counts and a voxel bitmap per try, integer
//                     atomics), the taken column compacted by a stable block scan, slots, rows
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

// out (rows, 3 + C) = [xyz | feats] of point_index, exact copies; NEG_ZERO: a row of index -1 is zeros
template <bool NEG_ZERO>
__global__ void __launch_bounds__(THREADS) rows_kernel(long long total, int c, const int32_t *__restrict__ point_index,
                                                        const float *__restrict__ xyz, const float *__restrict__ feats,
                                                        float *__restrict__ out) {
    const int w = 3 + c;
    for (long long e = (long long)blockIdx.x * THREADS + threadIdx.x; e < total; e += (long long)gridDim.x * THREADS) {
        const long long r = e / w;
        const int col = (int)(e - r * w);
        const int32_t i = __ldg(point_index + r);
        if (NEG_ZERO && i < 0) {
            out[e] = 0.f;
            continue;
        }
        const size_t p = (size_t)i;
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

// ---- training crops: the loader's random 1.5 m columns (pn2_scene_bank_bounds, pn2_scene_crops) ----
constexpr double HALF_XY = 0.75;   // half the column edge (m); z spans the scene
constexpr double CROP_PAD = 0.2;   // margin of the points taken into the crop
constexpr double CROP_CORE = 0.01; // margin of the scored points, the ones whose voxels count
constexpr int CROP_TRIES = 10;
constexpr unsigned CENTRE_SLOT = 0x80000000u;          // try t draws its centre with counter 2^31 + t
constexpr int VOX_KEYS = 32 * 31 * 62 + 32 * 62 + 62 + 1; // keys vx*31*62 + vy*62 + vz, vx, vy in 0..32, vz in 0..62
constexpr int VOX_WORDS = (VOX_KEYS + 31) / 32;
constexpr int TRY_HEAD = 8;       // try record: [labelled, NaN key seen, padded, valid, ...] then the occupancy bitmap
constexpr int TRY_STRIDE = 2048;  // words per (crop, try) record
constexpr int CROP_CHUNK = 8192;  // scene points per work item of a try or of the compaction
constexpr int CROP_ITEMS = CROP_CHUNK / THREADS;
constexpr int R_LAB = 0, R_NAN = 1, R_PAD = 2, R_VALID = 3;

static_assert(VOX_KEYS == 63551 && TRY_HEAD + VOX_WORDS <= TRY_STRIDE, "occupancy bitmap layout");
static_assert(CROP_ITEMS == 32, "the compaction keeps a thread's membership flags in one 32-bit mask");

__device__ __forceinline__ int centre_pos(uint64_t h, int b, int t, int count) {
    return sample_pos(h, b, (int)(CENTRE_SLOT + (unsigned)t), count);
}

// The loader's curmin / curmax in x and y (fp64: the fp32 centre widened, -/+ 0.75) and its z range [zmin, zmax] of the
// scene.  Every point lies within the scene's z range, so z sets no membership condition.
struct Column {
    double lo[2], hi[2], zmin, zext;
};

__device__ __forceinline__ Column column_at(const float *__restrict__ xyz, long long p, const float *__restrict__ bnd) {
    Column col;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const double v = (double)xyz[3 * (size_t)p + a];
        col.lo[a] = __dsub_rn(v, HALF_XY);
        col.hi[a] = __dadd_rn(v, HALF_XY);
    }
    col.zmin = (double)bnd[2];
    col.zext = __dsub_rn((double)bnd[5], col.zmin);
    return col;
}

// p >= curmin - margin and p <= curmax + margin in x and y, fp64
__device__ __forceinline__ bool in_column(const Column &col, float x, float y, double margin) {
    const double vx = x, vy = y;
    return vx >= __dsub_rn(col.lo[0], margin) && vx <= __dadd_rn(col.hi[0], margin) && vy >= __dsub_rn(col.lo[1], margin) &&
           vy <= __dadd_rn(col.hi[1], margin);
}

// ceil((p - curmin) / (curmax - curmin) * cells), the loader's fp64 order; -0.0 and 0.0 give the same key
__device__ __forceinline__ double vox(double p, double lo, double ext, double cells) {
    return ceil(__dmul_rn(__ddiv_rn(__dsub_rn(p, lo), ext), cells));
}

// Voxel key of a core point, or -1 for the one key value numpy gives every NaN (zero z extent makes all of them NaN).
// For finite points in the core vx, vy lie in -0..32 and vz in 0..62, so the range test fails for NaN only.
__device__ __forceinline__ int vox_key(const Column &col, float x, float y, float z) {
    const double vx = vox(x, col.lo[0], __dsub_rn(col.hi[0], col.lo[0]), 31.0);
    const double vy = vox(y, col.lo[1], __dsub_rn(col.hi[1], col.lo[1]), 31.0);
    const double vz = vox(z, col.zmin, col.zext, 62.0);
    if (!(vx >= 0.0 && vx <= 32.0 && vy >= 0.0 && vy <= 32.0 && vz >= 0.0 && vz <= 62.0)) return -1;
    return (int)vx * (31 * 62) + (int)vy * 62 + (int)vz;
}

__device__ __forceinline__ bool bad_scene(int sid, int s) { return sid < 0 || sid >= s; }

// one CTA per scene (strided): per-axis fp32 minimum and maximum, exact in any order
__global__ void __launch_bounds__(THREADS) bank_bounds_kernel(int s, const float *__restrict__ xyz, const long long *__restrict__ offsets,
                                                               float *__restrict__ bounds) {
    using Reduce = cub::BlockReduce<float, THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
    for (int k = blockIdx.x; k < s; k += gridDim.x) {
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (long long p = offsets[k] + threadIdx.x; p < offsets[k + 1]; p += THREADS)
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float v = xyz[3 * (size_t)p + a];
                lo[a] = fminf(lo[a], v);
                hi[a] = fmaxf(hi[a], v);
            }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float l = Reduce(tmp).Reduce(lo[a], cub::Min());
            __syncthreads();
            const float h = Reduce(tmp).Reduce(hi[a], cub::Max());
            __syncthreads();
            if (threadIdx.x == 0) bounds[6 * (size_t)k + a] = l, bounds[6 * (size_t)k + 3 + a] = h;
        }
    }
}

// h of this call, then step + 1.  Every later kernel of the call reads h, so the counter may move on here.
__global__ void crop_draw_kernel(uint64_t seed, long long *__restrict__ step, uint64_t *__restrict__ h) {
    const uint64_t st = (uint64_t)*step;
    *h = mix64(seed * 0x9E3779B97F4A7C15ull + st);
    *step = (long long)(st + 1);
}

// Work item (crop b, try t, chunk k of the scene): padded and labelled counts and the occupancy bits of the core points
// of CROP_CHUNK scene points.  Bits are gathered in shared memory and OR-ed into the try's record; counts combine by
// integer atomics (labelled) and per-chunk slots (padded, which the compaction also needs), so the result is exact and
// independent of CTA order.  Tries t >= 1 of a crop whose try 0 is valid are skipped.
__global__ void __launch_bounds__(THREADS) crop_try_kernel(int nb, int s, int t0, int ntries, int chunks, const float *__restrict__ xyz,
                                                            const long long *__restrict__ labels, const long long *__restrict__ offsets,
                                                            const float *__restrict__ bounds, const int32_t *__restrict__ scene_ids,
                                                            const uint64_t *__restrict__ hp, int32_t *__restrict__ rec,
                                                            int32_t *__restrict__ chunk_pad) {
    using Reduce = cub::BlockReduce<int, THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
    __shared__ uint32_t bits[VOX_WORDS];
    __shared__ int nan_key;
    const uint64_t h = *hp;
    const long long items = (long long)nb * ntries * chunks;
    for (long long it = blockIdx.x; it < items; it += gridDim.x) {
        const int k = (int)(it % chunks);
        const long long bt = it / chunks;
        const int t = t0 + (int)(bt % ntries), b = (int)(bt / ntries);
        const int sid = scene_ids[b];
        if (bad_scene(sid, s)) continue;
        if (t > 0 && rec[(size_t)b * CROP_TRIES * TRY_STRIDE + R_VALID]) continue;
        const long long off = offsets[sid];
        const int count = (int)(offsets[sid + 1] - off), p0 = k * CROP_CHUNK;
        if (p0 >= count) continue;
        int32_t *r = rec + ((size_t)b * CROP_TRIES + t) * TRY_STRIDE;
        const Column col = column_at(xyz, off + centre_pos(h, b, t, count), bounds + 6 * (size_t)sid);
        for (int w = threadIdx.x; w < VOX_WORDS; w += THREADS) bits[w] = 0;
        if (threadIdx.x == 0) nan_key = 0;
        __syncthreads();
        int pad = 0, lab = 0;
        const int p1 = min(count, p0 + CROP_CHUNK);
        for (int p = p0 + threadIdx.x; p < p1; p += THREADS) {
            const float *q = xyz + 3 * (size_t)(off + p);
            const float x = q[0], y = q[1];
            if (!in_column(col, x, y, CROP_PAD)) continue;
            ++pad;
            lab += labels[off + p] > 0;
            if (!in_column(col, x, y, CROP_CORE)) continue;
            const int key = vox_key(col, x, y, q[2]);
            if (key >= 0) atomicOr(&bits[key >> 5], 1u << (key & 31));
            else nan_key = 1;
        }
        pad = Reduce(tmp).Sum(pad);
        __syncthreads();
        lab = Reduce(tmp).Sum(lab);
        __syncthreads();  // bits and nan_key complete
        if (threadIdx.x == 0) {
            chunk_pad[((size_t)b * CROP_TRIES + t) * chunks + k] = pad;
            if (lab) atomicAdd(r + R_LAB, lab);
            if (nan_key) atomicOr(r + R_NAN, 1);
        }
        for (int w = threadIdx.x; w < VOX_WORDS; w += THREADS)
            if (bits[w]) atomicOr((uint32_t *)r + TRY_HEAD + w, bits[w]);
        __syncthreads();  // before the next item clears bits
    }
}

// Work item (crop b, try t): padded count, occupied keys (+1 for NaN) and the loader's test, fp64 in its order:
// labelled / padded >= 0.7 and keys / 31 / 31 / 62 >= 0.02.
__global__ void __launch_bounds__(THREADS) crop_judge_kernel(int nb, int s, int t0, int ntries, int chunks, const long long *__restrict__ offsets,
                                                              const int32_t *__restrict__ scene_ids, int32_t *__restrict__ rec,
                                                              const int32_t *__restrict__ chunk_pad) {
    using Reduce = cub::BlockReduce<int, THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
    for (int it = blockIdx.x; it < nb * ntries; it += gridDim.x) {
        const int t = t0 + it % ntries, b = it / ntries;
        const int sid = scene_ids[b];
        if (bad_scene(sid, s)) continue;
        if (t > 0 && rec[(size_t)b * CROP_TRIES * TRY_STRIDE + R_VALID]) continue;
        int32_t *r = rec + ((size_t)b * CROP_TRIES + t) * TRY_STRIDE;
        const int nch = ceil_div((int)(offsets[sid + 1] - offsets[sid]), CROP_CHUNK);
        const int32_t *cp = chunk_pad + ((size_t)b * CROP_TRIES + t) * chunks;
        int pad = 0, keys = 0;
        for (int k = threadIdx.x; k < nch; k += THREADS) pad += cp[k];
        for (int w = threadIdx.x; w < VOX_WORDS; w += THREADS) keys += __popc((uint32_t)r[TRY_HEAD + w]);
        pad = Reduce(tmp).Sum(pad);
        __syncthreads();
        keys = Reduce(tmp).Sum(keys);
        if (threadIdx.x == 0) {
            keys += r[R_NAN];
            r[R_PAD] = pad;
            r[R_VALID] = pad > 0 && __ddiv_rn((double)r[R_LAB], (double)pad) >= 0.7 &&
                         __ddiv_rn(__ddiv_rn(__ddiv_rn((double)keys, 31.0), 31.0), 62.0) >= 0.02;
        }
        __syncthreads();
    }
}

// Work item (crop b, chunk k): the taken try (the first valid one, else the tenth), then the scene-local indices of its
// padded points in chunk k, in ascending order, at local[b * max_count + (padded points of the chunks before k) ...]
// (a stable block scan).  Chunk 0 also writes the crop's center, tries, valid and padded count.
__global__ void __launch_bounds__(THREADS) crop_compact_kernel(int nb, int s, int chunks, int max_count, const float *__restrict__ xyz,
                                                                const long long *__restrict__ offsets, const float *__restrict__ bounds,
                                                                const int32_t *__restrict__ scene_ids, const uint64_t *__restrict__ hp,
                                                                const int32_t *__restrict__ rec, const int32_t *__restrict__ chunk_pad,
                                                                int32_t *__restrict__ local, int32_t *__restrict__ crop_count,
                                                                int32_t *__restrict__ center, int32_t *__restrict__ tries,
                                                                uint8_t *__restrict__ valid) {
    using Reduce = cub::BlockReduce<int, THREADS>;
    using Scan = cub::BlockScan<int, THREADS>;
    __shared__ typename Reduce::TempStorage rtmp;
    __shared__ typename Scan::TempStorage stmp;
    const uint64_t h = *hp;
    for (long long it = blockIdx.x; it < (long long)nb * chunks; it += gridDim.x) {
        const int k = (int)(it % chunks), b = (int)(it / chunks);
        const int sid = scene_ids[b];
        if (bad_scene(sid, s)) {
            if (k == 0 && threadIdx.x == 0) center[b] = -1, tries[b] = 0, valid[b] = 0, crop_count[b] = 0;
            continue;
        }
        const long long off = offsets[sid];
        const int count = (int)(offsets[sid + 1] - off), p0 = k * CROP_CHUNK;
        if (p0 >= count) continue;
        const int32_t *r0 = rec + (size_t)b * CROP_TRIES * TRY_STRIDE;
        int t = 0;
        while (t < CROP_TRIES - 1 && !r0[(size_t)t * TRY_STRIDE + R_VALID]) ++t;
        const int32_t *r = r0 + (size_t)t * TRY_STRIDE;
        const int c = centre_pos(h, b, t, count);
        if (k == 0 && threadIdx.x == 0) center[b] = c, tries[b] = t + 1, valid[b] = (uint8_t)r[R_VALID], crop_count[b] = r[R_PAD];
        const int32_t *cp = chunk_pad + ((size_t)b * CROP_TRIES + t) * chunks;
        int base = 0;
        for (int j = threadIdx.x; j < k; j += THREADS) base += cp[j];
        base = Reduce(rtmp).Sum(base);  // valid in thread 0
        const Column col = column_at(xyz, off + c, bounds + 6 * (size_t)sid);
        const int q0 = p0 + threadIdx.x * CROP_ITEMS;
        uint32_t in = 0;
#pragma unroll 4
        for (int i = 0; i < CROP_ITEMS; ++i) {
            const int p = q0 + i;
            if (p < count) {
                const float *q = xyz + 3 * (size_t)(off + p);
                if (in_column(col, q[0], q[1], CROP_PAD)) in |= 1u << i;
            }
        }
        // thread 0 feeds base into the scan, so every other thread's exclusive sum already includes it
        int rank;
        Scan(stmp).ExclusiveSum(threadIdx.x == 0 ? base + __popc(in) : __popc(in), rank);
        int32_t *out = local + (size_t)b * max_count + (threadIdx.x == 0 ? base : rank);
        for (; in; in &= in - 1) *out++ = q0 + __ffs(in) - 1;
        __syncthreads();
    }
}

// slot (b, j): bank row of position sample_pos(h, b, j, padded count) of the taken column, its target and weight
__global__ void __launch_bounds__(THREADS) crop_slot_kernel(long long total, int npoints, int s, int max_count, int num_classes,
                                                             const float *__restrict__ xyz, const long long *__restrict__ labels,
                                                             const long long *__restrict__ offsets, const float *__restrict__ bounds,
                                                             const int32_t *__restrict__ scene_ids, const uint64_t *__restrict__ hp,
                                                             const int32_t *__restrict__ local, const int32_t *__restrict__ crop_count,
                                                             const int32_t *__restrict__ center, const float *__restrict__ labelweights,
                                                             int32_t *__restrict__ point_index, long long *__restrict__ target,
                                                             float *__restrict__ weights) {
    const long long e = (long long)blockIdx.x * THREADS + threadIdx.x;
    if (e >= total) return;
    const int b = (int)(e / npoints), j = (int)(e - (long long)b * npoints);
    const int sid = scene_ids[b];
    // an empty column needs a non-finite centre (a finite one lies in its own column): nothing to draw from
    if (bad_scene(sid, s) || crop_count[b] == 0) {
        point_index[e] = -1;
        target[e] = 0;
        weights[e] = 0.f;
        return;
    }
    const long long off = offsets[sid];
    const long long p = off + local[(size_t)b * max_count + sample_pos(*hp, b, j, crop_count[b])];
    point_index[e] = (int32_t)p;
    const Column col = column_at(xyz, off + center[b], bounds + 6 * (size_t)sid);
    const bool core = in_column(col, xyz[3 * (size_t)p], xyz[3 * (size_t)p + 1], CROP_CORE);
    const long long l = labels[p];
    target[e] = l;
    float w = core ? 1.f : 0.f;
    if (labelweights) w = (l >= 0 && l < num_classes) ? __fmul_rn(labelweights[l], w) : 0.f;
    weights[e] = w;
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
    rows_kernel<false><<<strided_blocks(elems), THREADS, 0, s>>>(elems, c, point_index, xyz, feats, points);
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
    rows_kernel<false><<<strided_blocks(elems), THREADS, 0, s>>>(elems, c, point_index, xyz, feats, points);
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

extern "C" int pn2_scene_bank_bounds(int s, long long n, const float *xyz, const long long *offsets, float *bounds, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(s >= 1, "scene_bank_bounds: need s >= 1 scenes (s=%d)", s);
    PN2_REQUIRE(n >= 1 && n < (1ll << 31), "scene_bank_bounds: need 1 <= n < 2^31 points (n=%lld)", n);
    PN2_REQUIRE(xyz && offsets && bounds, "scene_bank_bounds: null pointer");
    bank_bounds_kernel<<<min(s, 4 * sm_count()), THREADS, 0, (cudaStream_t)stream>>>(s, xyz, offsets, bounds);
    PN2_LAUNCH_OK("bank_bounds_kernel");
    return PN2_OK;
}

extern "C" int pn2_scene_crops(int s, long long n, int c, int max_count, const float *xyz, const float *feats, const long long *labels,
                               const long long *offsets, const float *bounds, int b, const int32_t *scene_ids, int npoints,
                               unsigned long long seed, long long *step, const float *labelweights, int num_classes, int32_t *point_index,
                               float *points, long long *target, float *weights, int32_t *center, int32_t *tries, uint8_t *valid,
                               void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 1 && npoints >= 1 && c >= 0, "scene_crops: bad dims b=%d npoints=%d c=%d", b, npoints, c);
    PN2_REQUIRE((long long)b * npoints < (1ll << 31), "scene_crops: b * npoints must be < 2^31");
    PN2_REQUIRE(s >= 1 && n >= 1 && n < (1ll << 31), "scene_crops: need s >= 1 scenes and 1 <= n < 2^31 points (s=%d n=%lld)", s, n);
    PN2_REQUIRE(max_count >= 1 && max_count <= n, "scene_crops: max_count must be in [1, n] (max_count=%d)", max_count);
    PN2_REQUIRE(!labelweights || num_classes >= 1, "scene_crops: labelweights need num_classes >= 1");
    PN2_REQUIRE(xyz && (c == 0 || feats) && labels && offsets && bounds && scene_ids && step && point_index && points && target &&
                    weights && center && tries && valid,
                "scene_crops: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int chunks = ceil_div(max_count, CROP_CHUNK);
    auto round = [](size_t v) { return (v + 255) / 256 * 256; };
    const size_t h_bytes = 256, rec_bytes = round((size_t)b * CROP_TRIES * TRY_STRIDE * sizeof(int32_t)),
                 cp_bytes = round((size_t)b * CROP_TRIES * chunks * sizeof(int32_t)), cc_bytes = round((size_t)b * sizeof(int32_t)),
                 local_bytes = (size_t)b * max_count * sizeof(int32_t);
    Scratch scratch_mem(st);  // [h | try records | per-chunk padded counts | padded count per crop | compacted columns]
    PN2_CUDA(scratch_mem.alloc(h_bytes + rec_bytes + cp_bytes + cc_bytes + local_bytes));
    unsigned char *scratch = (unsigned char *)scratch_mem.ptr;
    uint64_t *h = (uint64_t *)scratch;
    int32_t *rec = (int32_t *)(scratch + h_bytes), *chunk_pad = (int32_t *)(scratch + h_bytes + rec_bytes);
    int32_t *crop_count = (int32_t *)(scratch + h_bytes + rec_bytes + cp_bytes);
    int32_t *local = (int32_t *)(scratch + h_bytes + rec_bytes + cp_bytes + cc_bytes);
    PN2_CUDA(cudaMemsetAsync(rec, 0, rec_bytes, st));
    crop_draw_kernel<<<1, 1, 0, st>>>((uint64_t)seed, step, h);
    PN2_LAUNCH_OK("crop_draw_kernel");
    const long long cap = 32ll * sm_count();
    auto ctas = [cap](long long items) { return (unsigned)(items < cap ? items : cap); };
    // try 0 of every crop first; tries 1-9 only where it failed (the other CTAs skip at once)
    crop_try_kernel<<<ctas((long long)b * chunks), THREADS, 0, st>>>(b, s, 0, 1, chunks, xyz, labels, offsets, bounds, scene_ids, h, rec,
                                                                      chunk_pad);
    PN2_LAUNCH_OK("crop_try_kernel");
    crop_judge_kernel<<<ctas(b), THREADS, 0, st>>>(b, s, 0, 1, chunks, offsets, scene_ids, rec, chunk_pad);
    PN2_LAUNCH_OK("crop_judge_kernel");
    crop_try_kernel<<<ctas((long long)b * (CROP_TRIES - 1) * chunks), THREADS, 0, st>>>(b, s, 1, CROP_TRIES - 1, chunks, xyz, labels, offsets,
                                                                                         bounds, scene_ids, h, rec, chunk_pad);
    PN2_LAUNCH_OK("crop_try_kernel");
    crop_judge_kernel<<<ctas((long long)b * (CROP_TRIES - 1)), THREADS, 0, st>>>(b, s, 1, CROP_TRIES - 1, chunks, offsets, scene_ids, rec,
                                                                                  chunk_pad);
    PN2_LAUNCH_OK("crop_judge_kernel");
    crop_compact_kernel<<<ctas((long long)b * chunks), THREADS, 0, st>>>(b, s, chunks, max_count, xyz, offsets, bounds, scene_ids, h, rec,
                                                                          chunk_pad, local, crop_count, center, tries, valid);
    PN2_LAUNCH_OK("crop_compact_kernel");
    const long long slots = (long long)b * npoints, elems = slots * (3 + c);
    crop_slot_kernel<<<blocks_for(slots), THREADS, 0, st>>>(slots, npoints, s, max_count, labelweights ? num_classes : 0, xyz, labels, offsets,
                                                            bounds, scene_ids, h, local, crop_count, center, labelweights, point_index,
                                                            target, weights);
    PN2_LAUNCH_OK("crop_slot_kernel");
    rows_kernel<true><<<strided_blocks(elems), THREADS, 0, st>>>(elems, c, point_index, xyz, feats, points);
    PN2_LAUNCH_OK("rows_kernel");
    return PN2_OK;
}
