// scatter_det.cu -- deterministic backward of gather / grouping / three_interpolate (SURVEY 8f row N1).
//
// The reference's backward kernels (utils/src/sampling_gpu.cu:46-83 gather_points_grad, group_points_gpu.cu:47-83
// group_points_grad, interpolate_gpu.cu:120-161 three_interpolate_grad) accumulate with atomicAdd, so the fp32 summation
// order -- and with it the low bits of every gradient -- changes from run to run.  Here the index list is inverted once
// (stable sort of (cloud * n + idx[p]) -> p; a segment-start table), and every output element sums ITS contributions
// in ascending source position: one fixed order, bit-identical results, no atomics.
//
//     grad_points[b, c, k] += sum over p in segment(b, k), ascending:  w[b, p] * grad_out[b, c, p / div]
//
// with div = 1, w = 1 for gather / grouping (p runs over the (npoints[, nsample]) index list) and div = 3 for
// three_interpolate (p runs over the (n, 3) neighbour list, the source column is the fine point p / 3).
// The stable sort is cub::DeviceRadixSort (plumbing, not the measured path); its temporary storage comes from the
// stream-ordered allocator, so the call is asynchronous and graph-capturable.
#include <cub/cub.cuh>

#include "common.cuh"

namespace pn2 {
namespace {

__global__ void inv_keys_kernel(long long total, long long J, int n, const int32_t *__restrict__ idx, uint32_t *__restrict__ keys,
                                int32_t *__restrict__ pos) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long b = e / J;
        keys[e] = (uint32_t)(b * n + idx[e]);
        pos[e] = (int32_t)(e - b * J);
    }
}

// seg_start[key] = first sorted slot whose key is >= key, for key in [0, b*n]; slots hold ascending keys
__global__ void seg_start_kernel(long long total, long long nkeys, const uint32_t *__restrict__ sorted, int32_t *__restrict__ seg_start) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e <= total; e += (long long)gridDim.x * blockDim.x) {
        const long long hi = e < total ? (long long)sorted[e] : nkeys;       // keys up to and including `hi` start at or before e
        const long long lo = e == 0 ? -1 : (long long)sorted[e - 1];         // keys <= lo started earlier
        for (long long k = lo + 1; k <= hi; ++k) seg_start[k] = (int32_t)e;
    }
}

constexpr int DET_THREADS = 128;
constexpr int DET_CH = 8;

// grid (ceil(n / DET_THREADS), ceil(c / DET_CH), b); thread <-> one destination point, DET_CH channels
__global__ void __launch_bounds__(DET_THREADS)
scatter_det_kernel(int c, int n, long long J, int div, const float *__restrict__ grad_out, const int32_t *__restrict__ seg_start,
                   const int32_t *__restrict__ pos, const float *__restrict__ weight, float *__restrict__ grad_points) {
    const int k = blockIdx.x * DET_THREADS + threadIdx.x;
    if (k >= n) return;
    const int b = blockIdx.z;
    const int c0 = blockIdx.y * DET_CH;
    const long long key = (long long)b * n + k;
    const int s0 = seg_start[key], s1 = seg_start[key + 1];
    if (s0 == s1) return;
    const long long cols = J / div;                      // columns of grad_out per channel
    const float *g = grad_out + ((size_t)b * c + c0) * cols;
    const float *w = weight ? weight + (size_t)b * J : nullptr;
    float acc[DET_CH];
#pragma unroll
    for (int q = 0; q < DET_CH; ++q) acc[q] = 0.f;
    const int cc = min(DET_CH, c - c0);
    for (int s = s0; s < s1; ++s) {
        const int p = pos[s];
        const int col = div == 1 ? p : p / div;
        const float wp = w ? __ldg(w + p) : 1.f;
#pragma unroll
        for (int q = 0; q < DET_CH; ++q)
            if (q < cc) {
                const float go = __ldg(g + (size_t)q * cols + col);
                acc[q] = __fadd_rn(acc[q], w ? __fmul_rn(go, wp) : go);
            }
    }
    float *dst = grad_points + ((size_t)b * c + c0) * n + k;
#pragma unroll
    for (int q = 0; q < DET_CH; ++q)
        if (q < cc) dst[(size_t)q * n] += acc[q];
}

// Channel-last variant over row matrices: thread <-> (destination point, channel), lanes along channels, so each
// contribution is a contiguous slice of one row of g_in; same per-element order and arithmetic as scatter_det_kernel.
// Every element of grad_points is written (0 for a point no row refers to).
__global__ void __launch_bounds__(256)
scatter_det_cl_kernel(long long total, int d, int n, long long J, int div, const float *__restrict__ g_in, int row_stride,
                      int col_offset, const int32_t *__restrict__ seg_start, const int32_t *__restrict__ pos,
                      const float *__restrict__ weight, float *__restrict__ grad_points) {
    const long long rows_per_cloud = J / div;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long key = e / d;  // b * n + k
        const int ch = (int)(e - key * d);
        const long long b = key / n;
        const int s0 = __ldg(seg_start + key), s1 = __ldg(seg_start + key + 1);
        const float *g = g_in + b * rows_per_cloud * row_stride + col_offset + ch;
        const float *w = weight ? weight + b * J : nullptr;
        float acc = 0.f;
        for (int s = s0; s < s1; ++s) {
            const int p = __ldg(pos + s);
            const int row = div == 1 ? p : p / div;
            const float go = __ldg(g + (long long)row * row_stride);
            acc = __fadd_rn(acc, w ? __fmul_rn(go, __ldg(w + p)) : go);
        }
        grad_points[e] = acc;
    }
}

}  // namespace

size_t segment_sort_scratch_bytes(long long total, long long nkeys) {
    int end_bit = 1;
    while ((1ll << end_bit) < nkeys) ++end_bit;
    size_t tmp_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (const uint32_t *)nullptr, (uint32_t *)nullptr, (const int32_t *)nullptr,
                                    (int32_t *)nullptr, (int)total, 0, end_bit);
    return ((size_t)total * sizeof(uint32_t) + 255) / 256 * 256 + tmp_bytes;
}

int segment_sort(long long total, long long nkeys, const uint32_t *keys_in, const int32_t *pos_in, void *scratch, int32_t *seg_start,
                 int32_t *pos, cudaStream_t s) {
    int end_bit = 1;
    while ((1ll << end_bit) < nkeys) ++end_bit;
    size_t tmp_bytes = 0;
    PN2_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (const uint32_t *)nullptr, (uint32_t *)nullptr, (const int32_t *)nullptr,
                                             (int32_t *)nullptr, (int)total, 0, end_bit, s));
    const size_t key_bytes = ((size_t)total * sizeof(uint32_t) + 255) / 256 * 256;
    uint32_t *keys_out = (uint32_t *)scratch;
    // LSD radix sort is stable: equal keys keep ascending source position
    PN2_CUDA(cub::DeviceRadixSort::SortPairs((unsigned char *)scratch + key_bytes, tmp_bytes, keys_in, keys_out, pos_in, pos, (int)total, 0,
                                             end_bit, s));
    const int blocks = (int)((total + 255) / 256 < 2048 ? (total + 255) / 256 : 2048);
    seg_start_kernel<<<blocks, 256, 0, s>>>(total, nkeys, keys_out, seg_start);
    PN2_LAUNCH_OK("seg_start_kernel");
    return PN2_OK;
}

}  // namespace pn2

extern "C" int pn2_inverse_index(int b, int n, long long j, const int32_t *idx, int32_t *seg_start, int32_t *pos, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && n >= 1 && j >= 0, "inverse_index: bad dims b=%d n=%d j=%lld", b, n, j);
    PN2_REQUIRE((long long)b * n < (1ll << 31) && (long long)b * j < (1ll << 31), "inverse_index: more than 2^31 keys");
    if (b == 0) return PN2_OK;
    PN2_REQUIRE(seg_start && (j == 0 || (idx && pos)), "inverse_index: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    const long long total = (long long)b * j, nkeys = (long long)b * n;
    if (total == 0) {
        PN2_CUDA(cudaMemsetAsync(seg_start, 0, (size_t)(nkeys + 1) * sizeof(int32_t), s));
        return PN2_OK;
    }
    const size_t key_bytes = ((size_t)total * sizeof(uint32_t) + 255) / 256 * 256;
    Scratch scratch_mem(s);  // [keys in | positions in | segment_sort scratch], released on every return below
    PN2_CUDA(scratch_mem.alloc(2 * key_bytes + segment_sort_scratch_bytes(total, nkeys)));
    unsigned char *scratch = (unsigned char *)scratch_mem.ptr;
    uint32_t *keys_in = (uint32_t *)scratch;
    int32_t *pos_in = (int32_t *)(scratch + key_bytes);
    const int blocks = (int)((total + 255) / 256 < 2048 ? (total + 255) / 256 : 2048);
    inv_keys_kernel<<<blocks, 256, 0, s>>>(total, j, n, idx, keys_in, pos_in);
    PN2_LAUNCH_OK("inv_keys_kernel");
    return segment_sort(total, nkeys, keys_in, pos_in, scratch + 2 * key_bytes, seg_start, pos, s);
}

extern "C" int pn2_scatter_rows_det(int b, int c, int n, long long j, int div, const float *grad_out, const int32_t *seg_start,
                                    const int32_t *pos, const float *weight, float *grad_points, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && c >= 0 && n >= 1 && j >= 0 && (div == 1 || div == 3), "scatter_rows_det: bad dims b=%d c=%d n=%d j=%lld div=%d", b, c,
                n, j, div);
    PN2_REQUIRE(j % div == 0, "scatter_rows_det: j=%lld is not a multiple of div=%d", j, div);
    if (b == 0 || c == 0 || j == 0) return PN2_OK;
    PN2_REQUIRE(grad_out && seg_start && pos && grad_points, "scatter_rows_det: null pointer");
    PN2_REQUIRE(b <= 65535 && (c + DET_CH - 1) / DET_CH <= 65535, "scatter_rows_det: b and c/8 must be <= 65535");
    dim3 grid((unsigned)((n + DET_THREADS - 1) / DET_THREADS), (unsigned)((c + DET_CH - 1) / DET_CH), (unsigned)b);
    scatter_det_kernel<<<grid, DET_THREADS, 0, (cudaStream_t)stream>>>(c, n, j, div, grad_out, seg_start, pos, weight, grad_points);
    PN2_LAUNCH_OK("scatter_det_kernel");
    return PN2_OK;
}

extern "C" int pn2_scatter_rows_det_cl(int b, int d, int n, long long j, int div, const float *g_in, int row_stride, int col_offset,
                                       const int32_t *seg_start, const int32_t *pos, const float *weight, float *grad_points, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && d >= 0 && n >= 1 && j >= 0 && (div == 1 || div == 3), "scatter_rows_det_cl: bad dims b=%d d=%d n=%d j=%lld div=%d",
                b, d, n, j, div);
    PN2_REQUIRE(j % div == 0, "scatter_rows_det_cl: j=%lld is not a multiple of div=%d", j, div);
    PN2_REQUIRE(col_offset >= 0 && row_stride >= col_offset + d, "scatter_rows_det_cl: row_stride=%d col_offset=%d d=%d", row_stride,
                col_offset, d);
    PN2_REQUIRE((long long)b * n < (1ll << 31) && (long long)b * j < (1ll << 31), "scatter_rows_det_cl: more than 2^31 keys");
    if (b == 0 || d == 0) return PN2_OK;
    PN2_REQUIRE(seg_start && grad_points && (j == 0 || (g_in && pos)), "scatter_rows_det_cl: null pointer");
    const long long total = (long long)b * n * d;
    const unsigned grid = (unsigned)((total + 255) / 256 < 8ll * sm_count() ? (total + 255) / 256 : 8ll * sm_count());
    scatter_det_cl_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(total, d, n, j, div, g_in, row_stride, col_offset, seg_start, pos, weight,
                                                                   grad_points);
    PN2_LAUNCH_OK("scatter_det_cl_kernel");
    return PN2_OK;
}
