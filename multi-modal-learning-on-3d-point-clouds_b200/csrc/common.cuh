// common.cuh -- shared helpers for libpn2_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "pn2_abi.h"

namespace pn2 {

// Error plumbing (abi.cu).  set_error returns `status` so call sites can `return set_error(...)`.
int set_error(int status, const char *fmt, ...);
void count_launch(int n = 1);
int sm_count();
// Stream-ordered scratch (cudaMallocAsync).  The first call on a device raises the pool's release threshold so that the
// memory stays in the pool between calls instead of going back to the driver at every synchronisation.
cudaError_t scratch_alloc(void **ptr, size_t bytes, cudaStream_t stream);
// Owner of one stream-ordered scratch block: the block goes back to the pool (cudaFreeAsync on the same stream) on EVERY
// way out of the entry point, error returns included.
struct Scratch {
    void *ptr = nullptr;
    cudaStream_t stream;
    explicit Scratch(cudaStream_t s) : stream(s) {}
    Scratch(const Scratch &) = delete;
    Scratch &operator=(const Scratch &) = delete;
    ~Scratch() {
        if (ptr) cudaFreeAsync(ptr, stream);
    }
    cudaError_t alloc(size_t bytes) { return scratch_alloc(&ptr, bytes, stream); }
};

// Stable inversion of a key list (scatter_det.cu): keys_in (total) with values in [0, nkeys), pos_in (total) the payload
// of each key -> pos (total) = the payloads in ascending key order, equal keys in their input order, and seg_start
// (nkeys + 1): seg_start[k] = first slot of pos whose key is >= k.  One device radix sort; `scratch` holds
// segment_sort_scratch_bytes(total, nkeys) bytes.  No host synchronisation.
size_t segment_sort_scratch_bytes(long long total, long long nkeys);
int segment_sort(long long total, long long nkeys, const uint32_t *keys_in, const int32_t *pos_in, void *scratch, int32_t *seg_start,
                 int32_t *pos, cudaStream_t s);

#define PN2_REQUIRE(cond, ...)                                             \
    do {                                                                   \
        if (!(cond)) return pn2::set_error(PN2_ERR_INVALID_ARGUMENT, __VA_ARGS__); \
    } while (0)

#define PN2_CUDA(call)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess)                                                               \
            return pn2::set_error(PN2_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__)); \
    } while (0)

#define PN2_LAUNCH_OK(name)                                                                   \
    do {                                                                                      \
        cudaError_t e__ = cudaGetLastError();                                                 \
        if (e__ != cudaSuccess)                                                               \
            return pn2::set_error(PN2_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e__)); \
        pn2::count_launch();                                                                  \
    } while (0)

// Squared distance with exactly the rounding sequence of the reference's kernels as built by
// nvcc -O2 (fmad contraction of utils/src/sampling_gpu.cu:133, ball_query_gpu.cu:33,
// interpolate_gpu.cu:36):  fma(dz,dz, fma(dx,dx, rn(dy*dy))).   (SURVEY.md F7)
__device__ __forceinline__ float dist_ref(float ax, float ay, float az, float bx, float by, float bz) {
    float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
    return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Largest power of two <= min(n, 1024): the reference's FPS block size, utils/src/cuda_utils.h:10-14.
inline int ref_block_size(int n) {
    int p = 1;
    while (p * 2 <= n && p * 2 <= 1024) p *= 2;
    return p;
}

}  // namespace pn2
