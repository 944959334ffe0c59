// interpolate.cu -- three nearest neighbours and inverse-distance interpolation.
// Replaces utils/src/interpolate_gpu.cu:9-161 (three_nn, three_interpolate, three_interpolate_grad).
//
// three_nn contract (SURVEY.md A.4): per unknown point, scanning known k = 0..m-1 ascending, a
// strict-'<' insertion into (best1 <= best2 <= best3); squared distances in the reference's fp32
// contraction order; +inf / index 0 when m < 3.  One thread per unknown point keeps that scan
// order; the known set is staged once per CTA in shared memory as float4 so every test is one
// broadcast LDS.128 instead of three dependent global loads per thread.
//
// three_interpolate: a thread owns one output point for a chunk of channels; idx and weight are
// read once (the reference re-reads them for every channel) and the stores of a warp are coalesced.
#include "common.cuh"

#include <algorithm>

namespace pn2 {
namespace {

constexpr int NN_THREADS = 256;
constexpr int NN_TILE = 2048;  // known points per tile: 32 KB of float4

struct Top3 {
    float d1, d2, d3;
    int i1, i2, i3;
};

__device__ __forceinline__ void top3_insert(Top3 &t, float d, int k) {
    // interpolate_gpu.cu:37-48; the reference compares in double, which orders float values identically
    if (d < t.d3) {
        if (d < t.d1) {
            t.d3 = t.d2; t.i3 = t.i2;
            t.d2 = t.d1; t.i2 = t.i1;
            t.d1 = d;    t.i1 = k;
        } else if (d < t.d2) {
            t.d3 = t.d2; t.i3 = t.i2;
            t.d2 = d;    t.i2 = k;
        } else {
            t.d3 = d;    t.i3 = k;
        }
    }
}

__device__ __forceinline__ Top3 three_nn_scan(int m, const float *__restrict__ known, float ux, float uy, float uz,
                                              float4 *tile) {
    Top3 t;
    t.d1 = t.d2 = t.d3 = __int_as_float(0x7f800000);  // (float)1e40 == +inf, interpolate_gpu.cu:28,50
    t.i1 = t.i2 = t.i3 = 0;
    for (int base = 0; base < m; base += NN_TILE) {
        const int tn = min(NN_TILE, m - base);
        __syncthreads();
        for (int p = threadIdx.x; p < tn; p += NN_THREADS) {
            const float *s = known + (size_t)(base + p) * 3;
            tile[p] = make_float4(s[0], s[1], s[2], 0.f);
        }
        __syncthreads();
        int p = 0;
        for (; p + 4 <= tn; p += 4) {
            float d[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float4 kp = tile[p + u];
                d[u] = dist_ref(ux, uy, uz, kp.x, kp.y, kp.z);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) top3_insert(t, d[u], base + p + u);
        }
        for (; p < tn; ++p) {
            const float4 kp = tile[p];
            top3_insert(t, dist_ref(ux, uy, uz, kp.x, kp.y, kp.z), base + p);
        }
    }
    return t;
}

__global__ void __launch_bounds__(NN_THREADS)
three_nn_kernel(int n, int m, const float *__restrict__ unknown, const float *__restrict__ known,
                float *__restrict__ dist2, int32_t *__restrict__ idx) {
    __shared__ float4 tile[NN_TILE];
    const int b = blockIdx.y;
    const int i = blockIdx.x * NN_THREADS + threadIdx.x;
    const int ic = min(i, n - 1);
    const float *u = unknown + ((size_t)b * n + ic) * 3;
    const Top3 t = three_nn_scan(m, known + (size_t)b * m * 3, u[0], u[1], u[2], tile);
    if (i < n) {
        float *od = dist2 + ((size_t)b * n + i) * 3;
        int32_t *oi = idx + ((size_t)b * n + i) * 3;
        od[0] = t.d1; od[1] = t.d2; od[2] = t.d3;
        oi[0] = t.i1; oi[1] = t.i2; oi[2] = t.i3;
    }
}

// three_nn + the reference's weight formula (model/pointnet2_utils.py:97, model/pointnet_util.py:206-208):
// dist = sqrt(d2); dist[dist < 1e-10] = 1e-10; w = 1/dist; w = w / (w0 + w1 + w2)
__global__ void __launch_bounds__(NN_THREADS)
three_nn_weights_kernel(int n, int m, const float *__restrict__ unknown, const float *__restrict__ known,
                        int32_t *__restrict__ idx, float *__restrict__ weight) {
    __shared__ float4 tile[NN_TILE];
    const int b = blockIdx.y;
    const int i = blockIdx.x * NN_THREADS + threadIdx.x;
    const int ic = min(i, n - 1);
    const float *u = unknown + ((size_t)b * n + ic) * 3;
    const Top3 t = three_nn_scan(m, known + (size_t)b * m * 3, u[0], u[1], u[2], tile);
    if (i < n) {
        float e1 = __fsqrt_rn(t.d1), e2 = __fsqrt_rn(t.d2), e3 = __fsqrt_rn(t.d3);
        e1 = e1 < 1e-10f ? 1e-10f : e1;
        e2 = e2 < 1e-10f ? 1e-10f : e2;
        e3 = e3 < 1e-10f ? 1e-10f : e3;
        const float w1 = __fdiv_rn(1.0f, e1), w2 = __fdiv_rn(1.0f, e2), w3 = __fdiv_rn(1.0f, e3);
        const float s = __fadd_rn(__fadd_rn(w1, w2), w3);
        float *ow = weight + ((size_t)b * n + i) * 3;
        int32_t *oi = idx + ((size_t)b * n + i) * 3;
        ow[0] = __fdiv_rn(w1, s); ow[1] = __fdiv_rn(w2, s); ow[2] = __fdiv_rn(w3, s);
        oi[0] = t.i1; oi[1] = t.i2; oi[2] = t.i3;
    }
}

constexpr int TI_THREADS = 256;
constexpr int TI_CH = 8;

// out[b,c,i] = fma(w2, f[b,c,i2], fma(w0, f[b,c,i0], rn(w1 * f[b,c,i1])))   (the reference's contraction,
// SURVEY.md 2.2 K8)
__global__ void __launch_bounds__(TI_THREADS)
three_interpolate_kernel(int c, int m, int n, const float *__restrict__ points, const int32_t *__restrict__ idx,
                         const float *__restrict__ weight, float *__restrict__ out) {
    const int i = blockIdx.x * TI_THREADS + threadIdx.x;
    if (i >= n) return;
    const int b = blockIdx.z;
    const int c0 = blockIdx.y * TI_CH;
    const int32_t *id = idx + ((size_t)b * n + i) * 3;
    const float *w = weight + ((size_t)b * n + i) * 3;
    const int i0 = id[0], i1 = id[1], i2 = id[2];
    const float w0 = w[0], w1 = w[1], w2 = w[2];
    const float *f = points + ((size_t)b * c + c0) * m;
    float *o = out + ((size_t)b * c + c0) * n + i;
    const int cc = min(TI_CH, c - c0);
    float a0[TI_CH], a1[TI_CH], a2[TI_CH];
#pragma unroll
    for (int k = 0; k < TI_CH; ++k)
        if (k < cc) {
            a0[k] = __ldg(f + (size_t)k * m + i0);
            a1[k] = __ldg(f + (size_t)k * m + i1);
            a2[k] = __ldg(f + (size_t)k * m + i2);
        }
#pragma unroll
    for (int k = 0; k < TI_CH; ++k)
        if (k < cc) __stcs(o + (size_t)k * n, __fmaf_rn(w2, a2[k], __fmaf_rn(w0, a0[k], __fmul_rn(w1, a1[k]))));
}

// Shared-memory variant: a CTA stages the coarse features of CC channels TRANSPOSED ([m][CC], so a neighbour's CC
// channels are contiguous: one LDS.128 per 4 channels), then every thread streams output points: lane <-> point keeps
// the stores of a warp coalesced along n.  HBM sees the coarse features once per CTA slice, idx/weight once per channel
// chunk, and the output once.
constexpr int TS_THREADS = 256;
constexpr int LC_GRAN = 32;  // points per warp granule of the lane-along-channel kernel

// T threads per CTA, MINB CTAs per SM (by the size of the staged tile).  With one or two CTAs per SM the index / weight
// vectors of the NEXT four points are loaded while the current four are interpolated (they are the only long-latency loads
// of the loop and 8-16 warps do not hide them; with three CTAs per SM the 85-register budget has no room for them).
template <int CC, int PAD, int T, int MINB>
__global__ void __launch_bounds__(T, MINB)
three_interpolate_smem_kernel(int c, int m, int n, const float *__restrict__ points, const int32_t *__restrict__ idx,
                              const float *__restrict__ weight, float *__restrict__ out) {
    constexpr int TS_THREADS = T;
    constexpr bool kPrefetch = MINB <= 2 && CC <= 8;  // wider tiles: enough work per index vector, and no registers to spare
    // row stride (floats): 16-byte aligned; PAD = 4 spreads the rows over the banks, PAD = 0 (CC = 4: 16 bytes per coarse
    // point) is the dense form that still fits when the coarse set is large (m <= 12800)
    constexpr int CCP = CC + PAD;
    extern __shared__ __align__(16) float tile[];  // [m][CCP]
    const int b = blockIdx.z;
    const int c0 = blockIdx.y * CC;
    const int nc = min(CC, c - c0);
    const float *f = points + ((size_t)b * c + c0) * m;
    // transposing stage: lanes run along m (coalesced 128-byte reads of four channel rows), each thread writes the four
    // channels of its point as ONE 16-byte store; row stride CCP = CC + 4 puts consecutive points 4 banks apart, so a
    // quarter warp covers all 32 banks (conflict free)
    for (int cq = 0; cq < CC / 4; ++cq)
        for (int k = threadIdx.x; k < m; k += TS_THREADS) {
            float4 v;
            v.x = 4 * cq + 0 < nc ? __ldg(f + (size_t)(4 * cq + 0) * m + k) : 0.f;
            v.y = 4 * cq + 1 < nc ? __ldg(f + (size_t)(4 * cq + 1) * m + k) : 0.f;
            v.z = 4 * cq + 2 < nc ? __ldg(f + (size_t)(4 * cq + 2) * m + k) : 0.f;
            v.w = 4 * cq + 3 < nc ? __ldg(f + (size_t)(4 * cq + 3) * m + k) : 0.f;
            *reinterpret_cast<float4 *>(tile + (size_t)k * CCP + 4 * cq) = v;
        }
    __syncthreads();
    float *ob = out + ((size_t)b * c + c0) * n;
    const int32_t *idb = idx + (size_t)b * n * 3;
    const float *wb = weight + (size_t)b * n * 3;
    if ((n & 3) == 0 && ((uintptr_t)idb & 15) == 0 && ((uintptr_t)wb & 15) == 0 && ((uintptr_t)ob & 15) == 0) {
        // four consecutive points per thread: their 12 indices / 12 weights are three 128-bit loads each, and every
        // channel's four results leave as one 128-bit streaming store
        const int n4 = n / 4;
        const int per = (n4 + gridDim.x - 1) / gridDim.x;
        const int q0 = blockIdx.x * per, q1 = min(n4, q0 + per);
        int4 kv[3], kn[3];
        float4 wv[3], wn[3];
        auto load_iw = [&](int q, int4 (&ki)[3], float4 (&wi)[3]) {
#pragma unroll
            for (int u = 0; u < 3; ++u) {
                ki[u] = make_int4(0, 0, 0, 0);
                wi[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (q < q1) {
                    ki[u] = __ldcs(reinterpret_cast<const int4 *>(idb) + (size_t)q * 3 + u);
                    wi[u] = __ldcs(reinterpret_cast<const float4 *>(wb) + (size_t)q * 3 + u);
                }
            }
        };
        if (kPrefetch) load_iw(q0 + threadIdx.x, kn, wn);
        for (int q = q0 + threadIdx.x; q < q1; q += TS_THREADS) {
            if (kPrefetch) {
#pragma unroll
                for (int u = 0; u < 3; ++u) { kv[u] = kn[u]; wv[u] = wn[u]; }
                load_iw(q + TS_THREADS, kn, wn);
            } else {
                load_iw(q, kv, wv);
            }
            int k[12];
            float w[12];
#pragma unroll
            for (int u = 0; u < 3; ++u) {
                k[4 * u] = kv[u].x; k[4 * u + 1] = kv[u].y; k[4 * u + 2] = kv[u].z; k[4 * u + 3] = kv[u].w;
                w[4 * u] = wv[u].x; w[4 * u + 1] = wv[u].y; w[4 * u + 2] = wv[u].z; w[4 * u + 3] = wv[u].w;
            }
#pragma unroll
            for (int cq = 0; cq < CC / 4; ++cq) {
                float r[4][4];  // [point][channel]
#pragma unroll
                for (int pt = 0; pt < 4; ++pt) {
                    const float4 a0 = *reinterpret_cast<const float4 *>(tile + (size_t)k[3 * pt] * CCP + 4 * cq);
                    const float4 a1 = *reinterpret_cast<const float4 *>(tile + (size_t)k[3 * pt + 1] * CCP + 4 * cq);
                    const float4 a2 = *reinterpret_cast<const float4 *>(tile + (size_t)k[3 * pt + 2] * CCP + 4 * cq);
                    const float w0 = w[3 * pt], w1 = w[3 * pt + 1], w2 = w[3 * pt + 2];
                    r[pt][0] = __fmaf_rn(w2, a2.x, __fmaf_rn(w0, a0.x, __fmul_rn(w1, a1.x)));
                    r[pt][1] = __fmaf_rn(w2, a2.y, __fmaf_rn(w0, a0.y, __fmul_rn(w1, a1.y)));
                    r[pt][2] = __fmaf_rn(w2, a2.z, __fmaf_rn(w0, a0.z, __fmul_rn(w1, a1.z)));
                    r[pt][3] = __fmaf_rn(w2, a2.w, __fmaf_rn(w0, a0.w, __fmul_rn(w1, a1.w)));
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (4 * cq + u < nc)
                        __stcs(reinterpret_cast<float4 *>(ob + (size_t)(4 * cq + u) * n) + q,
                               make_float4(r[0][u], r[1][u], r[2][u], r[3][u]));
            }
        }
        return;
    }
    const int per = (n + gridDim.x - 1) / gridDim.x;
    const int i0 = blockIdx.x * per, i1 = min(n, i0 + per);
    for (int i = i0 + threadIdx.x; i < i1; i += TS_THREADS) {
        const int32_t *id = idb + (size_t)i * 3;
        const float *w = wb + (size_t)i * 3;
        const int k0 = __ldcs(id), k1 = __ldcs(id + 1), k2 = __ldcs(id + 2);
        const float w0 = __ldcs(w), w1 = __ldcs(w + 1), w2 = __ldcs(w + 2);
        const float *r0 = tile + (size_t)k0 * CCP, *r1 = tile + (size_t)k1 * CCP, *r2 = tile + (size_t)k2 * CCP;
#pragma unroll
        for (int q = 0; q < CC / 4; ++q) {
            const float4 a0 = *reinterpret_cast<const float4 *>(r0 + 4 * q);
            const float4 a1 = *reinterpret_cast<const float4 *>(r1 + 4 * q);
            const float4 a2 = *reinterpret_cast<const float4 *>(r2 + 4 * q);
            const float v[4] = {__fmaf_rn(w2, a2.x, __fmaf_rn(w0, a0.x, __fmul_rn(w1, a1.x))),
                                __fmaf_rn(w2, a2.y, __fmaf_rn(w0, a0.y, __fmul_rn(w1, a1.y))),
                                __fmaf_rn(w2, a2.z, __fmaf_rn(w0, a0.z, __fmul_rn(w1, a1.z))),
                                __fmaf_rn(w2, a2.w, __fmaf_rn(w0, a0.w, __fmul_rn(w1, a1.w)))};
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (4 * q + u < nc) __stcs(ob + (size_t)(4 * q + u) * n + i, v[u]);
        }
    }
}

// One channel per CTA for coarse sets beyond the tiled kernel (12800 < m <= 51200): the channel row is copied to shared
// memory as it lies (coalesced), each point costs three LDS.32 and one streaming store.
__global__ void __launch_bounds__(TS_THREADS, 2)
three_interpolate_row_kernel(int c, int m, int n, const float *__restrict__ points, const int32_t *__restrict__ idx,
                             const float *__restrict__ weight, float *__restrict__ out) {
    extern __shared__ __align__(16) float tile[];  // [m]
    const int b = blockIdx.z, ch = blockIdx.y;
    const float *f = points + ((size_t)b * c + ch) * m;
    for (int k = threadIdx.x; k < m; k += TS_THREADS) tile[k] = __ldg(f + k);
    __syncthreads();
    float *ob = out + ((size_t)b * c + ch) * n;
    const int32_t *idb = idx + (size_t)b * n * 3;
    const float *wb = weight + (size_t)b * n * 3;
    const int per = (n + gridDim.x - 1) / gridDim.x;
    const int i0 = blockIdx.x * per, i1 = min(n, i0 + per);
    for (int i = i0 + threadIdx.x; i < i1; i += TS_THREADS) {
        const int32_t *id = idb + (size_t)i * 3;
        const float *w = wb + (size_t)i * 3;
        const float a0 = tile[id[0]], a1 = tile[id[1]], a2 = tile[id[2]];
        __stcs(ob + i, __fmaf_rn(w[2], a2, __fmaf_rn(w[0], a0, __fmul_rn(w[1], a1))));
    }
}

template <int CC, int PAD, int T, int MINB>
int launch_interp_smem_as(dim3 grid, size_t smem, int c, int m, int n, const float *points, const int32_t *idx, const float *weight,
                          float *out, cudaStream_t s) {
    auto kern = three_interpolate_smem_kernel<CC, PAD, T, MINB>;
    PN2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, T, smem, s>>>(c, m, n, points, idx, weight, out);
    PN2_LAUNCH_OK("three_interpolate");
    return PN2_OK;
}

template <int CC, int PAD = 4>
int launch_interp_smem(int b, int c, int m, int n, const float *points, const int32_t *idx, const float *weight, float *out,
                       cudaStream_t s) {
    const int chunks = ceil_div(c, CC);
    const size_t smem = (size_t)m * (CC + PAD) * sizeof(float);
    const int per_sm = smem <= 72 * 1024 ? 3 : (smem <= 110 * 1024 ? 2 : 1);
    // split the points of a (cloud, channel chunk) until the grid gives two full waves, but keep at least 2*m points
    // per CTA so the staging stays a small part of its work
    int nsplit = 1;
    while ((long long)nsplit * chunks * b < 2ll * per_sm * sm_count() && n / (nsplit + 1) >= 2 * m) ++nsplit;
    dim3 grid(nsplit, chunks, b);
    // one CTA per SM (large coarse sets): 512 threads, so 16 warps stream the points
    if (per_sm == 3) return launch_interp_smem_as<CC, PAD, 256, 3>(grid, smem, c, m, n, points, idx, weight, out, s);
    if (per_sm == 2) return launch_interp_smem_as<CC, PAD, 256, 2>(grid, smem, c, m, n, points, idx, weight, out, s);
    return launch_interp_smem_as<CC, PAD, 512, 1>(grid, smem, c, m, n, points, idx, weight, out, s);
}

// Lane-along-channel kernel (32 channels per tile, coarse sets up to ~1400 points).
//
// The tiled kernel above spends its shared-memory wavefronts on bank conflicts: each lane reads 16 bytes of its OWN random
// coarse row, so the 8 lanes of a quarter warp collide in the 8 four-bank groups (ncu: 5.2 M conflict wavefronts of 8.6 M,
// LSU data pipe 91 % busy while active; profiles/r1_hbm_ops_ncu_full_summary.csv).  Here the LPR = CC/4 = 8 lanes of a
// group read the 32 channels of ONE coarse row: a quarter warp reads one whole 128-byte row, conflict free whatever the
// indices are.  A group owns EIGHT CONSECUTIVE points of a 32-point granule (one per step) and keeps its 4 channels x 8
// points in registers; chunk q of a row holds the channels q, q + 8, q + 16, q + 24.  Rows are XOR-swizzled by (k >> 2) so
// that the transposing stage is conflict free as well.
// idx / weight: each warp keeps LC_DEPTH granules in flight in a cp.async ring (the 384 + 384 bytes of a granule as they lie
// in global memory); a step reads its point's six words with broadcast LDS.32.
// Stores: a 256-bit store is issued a quarter warp at a time and costs one LSU wavefront per distinct 128-byte line, so
// the accumulators are first exchanged by shuffles (same register in every lane, no selects) until the lanes of a
// quarter hold contiguous bytes of a channel row; a quarter then writes two whole lines (stores: 20 -> 8 us of the fp1 shape).
// Persistent CTAs: the (cloud, channel tile, granule) space is cut into gridDim.x contiguous ranges, so a CTA stages at
// most two tiles more than it has whole (cloud, tile) pairs and there is no partial last wave.
// Time split at the fp1 shape (45 us), measured by switching the stores or the row reads off: stores 8 us, row reads 6 us,
// the rest (stage 2 x 128 KB per CTA, ring, arithmetic, shuffles) 31 us.  768- and 1024-thread CTAs (80 / 64 registers)
// were slower: 59.4 / 65.5 us against 49.2 at 512 threads (before the shuffle exchange; profiles/README.md).

// Transposing stage: tile4[k][q ^ ((k >> 2) & (LPR - 1))] = channels q + LPR * {0,1,2,3} of coarse point k (zero beyond nc).
// Vector form: an item = four consecutive points of four channel rows (four coalesced 128-bit loads) -> four swizzled
// 16-byte chunks; a thread issues the loads of four items before the first store, so 16 loads are in flight per thread.
template <int LPR, int T>
__device__ __forceinline__ void lac_stage_tile(float4 *tile4, const float *__restrict__ f, int m, int nc, int tid) {
    if ((m & 3) == 0 && ((uintptr_t)f & 15) == 0) {
        const int m4 = m >> 2;
        const int items = LPR * m4;
        constexpr int NB = 4;  // items per thread and batch
        for (int base = 0; base < items; base += NB * T) {
            float4 r[NB][4];
            int cqs[NB], is[NB];
#pragma unroll
            for (int u = 0; u < NB; ++u) {
                const int it = base + u * T + tid;
                const int cq = it / m4, i = it - cq * m4;
                cqs[u] = cq;
                is[u] = i;
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    r[u][e] = it < items && cq + LPR * e < nc ? __ldg(reinterpret_cast<const float4 *>(f + (size_t)(cq + LPR * e) * m) + i)
                                                              : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < NB; ++u) {
                if (base + u * T + tid >= items) continue;
                float4 *d = tile4 + (size_t)(4 * is[u]) * LPR + (cqs[u] ^ (is[u] & (LPR - 1)));
                d[0] = make_float4(r[u][0].x, r[u][1].x, r[u][2].x, r[u][3].x);
                d[LPR] = make_float4(r[u][0].y, r[u][1].y, r[u][2].y, r[u][3].y);
                d[2 * LPR] = make_float4(r[u][0].z, r[u][1].z, r[u][2].z, r[u][3].z);
                d[3 * LPR] = make_float4(r[u][0].w, r[u][1].w, r[u][2].w, r[u][3].w);
            }
        }
    } else {
        for (int cq = 0; cq < LPR; ++cq)
            for (int k = tid; k < m; k += T) {
                float4 v;
                v.x = cq < nc ? __ldg(f + (size_t)cq * m + k) : 0.f;
                v.y = cq + LPR < nc ? __ldg(f + (size_t)(cq + LPR) * m + k) : 0.f;
                v.z = cq + 2 * LPR < nc ? __ldg(f + (size_t)(cq + 2 * LPR) * m + k) : 0.f;
                v.w = cq + 3 * LPR < nc ? __ldg(f + (size_t)(cq + 3 * LPR) * m + k) : 0.f;
                tile4[(size_t)k * LPR + (cq ^ ((k >> 2) & (LPR - 1)))] = v;
            }
    }
}

constexpr int LC_DEPTH = 4;  // granules of idx / weight in flight per warp (cp.async ring)

template <int CC, int T>
__global__ void __launch_bounds__(T, T <= 256 ? 2 : 1)
three_interpolate_lac_kernel(int c, int m, int n, int chunks, int gpp, long long total_gran,
                             const float *__restrict__ points, const int32_t *__restrict__ idx,
                             const float *__restrict__ weight, float *__restrict__ out) {
    constexpr int LPR = CC / 4;    // lanes per coarse row = lanes per group
    constexpr int PPI = 32 / LPR;  // groups per warp
    constexpr int GRAN = LC_GRAN;  // points per warp granule
    constexpr int RUNS = GRAN / (8 * PPI);  // eight-point runs per group and granule
    constexpr int WARPS = T / 32;
    constexpr int SLOT_WORDS = GRAN * 6;  // 3 indices then 3 weights per point, as they lie in global memory
    extern __shared__ __align__(16) float4 lac_smem[];
    float4 *tile4 = lac_smem;  // [m][LPR]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int j = lane % LPR, g = lane / LPR;
    int32_t *ring = reinterpret_cast<int32_t *>(lac_smem + (size_t)m * LPR) + (size_t)warp * LC_DEPTH * SLOT_WORDS;
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring);
    const char *tile_bytes = reinterpret_cast<const char *>(tile4);
    const int j16 = j << 4;
    // byte offset of a lane's chunk of coarse row k (swizzle included)
    auto row_off = [&](int k) { return (((k * LPR) | ((k >> 2) & (LPR - 1))) << 4) ^ j16; };

    long long gq = total_gran * blockIdx.x / gridDim.x;
    const long long gq_end = total_gran * (blockIdx.x + 1) / gridDim.x;
    while (gq < gq_end) {
        const int pair = (int)(gq / gpp);
        const int gi0 = (int)(gq - (long long)pair * gpp);
        const long long seg_end = min(gq_end, (long long)(pair + 1) * gpp);
        const int gi1 = gi0 + (int)(seg_end - gq);
        gq = seg_end;
        const int bb = pair / chunks, c0 = (pair - bb * chunks) * CC;
        const int nc = min(CC, c - c0);
        const int32_t *idb = idx + (size_t)bb * n * 3;
        const float *wb = weight + (size_t)bb * n * 3;
        float *ob = out + ((size_t)bb * c + c0) * n;
        // granule gi -> ring slot: 12 * points bytes of idx and of weight, in 16-byte pieces (n % 8 == 0: whole pieces)
        auto issue = [&](int gi, int slot) {
            if (gi < gi1) {
                const int p0 = gi * GRAN;
                const int pieces = min(GRAN, n - p0) * 3 / 4;
                const uint32_t dst = ring_s + (uint32_t)slot * SLOT_WORDS * 4;
                for (int q = lane; q < pieces; q += 32) {
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + q * 16), "l"(idb + (size_t)p0 * 3 + q * 4) : "memory");
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + GRAN * 12 + q * 16), "l"(wb + (size_t)p0 * 3 + q * 4)
                                 : "memory");
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        __syncwarp();  // the warp has consumed every slot of the previous segment
#pragma unroll
        for (int d = 0; d < LC_DEPTH - 1; ++d) issue(gi0 + warp + d * WARPS, d);  // in flight during the stage
        __syncthreads();  // every warp is done with the previous tile
        lac_stage_tile<LPR, T>(tile4, points + ((size_t)bb * c + c0) * m, m, nc, tid);
        __syncthreads();
        int slot = 0;
        for (int gi = gi0 + warp; gi < gi1; gi += WARPS) {
            __syncwarp();  // the slot refilled below was read in the previous iteration
            issue(gi + (LC_DEPTH - 1) * WARPS, slot == 0 ? LC_DEPTH - 1 : slot - 1);
            asm volatile("cp.async.wait_group %0;" ::"n"(LC_DEPTH - 1) : "memory");
            __syncwarp();  // every lane's pieces of this granule have landed
            const int32_t *ri = ring + slot * SLOT_WORDS;
            const float *rw = reinterpret_cast<const float *>(ri + GRAN * 3);
            slot = slot == LC_DEPTH - 1 ? 0 : slot + 1;
#pragma unroll
            for (int run = 0; run < RUNS; ++run) {
                // the group's eight points, within the granule (the PPI groups of a warp own consecutive runs)
                const int q0 = 8 * PPI * run + 8 * g;
                const int pw = gi * GRAN + 8 * PPI * run;  // the warp's 8 * PPI points of this run
                float acc[4][8];
#pragma unroll
                for (int u = 0; u < 4; ++u)
#pragma unroll
                    for (int s = 0; s < 8; ++s) acc[u][s] = 0.f;
                if (pw + 8 * g < n) {  // n % 8 == 0: a group's run is whole or absent (its ring words may be stale)
#pragma unroll
                    for (int s = 0; s < 8; ++s) {
                        const int k0 = ri[3 * (q0 + s)], k1 = ri[3 * (q0 + s) + 1], k2 = ri[3 * (q0 + s) + 2];
                        const float w0 = rw[3 * (q0 + s)], w1 = rw[3 * (q0 + s) + 1], w2 = rw[3 * (q0 + s) + 2];
                        const float4 a0 = *reinterpret_cast<const float4 *>(tile_bytes + row_off(k0));
                        const float4 a1 = *reinterpret_cast<const float4 *>(tile_bytes + row_off(k1));
                        const float4 a2 = *reinterpret_cast<const float4 *>(tile_bytes + row_off(k2));
                        // the reference's contraction (K8): fma(w2, f2, fma(w0, f0, rn(w1 * f1)))
                        acc[0][s] = __fmaf_rn(w2, a2.x, __fmaf_rn(w0, a0.x, __fmul_rn(w1, a1.x)));
                        acc[1][s] = __fmaf_rn(w2, a2.y, __fmaf_rn(w0, a0.y, __fmul_rn(w1, a1.y)));
                        acc[2][s] = __fmaf_rn(w2, a2.z, __fmaf_rn(w0, a0.z, __fmul_rn(w1, a1.z)));
                        acc[3][s] = __fmaf_rn(w2, a2.w, __fmaf_rn(w0, a0.w, __fmul_rn(w1, a1.w)));
                    }
                }
                // Element u of lane (g, j) is channel j + LPR * u of the points 8 g .. 8 g + 7.  A 256-bit store is issued a
                // quarter warp at a time, so the lanes of a QUARTER have to cover contiguous bytes: for store u, lane
                // (Q, l) takes over channel LPR * u + 2 Q + (l >> 2), points 8 (l & 3) .. + 7, from lane (g = l & 3,
                // j = 2 Q + (l >> 2)) -- eight shuffles of the same register in every lane, no selects; a quarter then
                // writes two whole 128-byte lines.
                static_assert(CC == 32, "the store transpose is written for eight lanes per row");
                const int l = lane & 7, Q = lane >> 3;
                const int src = (l & 3) * 8 + 2 * Q + (l >> 2);
                const int prun = pw + 8 * (l & 3);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    float v[8];
#pragma unroll
                    for (int s = 0; s < 8; ++s) v[s] = __shfl_sync(0xffffffffu, acc[u][s], src);
                    const int ch = LPR * u + 2 * Q + (l >> 2);
                    if (ch < nc && prun < n)
                        asm volatile("st.global.cs.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(ob + (size_t)ch * n + prun), "f"(v[0]),
                                     "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                                     : "memory");
                }
            }
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

int g_interp_mode = 0;  // developer knob (pn2_debug_set_interp_mode): 0 auto, 1 tiled kernels only, 32 the lane-along-channel
                        // kernel wherever it applies (32 | 256: 256-thread CTAs, two per SM); any other value = auto

inline size_t lac_smem_bytes(int m, int cc, int threads) {
    return (size_t)m * cc * 4 + (size_t)(threads / 32) * LC_DEPTH * LC_GRAN * 24;
}
inline bool lac_fits(int m, int cc, int threads) { return (threads <= 256 ? 2 : 1) * (lac_smem_bytes(m, cc, threads) + 1024) <= 233472; }

template <int CC, int T>
int launch_interp_lac(int b, int c, int m, int n, const float *points, const int32_t *idx, const float *weight, float *out,
                      cudaStream_t s) {
    const int chunks = ceil_div(c, CC);
    const int gpp = ceil_div(n, LC_GRAN);
    const long long total = (long long)b * chunks * gpp;
    const size_t smem = lac_smem_bytes(m, CC, T);
    const int grid = (int)std::min<long long>((long long)(T <= 256 ? 2 : 1) * sm_count(), std::max<long long>(1, total / (T / 32)));
    PN2_CUDA(cudaFuncSetAttribute(three_interpolate_lac_kernel<CC, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    three_interpolate_lac_kernel<CC, T><<<grid, T, smem, s>>>(c, m, n, chunks, gpp, total, points, idx, weight, out);
    PN2_LAUNCH_OK("three_interpolate");
    return PN2_OK;
}

// grad_points[b,c,idx_j] += grad_out[b,c,i] * w_j   (interpolate_gpu.cu:120-142)
__global__ void __launch_bounds__(TI_THREADS)
three_interpolate_grad_kernel(int c, int n, int m, const float *__restrict__ grad_out, const int32_t *__restrict__ idx,
                              const float *__restrict__ weight, float *__restrict__ grad_points) {
    const int i = blockIdx.x * TI_THREADS + threadIdx.x;
    if (i >= n) return;
    const int b = blockIdx.z;
    const int c0 = blockIdx.y * TI_CH;
    const int32_t *id = idx + ((size_t)b * n + i) * 3;
    const float *w = weight + ((size_t)b * n + i) * 3;
    const int i0 = id[0], i1 = id[1], i2 = id[2];
    const float w0 = w[0], w1 = w[1], w2 = w[2];
    const float *g = grad_out + ((size_t)b * c + c0) * n + i;
    float *gp = grad_points + ((size_t)b * c + c0) * m;
    const int cc = min(TI_CH, c - c0);
#pragma unroll
    for (int k = 0; k < TI_CH; ++k)
        if (k < cc) {
            const float go = __ldcs(g + (size_t)k * n);
            atomicAdd(gp + (size_t)k * m + i0, __fmul_rn(go, w0));
            atomicAdd(gp + (size_t)k * m + i1, __fmul_rn(go, w1));
            atomicAdd(gp + (size_t)k * m + i2, __fmul_rn(go, w2));
        }
}

}  // namespace
}  // namespace pn2

extern "C" void pn2_debug_set_interp_mode(int mode) { pn2::g_interp_mode = mode; }

extern "C" int pn2_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2, int32_t *idx,
                            void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && n >= 0 && m >= 0, "three_nn: bad dims b=%d n=%d m=%d", b, n, m);
    if (b == 0 || n == 0) return PN2_OK;
    PN2_REQUIRE(unknown && dist2 && idx && (known || m == 0), "three_nn: null pointer");
    PN2_REQUIRE(b <= 65535, "three_nn: b exceeds the grid limit");
    dim3 grid(ceil_div(n, NN_THREADS), b);
    three_nn_kernel<<<grid, NN_THREADS, 0, (cudaStream_t)stream>>>(n, m, unknown, known, dist2, idx);
    PN2_LAUNCH_OK("three_nn");
    return PN2_OK;
}

extern "C" int pn2_three_nn_weights(int b, int n, int m, const float *unknown, const float *known, int32_t *idx,
                                    float *weight, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && n >= 0 && m >= 0, "three_nn_weights: bad dims b=%d n=%d m=%d", b, n, m);
    if (b == 0 || n == 0) return PN2_OK;
    PN2_REQUIRE(unknown && weight && idx && (known || m == 0), "three_nn_weights: null pointer");
    PN2_REQUIRE(b <= 65535, "three_nn_weights: b exceeds the grid limit");
    dim3 grid(ceil_div(n, NN_THREADS), b);
    three_nn_weights_kernel<<<grid, NN_THREADS, 0, (cudaStream_t)stream>>>(n, m, unknown, known, idx, weight);
    PN2_LAUNCH_OK("three_nn_weights");
    return PN2_OK;
}

extern "C" int pn2_three_interpolate(int b, int c, int m, int n, const float *points, const int32_t *idx,
                                     const float *weight, float *out, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && c >= 0 && m >= 1 && n >= 0, "three_interpolate: bad dims b=%d c=%d m=%d n=%d", b, c, m, n);
    if (b == 0 || c == 0 || n == 0) return PN2_OK;
    PN2_REQUIRE(points && idx && weight && out, "three_interpolate: null pointer");
    PN2_REQUIRE(b <= 65535 && ceil_div(c, TI_CH) <= 65535, "three_interpolate: b or c exceeds the grid limits");
    if (g_interp_mode != 1 && (n & 7) == 0 && ((uintptr_t)out & 31) == 0 && (((uintptr_t)idx | (uintptr_t)weight) & 15) == 0) {
        // lane-along-channel kernel (three_interpolate_lac_kernel): 256-bit stores need 32-byte aligned rows, the cp.async ring
        // 16-byte aligned idx / weight.  Measured (scripts/interp_sweep.py, profiles/r1_interp_sweep_lac.jsonl): fp1 shape (b 32,
        // c 128, m 1024, n 8192) 57 -> 45 us = 53 % of HBM, 20-40 % faster at m <= 256; no gain with too little work per SM.
        cudaStream_t st = (cudaStream_t)stream;
        const bool forced = g_interp_mode == 32 || g_interp_mode == (32 | 256);
        const int threads = forced ? (g_interp_mode == 32 ? 512 : 256) : (lac_fits(m, 32, 256) ? 256 : 512);
        const long long granules = (long long)b * ceil_div(c, 32) * ceil_div(n, LC_GRAN);
        const bool wanted = forced || (c >= 32 && n >= 2 * m && (m <= 512 || granules >= 16ll * sm_count()));
        if (wanted && lac_fits(m, 32, threads)) {
            if (threads == 512) return launch_interp_lac<32, 512>(b, c, m, n, points, idx, weight, out, st);
            return launch_interp_lac<32, 256>(b, c, m, n, points, idx, weight, out, st);
        }
    }
    // upsampling (n >> m) with a coarse set that fits in shared memory: stage it (three_interpolate_smem_kernel)
    if (n >= 2 * m && (long long)b * c >= 64) {
        // prefer a tile that lets two CTAs share an SM (one stages while the other streams), else the widest that fits
        const long long three = 72 * 1024 / 4, two = 110 * 1024 / 4, one = 200 * 1024 / 4;  // floats
        cudaStream_t st = (cudaStream_t)stream;
        if ((long long)m * 20 <= three && c >= 16) return launch_interp_smem<16>(b, c, m, n, points, idx, weight, out, st);
        if ((long long)m * 12 <= three) return launch_interp_smem<8>(b, c, m, n, points, idx, weight, out, st);
        if ((long long)m * 36 <= two && c >= 32) return launch_interp_smem<32>(b, c, m, n, points, idx, weight, out, st);
        if ((long long)m * 20 <= two && c >= 16) return launch_interp_smem<16>(b, c, m, n, points, idx, weight, out, st);
        if ((long long)m * 12 <= two) return launch_interp_smem<8>(b, c, m, n, points, idx, weight, out, st);
        if ((long long)m * 36 <= one && c >= 32) return launch_interp_smem<32>(b, c, m, n, points, idx, weight, out, st);
        if ((long long)m * 20 <= one && c >= 16) return launch_interp_smem<16>(b, c, m, n, points, idx, weight, out, st);
        if ((long long)m * 12 <= one) return launch_interp_smem<8>(b, c, m, n, points, idx, weight, out, st);
        // large coarse sets: dense 4-channel tiles (m <= 12800), then one channel row per CTA (m <= 51200)
        if ((long long)m * 4 <= one) return launch_interp_smem<4, 0>(b, c, m, n, points, idx, weight, out, st);
        if ((long long)m <= one && c <= 65535) {
            const size_t smem = (size_t)m * sizeof(float);
            const int per_sm = smem <= 110 * 1024 ? 2 : 1;
            int nsplit = 1;
            while ((long long)nsplit * c * b < 2ll * per_sm * sm_count() && n / (nsplit + 1) >= 2 * m) ++nsplit;
            PN2_CUDA(cudaFuncSetAttribute(three_interpolate_row_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            three_interpolate_row_kernel<<<dim3(nsplit, c, b), TS_THREADS, smem, st>>>(c, m, n, points, idx, weight, out);
            PN2_LAUNCH_OK("three_interpolate");
            return PN2_OK;
        }
    }
    dim3 grid(ceil_div(n, TI_THREADS), ceil_div(c, TI_CH), b);
    three_interpolate_kernel<<<grid, TI_THREADS, 0, (cudaStream_t)stream>>>(c, m, n, points, idx, weight, out);
    PN2_LAUNCH_OK("three_interpolate");
    return PN2_OK;
}

extern "C" int pn2_three_interpolate_grad(int b, int c, int n, int m, const float *grad_out, const int32_t *idx,
                                          const float *weight, float *grad_points, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && c >= 0 && m >= 1 && n >= 0, "three_interpolate_grad: bad dims b=%d c=%d n=%d m=%d", b, c, n, m);
    if (b == 0 || c == 0 || n == 0) return PN2_OK;
    PN2_REQUIRE(grad_out && idx && weight && grad_points, "three_interpolate_grad: null pointer");
    PN2_REQUIRE(b <= 65535 && ceil_div(c, TI_CH) <= 65535, "three_interpolate_grad: b or c exceeds the grid limits");
    dim3 grid(ceil_div(n, TI_THREADS), ceil_div(c, TI_CH), b);
    three_interpolate_grad_kernel<<<grid, TI_THREADS, 0, (cudaStream_t)stream>>>(c, n, m, grad_out, idx, weight, grad_points);
    PN2_LAUNCH_OK("three_interpolate_grad");
    return PN2_OK;
}
