// train_mlp.cu -- the shared-MLP layer of the SA / FP blocks in TRAINING mode (BatchNorm with batch statistics, or with
// its running statistics when torch's rule says so: see train_bn_running_kernel), fp32.
//
// Replaces, per layer of model/pointnet_util.py:105-107 / 162-165 / 218-220 run under autograd,
//     Conv2d/Conv1d 1x1 (cuDNN fprop, dgrad, wgrad) + BatchNorm (forward statistics, normalise, backward reductions,
//     backward elementwise) + ReLU (forward, backward mask)
// i.e. nine library / elementwise passes over (rows x channels) activations, by four kernels on channel-last row
// matrices (a row = one (centroid, sample) pair or one point):
//
//   forward      z = act_in(x) W^T + b          and, in the same pass, the per-channel sum / sum of squares of z
//                (act_in = the PREVIOUS layer's BatchNorm + ReLU applied while the operand is loaded: normalised
//                activations are never written; only the pre-BatchNorm z of every layer is kept for the backward)
//   bwd reduce   S1 = sum_r dy, S2 = sum_r dy z  with dy = g [scale z + shift > 0]   (BatchNorm backward needs both)
//   bwd input    g_in = dz W                    with dz = ca dy + cb + cc z built while the operand is loaded
//   bwd weight   dW += dz^T act_in(x)           (row range per CTA, fp32 atomics into dW like the reference's backwards)
//
// BatchNorm algebra (training mode, biased variance, eps as torch): zhat = (z - mu) rstd, y = gamma zhat + beta,
// a = relu(y);  dL/dz = gamma rstd (dy - mean(dy) - zhat mean(dy zhat)) = ca dy + cb + cc z per channel with
//   ca = gamma rstd,  cc = -gamma rstd^3 (S2 - mu S1) / R,  cb = -ca S1 / R - cc mu;  dgamma = rstd (S2 - mu S1), dbeta = S1.
// The host side (pn2_b200/train_mlp.py) turns the sums into these coefficients (tiny per-channel tensors).
//
// All four are the same register-tiled SIMT GEMM (128 x NT output tile, 256 threads, k-chunks of 16 double buffered in
// shared memory, FFMA): the 1e-5 parity path.  Widths are arbitrary (16 .. 1536 in the MSG stack).
#include <type_traits>

#include "common.cuh"

namespace pn2 {
namespace {

constexpr int TG_THREADS = 256;
constexpr int TG_KC = 16;
constexpr int TG_M = 128;

template <int NT, int MT = TG_M>
struct TileShape {
    static constexpr int TX = NT / 4;             // threads along n (4 columns each)
    static constexpr int TY = TG_THREADS / TX;    // threads along m
    static constexpr int TM = MT / TY;            // rows per thread (1, 2 or a multiple of 4)
    static constexpr int AS = MT + 4, BS = NT + 4;
    static constexpr size_t smem_floats = 2 * TG_KC * (AS + BS);
    static_assert(TM >= 1 && (TM < 4 || TM % 4 == 0), "tile shape");
};

// acc[TM][4] += As[k][ty*TM .. ] * Bs[k][tx*4 ..] over one staged k-chunk
template <int NT, int MT = TG_M>
__device__ __forceinline__ void mma_chunk(const float *__restrict__ As, const float *__restrict__ Bs, float (&acc)[TileShape<NT, MT>::TM][4],
                                          int ty, int tx) {
    using S = TileShape<NT, MT>;
#pragma unroll
    for (int kk = 0; kk < TG_KC; ++kk) {
        float a[S::TM], b[4];
        if constexpr (S::TM >= 4) {
#pragma unroll
            for (int i = 0; i < S::TM; i += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(As + kk * S::AS + ty * S::TM + i);
                a[i] = v.x; a[i + 1] = v.y; a[i + 2] = v.z; a[i + 3] = v.w;
            }
        } else {
#pragma unroll
            for (int i = 0; i < S::TM; ++i) a[i] = As[kk * S::AS + ty * S::TM + i];
        }
        const float4 w = *reinterpret_cast<const float4 *>(Bs + kk * S::BS + tx * 4);
        b[0] = w.x; b[1] = w.y; b[2] = w.z; b[3] = w.w;
#pragma unroll
        for (int i = 0; i < S::TM; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
}

// ---- operand loaders: 4 consecutive k of one row (k-contiguous operands) -------------------------------------------------
struct ActIn {  // x with the previous layer's BatchNorm + ReLU folded in (scale == nullptr: identity)
    const float *x, *scale, *shift;
    long long rows;
    int c;
    __device__ __forceinline__ float one(long long r, int k) const {
        if (r >= rows || k >= c) return 0.f;
        float v = __ldg(x + r * c + k);
        if (scale) v = fmaxf(fmaf(v, __ldg(scale + k), __ldg(shift + k)), 0.f);
        return v;
    }
    // The load of an operand chunk is split in two: raw() issues the long-latency loads of the row data and nothing that
    // depends on them, finish() applies the per-channel transform.  The GEMM loops call raw() for chunk c + 1, multiply chunk
    // c, and only then finish() + store: with the transform inside the load the first dependent FFMA stalled the warp on the
    // loads (in-order issue) BEFORE the multiplies of the current chunk, so no load latency was ever hidden (ncu: the
    // transform's FFMA / FSEL carry the long-scoreboard samples, FMA pipe 10-13 % busy).
    struct Raw {
        float4 v;
    };
    __device__ __forceinline__ bool fast(long long r, int k) const { return r < rows && k + 3 < c && (c & 3) == 0; }
    __device__ __forceinline__ Raw raw(long long r, int k) const {  // k % 4 == 0
        Raw q;
        if (fast(r, k)) q.v = __ldg(reinterpret_cast<const float4 *>(x + r * c + k));
        else q.v = make_float4(one(r, k), one(r, k + 1), one(r, k + 2), one(r, k + 3));  // ragged edge: final values at once
        return q;
    }
    __device__ __forceinline__ float4 finish(const Raw &q, long long r, int k) const {
        float4 v = q.v;
        if (scale && fast(r, k)) {
            const float4 s = __ldg(reinterpret_cast<const float4 *>(scale + k)), t = __ldg(reinterpret_cast<const float4 *>(shift + k));
            v.x = fmaxf(fmaf(v.x, s.x, t.x), 0.f); v.y = fmaxf(fmaf(v.y, s.y, t.y), 0.f);
            v.z = fmaxf(fmaf(v.z, s.z, t.z), 0.f); v.w = fmaxf(fmaf(v.w, s.w, t.w), 0.f);
        }
        return v;
    }
};

struct DzIn {  // dz = ca * g * [scale z + shift > 0] + cb + cc * z, built from g and z
    const float *g, *z, *scale, *shift, *ca, *cb, *cc;
    long long rows;
    int c;
    __device__ __forceinline__ float one(long long r, int k) const {
        if (r >= rows || k >= c) return 0.f;
        const float zz = __ldg(z + r * c + k), gg = __ldg(g + r * c + k);
        const float dy = fmaf(zz, __ldg(scale + k), __ldg(shift + k)) > 0.f ? gg : 0.f;
        return fmaf(__ldg(cc + k), zz, fmaf(__ldg(ca + k), dy, __ldg(cb + k)));
    }
    struct Raw {
        float4 z, g;  // ragged edge: z holds the final values
    };
    __device__ __forceinline__ bool fast(long long r, int k) const { return r < rows && k + 3 < c && (c & 3) == 0; }
    __device__ __forceinline__ Raw raw(long long r, int k) const {
        Raw q;
        if (fast(r, k)) {
            q.z = __ldg(reinterpret_cast<const float4 *>(z + r * c + k));
            q.g = __ldg(reinterpret_cast<const float4 *>(g + r * c + k));
        } else {
            q.z = make_float4(one(r, k), one(r, k + 1), one(r, k + 2), one(r, k + 3));
            q.g = q.z;
        }
        return q;
    }
    __device__ __forceinline__ float4 finish(const Raw &q, long long r, int k) const {
        if (!fast(r, k)) return q.z;
        const float4 zz = q.z, gg = q.g;
        const float4 s = __ldg(reinterpret_cast<const float4 *>(scale + k)), t = __ldg(reinterpret_cast<const float4 *>(shift + k));
        const float4 a = __ldg(reinterpret_cast<const float4 *>(ca + k)), b = __ldg(reinterpret_cast<const float4 *>(cb + k));
        const float4 cq = __ldg(reinterpret_cast<const float4 *>(cc + k));
        float4 o;
        o.x = fmaf(cq.x, zz.x, fmaf(a.x, fmaf(zz.x, s.x, t.x) > 0.f ? gg.x : 0.f, b.x));
        o.y = fmaf(cq.y, zz.y, fmaf(a.y, fmaf(zz.y, s.y, t.y) > 0.f ? gg.y : 0.f, b.y));
        o.z = fmaf(cq.z, zz.z, fmaf(a.z, fmaf(zz.z, s.z, t.z) > 0.f ? gg.z : 0.f, b.z));
        o.w = fmaf(cq.w, zz.w, fmaf(a.w, fmaf(zz.w, s.w, t.w) > 0.f ? gg.w : 0.f, b.w));
        return o;
    }
};

// First-layer operands of a whole SA scale / FP block (pn2_rows), read where they lie: the grouped / interpolated row
// matrix of the reference's composition is never materialised.  Same raw() / finish() split as ActIn.
struct GroupIn {  // row (bb*m + s)*k + j: xyz columns [xc0, xc0 + 3) = xyz[p] - new_xyz[s], feature columns [fc0, fc0 + d) = feat[p]
    const float *xyz, *new_xyz, *feat;
    const int32_t *idx;
    long long rows;
    int c, n, m, k, d, xc0, fc0;
    // feature rows are float4-loadable (d % 4 == 0, 16-byte aligned).  Only PN2_ORDER_FEAT_FIRST (MSG, fc0 = 0) puts a
    // 4-aligned k-chunk on 4-aligned feature columns; with xyz first (SSG, fc0 = 3) every feature element is a scalar load,
    // as the materialised (rows, 3 + d) operand of the composition was
    bool vec;
    struct Raw {
        float4 v, ctr;  // finish() = v - ctr (ctr = 0 outside the xyz columns)
    };
    __device__ __forceinline__ Raw raw(long long r, int kc) const {
        Raw q;
        q.v = q.ctr = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r >= rows) return q;
        const int row = (int)r, bs = row / k;
        const long long pt = (long long)(bs / m) * n + __ldg(idx + row);
        if (vec && kc >= fc0 && kc + 3 < fc0 + d && ((kc - fc0) & 3) == 0) {
            q.v = __ldg(reinterpret_cast<const float4 *>(feat + pt * d + (kc - fc0)));
            return q;
        }
        float v[4], t[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int col = kc + e;
            v[e] = t[e] = 0.f;
            if (col >= c) continue;
            if (col >= xc0 && col < xc0 + 3) {
                v[e] = __ldg(xyz + pt * 3 + (col - xc0));
                t[e] = __ldg(new_xyz + (long long)bs * 3 + (col - xc0));
            } else {
                v[e] = __ldg(feat + pt * d + (col - fc0));
            }
        }
        q.v = make_float4(v[0], v[1], v[2], v[3]);
        q.ctr = make_float4(t[0], t[1], t[2], t[3]);
        return q;
    }
    __device__ __forceinline__ float4 finish(const Raw &q, long long, int) const {
        // the centring of sample_and_group: one fp32 subtraction (x - 0 == x bit for bit in the feature columns)
        return make_float4(__fsub_rn(q.v.x, q.ctr.x), __fsub_rn(q.v.y, q.ctr.y), __fsub_rn(q.v.z, q.ctr.z), __fsub_rn(q.v.w, q.ctr.w));
    }
};

struct InterpIn {  // row bb*n + i: columns [0, ds) = skip[i], [ds, ds + d) = three_interpolate(feat, idx[i], weight[i])
    const float *skip, *feat, *weight;
    const int32_t *idx;  // NULL: m == 1, the one coarse row repeated
    long long rows;
    int c, n, m, d, ds;
    bool vec_skip, vec_feat;  // float4-loadable rows
    struct Raw {
        float4 a0, a1, a2;  // a1 holds the final value of skip / repeated / out-of-range columns
    };
    __device__ __forceinline__ bool direct(long long r, int col) const { return r >= rows || col >= c || col < ds || !idx; }
    __device__ __forceinline__ Raw raw(long long r, int kc) const {
        Raw q;
        q.a0 = q.a1 = q.a2 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r >= rows) return q;
        const long long cloud = r / n;
        int i0 = 0, i1 = 0, i2 = 0;
        if (idx && kc + 3 >= ds) {
            i0 = __ldg(idx + r * 3); i1 = __ldg(idx + r * 3 + 1); i2 = __ldg(idx + r * 3 + 2);
        }
        const float *f0 = feat + (cloud * m + i0) * d - ds, *f1 = feat + (cloud * m + i1) * d - ds, *f2 = feat + (cloud * m + i2) * d - ds;
        if (vec_skip && kc + 3 < ds) {
            q.a1 = __ldg(reinterpret_cast<const float4 *>(skip + r * ds + kc));
            return q;
        }
        if (vec_feat && kc >= ds && kc + 3 < c && ((kc - ds) & 3) == 0) {
            q.a1 = __ldg(reinterpret_cast<const float4 *>(f1 + kc));
            if (idx) {
                q.a0 = __ldg(reinterpret_cast<const float4 *>(f0 + kc));
                q.a2 = __ldg(reinterpret_cast<const float4 *>(f2 + kc));
            }
            return q;
        }
        float a0[4], a1[4], a2[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int col = kc + e;
            a0[e] = a1[e] = a2[e] = 0.f;
            if (col >= c) continue;
            if (col < ds) {
                a1[e] = __ldg(skip + r * ds + col);
            } else {
                a1[e] = __ldg(f1 + col);
                if (idx) { a0[e] = __ldg(f0 + col); a2[e] = __ldg(f2 + col); }
            }
        }
        q.a0 = make_float4(a0[0], a0[1], a0[2], a0[3]);
        q.a1 = make_float4(a1[0], a1[1], a1[2], a1[3]);
        q.a2 = make_float4(a2[0], a2[1], a2[2], a2[3]);
        return q;
    }
    // the weights are read here, not in raw(): the row's idx load above already brought their cache line on chip, and
    // three more live registers per staged operand made the widest weight-gradient tile spill
    __device__ __forceinline__ float one(float w0, float w1, float w2, float a0, float a1, float a2, long long r, int col) const {
        // three_interpolate's order (interpolate.cu)
        return direct(r, col) ? a1 : __fmaf_rn(w2, a2, __fmaf_rn(w0, a0, __fmul_rn(w1, a1)));
    }
    __device__ __forceinline__ float4 finish(const Raw &q, long long r, int kc) const {
        float w0 = 0.f, w1 = 0.f, w2 = 0.f;
        if (r < rows && idx && kc + 3 >= ds) {
            w0 = __ldg(weight + r * 3); w1 = __ldg(weight + r * 3 + 1); w2 = __ldg(weight + r * 3 + 2);
        }
        return make_float4(one(w0, w1, w2, q.a0.x, q.a1.x, q.a2.x, r, kc), one(w0, w1, w2, q.a0.y, q.a1.y, q.a2.y, r, kc + 1),
                           one(w0, w1, w2, q.a0.z, q.a1.z, q.a2.z, r, kc + 2), one(w0, w1, w2, q.a0.w, q.a1.w, q.a2.w, r, kc + 3));
    }
};

struct AllIn {  // row r = bb*n + i of a group_all SA layer: columns [0, 3) = xyz[r], [3, 3 + d) = feat[r] (not centred)
    const float *xyz, *feat;
    long long rows;
    int c, d;
    // the feature columns start at 3, so no 4-aligned k-chunk lies on 4-aligned feature columns: scalar loads, as for
    // the materialised (rows, 3 + d) operand of the composition
    struct Raw {
        float4 v;
    };
    __device__ __forceinline__ Raw raw(long long r, int kc) const {
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int col = kc + e;
            v[e] = r >= rows || col >= c ? 0.f : (col < 3 ? __ldg(xyz + r * 3 + col) : __ldg(feat + r * d + (col - 3)));
        }
        Raw q;
        q.v = make_float4(v[0], v[1], v[2], v[3]);
        return q;
    }
    __device__ __forceinline__ float4 finish(const Raw &q, long long, int) const { return q.v; }
};

struct WeightIn {  // w (n_total, k_total) row-major: 4 consecutive k of output column n
    const float *w;
    int n_total, k_total;
    __device__ __forceinline__ float4 four(int n, int k) const {
        if (n < n_total && k + 3 < k_total && (k_total & 3) == 0) return __ldg(reinterpret_cast<const float4 *>(w + (size_t)n * k_total + k));
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = (n < n_total && k + e < k_total) ? __ldg(w + (size_t)n * k_total + k + e) : 0.f;
        return make_float4(v[0], v[1], v[2], v[3]);
    }
};

// C[128 x NT] = A[rows m0.., K] * B[n0.., K]^T with k-contiguous operands (forward and input-gradient products).
template <int NT, class LA>
__device__ __forceinline__ void gemm_rows(const LA &la, const WeightIn &lb, long long m0, int n0, int K, float *smem,
                                          float (&acc)[TileShape<NT>::TM][4]) {
    using S = TileShape<NT>;
    float *As = smem, *Bs = smem + 2 * TG_KC * S::AS;
    const int tid = threadIdx.x, tx = tid % S::TX, ty = tid / S::TX;
    // A: 128 rows x 16 k = 512 float4; thread -> (row = q / 4, kq = q % 4) for q = tid, tid + 256
    // B: NT columns x 16 k = NT * 4 float4
    constexpr int BQ = (NT * 4 + TG_THREADS - 1) / TG_THREADS;
    typename LA::Raw ra[2];
    float4 rb[BQ];
    auto load = [&](int k0) {  // long-latency loads only (see ActIn::raw)
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int q = tid + u * TG_THREADS;
            ra[u] = la.raw(m0 + (q >> 2), k0 + 4 * (q & 3));
        }
#pragma unroll
        for (int u = 0; u < BQ; ++u) {
            const int q = tid + u * TG_THREADS;
            rb[u] = q < NT * 4 ? lb.four(n0 + (q >> 2), k0 + 4 * (q & 3)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto store = [&](int buf, int k0) {
        float *a = As + buf * TG_KC * S::AS, *b = Bs + buf * TG_KC * S::BS;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int q = tid + u * TG_THREADS, r = q >> 2, kq = 4 * (q & 3);
            const float4 v = la.finish(ra[u], m0 + r, k0 + kq);
            a[(kq + 0) * S::AS + r] = v.x; a[(kq + 1) * S::AS + r] = v.y;
            a[(kq + 2) * S::AS + r] = v.z; a[(kq + 3) * S::AS + r] = v.w;
        }
#pragma unroll
        for (int u = 0; u < BQ; ++u) {
            const int q = tid + u * TG_THREADS;
            if (q < NT * 4) {
                const int n = q >> 2, kq = 4 * (q & 3);
                b[(kq + 0) * S::BS + n] = rb[u].x; b[(kq + 1) * S::BS + n] = rb[u].y;
                b[(kq + 2) * S::BS + n] = rb[u].z; b[(kq + 3) * S::BS + n] = rb[u].w;
            }
        }
    };
#pragma unroll
    for (int i = 0; i < S::TM; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int nchunks = (K + TG_KC - 1) / TG_KC;
    load(0);
    store(0, 0);
    __syncthreads();
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) load((c + 1) * TG_KC);
        mma_chunk<NT>(As + (c & 1) * TG_KC * S::AS, Bs + (c & 1) * TG_KC * S::BS, acc, ty, tx);
        if (c + 1 < nchunks) store((c + 1) & 1, (c + 1) * TG_KC);
        __syncthreads();
    }
}

// ---- forward: z = act_in(x) W^T + b, per-channel sum / sum of squares of z ---------------------------------------------------
// STATS = false (stats == NULL: every layer whose BatchNorm normalises with its running statistics) stores z only: no
// column-sum shuffles, no shared-memory partials, no float64 atomics
template <int NT, class LX, bool STATS>
__global__ void __launch_bounds__(TG_THREADS, 2)
train_linear_fwd_kernel(LX xin, WeightIn w, const float *__restrict__ bias, float *__restrict__ z, double *__restrict__ stats,
                        long long tiles) {
    using S = TileShape<NT>;
    extern __shared__ __align__(16) float smem[];
    __shared__ float cpart[2][TG_THREADS / 32][NT];  // per-warp partial sums of the tile's columns (sum, sum of squares)
    __shared__ float tpiv[NT];                       // the tile's pivots (its first row of z)
    const int cout = w.n_total, cin = w.k_total;
    const int tid = threadIdx.x, tx = tid % S::TX, ty = tid / S::TX;
    const int ntn = (cout + NT - 1) / NT;
    for (long long t = blockIdx.x; t < tiles * ntn; t += gridDim.x) {
        const long long mt = t / ntn;
        const int n0 = (int)(t - mt * ntn) * NT;
        const long long m0 = mt * TG_M;
        float acc[S::TM][4];
        gemm_rows<NT>(xin, w, m0, n0, cin, smem, acc);
        float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
        const int col = n0 + tx * 4;
        float bv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) bv[j] = col + j < cout ? __ldg(bias + col + j) : 0.f;
        // The statistics are summed CENTRED on a pivot p per column, the tile's first row: s1 = sum (z - p), s2 =
        // sum (z - p)^2, expanded to sum z = s1 + n p and sum z^2 = s2 + 2 p s1 + n p^2 in fp64.  An fp32 sum of z^2 loses
        // (mean / std)^2 of its relative precision in var = E[z^2] - mean^2 (1e-4 relative at mean / std = 100); the
        // centred sums lose nothing to the mean, and both expansions use the same s1, so the rounding of s1 cancels in var.
        float pv[4] = {0.f, 0.f, 0.f, 0.f};
        if constexpr (STATS) {
            if (ty == 0) {  // row m0 (always valid) is row 0 of the ty == 0 threads
#pragma unroll
                for (int j = 0; j < 4; ++j) tpiv[tx * 4 + j] = acc[0][j] + bv[j];
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 4; ++j) pv[j] = tpiv[tx * 4 + j];
        }
#pragma unroll
        for (int i = 0; i < S::TM; ++i) {
            const long long r = m0 + ty * S::TM + i;
            if (r >= xin.rows) continue;
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                v[j] = acc[i][j] + bv[j];
                if (STATS && col + j < cout) {
                    const float dv = v[j] - pv[j];
                    s1[j] += dv;
                    s2[j] = fmaf(dv, dv, s2[j]);
                }
            }
            if (col + 3 < cout && (cout & 3) == 0) {
                *reinterpret_cast<float4 *>(z + r * cout + col) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (col + j < cout) z[r * cout + col + j] = v[j];
            }
        }
        if constexpr (!STATS) continue;
        // column sums: lanes of a warp that share tx (32 / TX rows of threads) by shuffles, the 8 warps through shared
        // memory (shared-memory float atomics compile to compare-and-swap loops: 8-way contended, they were 7 % of the
        // kernel's instructions and a quarter of its stall samples)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int o = S::TX; o < 32; o <<= 1) {
                s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], o);
                s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], o);
            }
        }
        if ((tid & 31) < S::TX) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                cpart[0][tid >> 5][tx * 4 + j] = s1[j];
                cpart[1][tid >> 5][tx * 4 + j] = s2[j];
            }
        }
        __syncthreads();
        if (tid < NT && n0 + tid < cout) {
            float t1 = 0.f, t2 = 0.f;
#pragma unroll
            for (int w8 = 0; w8 < TG_THREADS / 32; ++w8) {
                t1 += cpart[0][w8][tid];
                t2 += cpart[1][w8][tid];
            }
            const double p = (double)tpiv[tid], n = (double)min((long long)TG_M, xin.rows - m0);
            atomicAdd(stats + n0 + tid, fma(n, p, (double)t1));
            atomicAdd(stats + (size_t)cout + n0 + tid, (double)t2 + p * (2.0 * (double)t1 + n * p));
        }
        __syncthreads();
    }
}

// ---- backward reductions of BatchNorm: S1 = sum dy, S2 = sum dy z -------------------------------------------------------------
__global__ void __launch_bounds__(256)
train_bn_bwd_reduce_kernel(long long rows, int c, const float *__restrict__ g, const float *__restrict__ z, const float *__restrict__ scale,
                           const float *__restrict__ shift, double *__restrict__ sums) {
    // lanes along channels (coalesced rows), the 8 warps of a CTA and the CTAs of the grid along rows.
    // Each lane reduces sum dy (z - p) about a pivot p = the first z of its row range and adds p sum dy back in fp64: the
    // coefficients use S2 - mean S1, which an fp32 sum of dy z buries under its rounding once |mean| >> std.  S1 is
    // combined across the warps in fp64 too, so S2 carries exactly the S1 its pivot terms were formed from.
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ double red[2][8][32];
    const long long r0 = (long long)blockIdx.x * 8 + warp;
    for (int c0 = 0; c0 < c; c0 += 32) {
        const int ch = c0 + lane;
        float s1 = 0.f, s2 = 0.f, p = 0.f;
        if (ch < c) {
            const float sc = __ldg(scale + ch), sh = __ldg(shift + ch);
            if (r0 < rows) p = __ldg(z + r0 * c + ch);
            for (long long r = r0; r < rows; r += (long long)gridDim.x * 8) {
                const float zz = __ldg(z + r * c + ch), gg = __ldg(g + r * c + ch);
                const float dy = fmaf(zz, sc, sh) > 0.f ? gg : 0.f;
                s1 += dy;
                s2 = fmaf(dy, zz - p, s2);
            }
        }
        red[0][warp][lane] = (double)s1;
        red[1][warp][lane] = fma((double)p, (double)s1, (double)s2);
        __syncthreads();
        if (warp < 2 && ch < c) {
            double t = 0.0;
#pragma unroll
            for (int w8 = 0; w8 < 8; ++w8) t += red[warp][w8][lane];
            atomicAdd(sums + (size_t)warp * c + ch, t);
        }
        __syncthreads();
    }
}

// ---- backward, input gradient: g_in = dz W  (W^T given as wt (cin, cout) row-major) -------------------------------------------
// SPLIT (first layer of an FP block): columns < split go to g_skip (rows, split), the others to g_in (rows, cin - split);
// either may be NULL
template <int NT, bool SPLIT>
__global__ void __launch_bounds__(TG_THREADS, 2)
train_linear_bwd_input_kernel(DzIn dz, WeightIn wt, float *__restrict__ g_in, float *__restrict__ g_skip, int split, long long tiles) {
    using S = TileShape<NT>;
    extern __shared__ __align__(16) float smem[];
    const int cin = wt.n_total, cout = wt.k_total;
    const int tid = threadIdx.x, tx = tid % S::TX, ty = tid / S::TX;
    const int ntn = (cin + NT - 1) / NT;
    for (long long t = blockIdx.x; t < tiles * ntn; t += gridDim.x) {
        const long long mt = t / ntn;
        const int n0 = (int)(t - mt * ntn) * NT;
        const long long m0 = mt * TG_M;
        float acc[S::TM][4];
        gemm_rows<NT>(dz, wt, m0, n0, cout, smem, acc);
        const int col = n0 + tx * 4;
#pragma unroll
        for (int i = 0; i < S::TM; ++i) {
            const long long r = m0 + ty * S::TM + i;
            if (r >= dz.rows) continue;
            if constexpr (SPLIT) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int cj = col + j;
                    if (cj >= cin) continue;
                    if (cj < split) {
                        if (g_skip) g_skip[r * split + cj] = acc[i][j];
                    } else if (g_in) {
                        g_in[r * (cin - split) + (cj - split)] = acc[i][j];
                    }
                }
            } else if (col + 3 < cin && (cin & 3) == 0) {
                *reinterpret_cast<float4 *>(g_in + r * cin + col) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (col + j < cin) g_in[r * cin + col + j] = acc[i][j];
            }
        }
    }
}

// ---- backward, weight gradient: dW[co][ci] += sum_r dz[r][co] act_in(x)[r][ci] over a row range per CTA -----------------------
// Both operands are contiguous along their channel (row-major activations), so the k-chunk (16 rows) is staged as it lies:
// As[k][co], Bs[k][ci].  Output tile 128 (co) x NT (ci); the CTA walks its rows once per output tile.
template <int NT, int MT, class LX>
__global__ void __launch_bounds__(TG_THREADS, 2)
train_linear_bwd_weight_kernel(DzIn dz, LX xin, float *__restrict__ dw, long long rows_per_cta) {
    using S = TileShape<NT, MT>;
    extern __shared__ __align__(16) float smem[];
    float *As = smem, *Bs = smem + 2 * TG_KC * S::AS;
    const int cout = dz.c, cin = xin.c;
    const int tid = threadIdx.x, tx = tid % S::TX, ty = tid / S::TX;
    const long long r_begin = (long long)blockIdx.x * rows_per_cta;
    const long long r_end = min(dz.rows, r_begin + rows_per_cta);
    if (r_begin >= r_end) return;
    const int nchunks = (int)((r_end - r_begin + TG_KC - 1) / TG_KC);
    constexpr int BQ = (NT * 4 + TG_THREADS - 1) / TG_THREADS;
    // blockIdx.y = output tile (m0, n0): deep layers have few rows but many tiles, shallow ones the opposite
    const int ntn = (cin + NT - 1) / NT;
        {
            const int m0 = (int)(blockIdx.y / ntn) * MT, n0 = (int)(blockIdx.y % ntn) * NT;
            float acc[S::TM][4];
#pragma unroll
            for (int i = 0; i < S::TM; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
            constexpr int AQ = (MT * 4 + TG_THREADS - 1) / TG_THREADS;
            DzIn::Raw ra[AQ];
            typename LX::Raw rb[BQ];
            // A chunk: 16 rows x MT co = MT * 4 float4: q -> (k = q / (MT / 4), co4 = q % (MT / 4));  B chunk: 16 rows x NT ci
            // rows past the CTA's range are read as rows past the end of the matrix (zeros)
            auto load = [&](long long r0) {  // long-latency loads only (see ActIn::raw)
#pragma unroll
                for (int u = 0; u < AQ; ++u) {
                    const int q = tid + u * TG_THREADS;
                    const long long r = r0 + q / (MT / 4);
                    if (q < MT * 4) ra[u] = dz.raw(r < r_end ? r : dz.rows, m0 + 4 * (q % (MT / 4)));
                }
#pragma unroll
                for (int u = 0; u < BQ; ++u) {
                    const int q = tid + u * TG_THREADS;
                    const long long r = r0 + q / (NT / 4);
                    if (q < NT * 4) rb[u] = xin.raw(r < r_end ? r : xin.rows, n0 + 4 * (q % (NT / 4)));
                }
            };
            auto store = [&](int buf, long long r0) {
                float *a = As + buf * TG_KC * S::AS, *b = Bs + buf * TG_KC * S::BS;
#pragma unroll
                for (int u = 0; u < AQ; ++u) {
                    const int q = tid + u * TG_THREADS;
                    const long long r = r0 + q / (MT / 4);
                    if (q < MT * 4)
                        *reinterpret_cast<float4 *>(a + (q / (MT / 4)) * S::AS + 4 * (q % (MT / 4))) =
                            dz.finish(ra[u], r < r_end ? r : dz.rows, m0 + 4 * (q % (MT / 4)));
                }
#pragma unroll
                for (int u = 0; u < BQ; ++u) {
                    const int q = tid + u * TG_THREADS;
                    const long long r = r0 + q / (NT / 4);
                    if (q < NT * 4)
                        *reinterpret_cast<float4 *>(b + (q / (NT / 4)) * S::BS + 4 * (q % (NT / 4))) =
                            xin.finish(rb[u], r < r_end ? r : xin.rows, n0 + 4 * (q % (NT / 4)));
                }
            };
            __syncthreads();  // the previous output tile's last chunk has been consumed
            load(r_begin);
            store(0, r_begin);
            __syncthreads();
            for (int c = 0; c < nchunks; ++c) {
                if (c + 1 < nchunks) load(r_begin + (long long)(c + 1) * TG_KC);
                mma_chunk<NT, MT>(As + (c & 1) * TG_KC * S::AS, Bs + (c & 1) * TG_KC * S::BS, acc, ty, tx);
                if (c + 1 < nchunks) store((c + 1) & 1, r_begin + (long long)(c + 1) * TG_KC);
                __syncthreads();
            }
#pragma unroll
            for (int i = 0; i < S::TM; ++i) {
                const int co = m0 + ty * S::TM + i;
                if (co >= cout) continue;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int ci = n0 + tx * 4 + j;
                    if (ci < cin) atomicAdd(dw + (size_t)co * cin + ci, acc[i][j]);
                }
            }
        }
}

// ---- the BatchNorm + ReLU of the LAST layer of a stack, materialised (what the max-pool / the next block consumes) ------------
__global__ void __launch_bounds__(256)
train_bn_relu_kernel(long long total4, int c, const float *__restrict__ z, const float *__restrict__ scale, const float *__restrict__ shift,
                     float *__restrict__ a) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < total4; e += (long long)gridDim.x * 256) {
        const int k = (int)((e * 4) % c);
        const float4 v = __ldg(reinterpret_cast<const float4 *>(z) + e);
        const float4 s = __ldg(reinterpret_cast<const float4 *>(scale + k)), t = __ldg(reinterpret_cast<const float4 *>(shift + k));
        reinterpret_cast<float4 *>(a)[e] = make_float4(fmaxf(fmaf(v.x, s.x, t.x), 0.f), fmaxf(fmaf(v.y, s.y, t.y), 0.f),
                                                       fmaxf(fmaf(v.z, s.z, t.z), 0.f), fmaxf(fmaf(v.w, s.w, t.w), 0.f));
    }
}
__global__ void __launch_bounds__(256)
train_bn_relu_scalar_kernel(long long total, int c, const float *__restrict__ z, const float *__restrict__ scale,
                            const float *__restrict__ shift, float *__restrict__ a) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < total; e += (long long)gridDim.x * 256) {
        const int k = (int)(e % c);
        a[e] = fmaxf(fmaf(__ldg(z + e), __ldg(scale + k), __ldg(shift + k)), 0.f);
    }
}

// ---- last layer of an SA scale: BatchNorm + ReLU + max over the k rows of a group, the winning row kept for the backward ------
// thread <-> (group, channel), lanes along channels: every z row is read coalesced; the (rows, c) activation is never written
__global__ void __launch_bounds__(256)
train_bn_relu_max_kernel(long long groups, int k, int c, const float *__restrict__ z, const float *__restrict__ scale,
                         const float *__restrict__ shift, float *__restrict__ out, int out_stride, int out_offset,
                         uint8_t *__restrict__ arg) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < groups * c; e += (long long)gridDim.x * 256) {
        const long long gr = e / c;
        const int ch = (int)(e - gr * c);
        const float sc = __ldg(scale + ch), sh = __ldg(shift + ch);
        const float *zr = z + gr * k * c + ch;
        float best = fmaxf(fmaf(__ldg(zr), sc, sh), 0.f);
        int bj = 0;
        for (int j = 1; j < k; ++j) {
            const float a = fmaxf(fmaf(__ldg(zr + (long long)j * c), sc, sh), 0.f);
            if (a > best) {  // strict: the first maximum wins, as torch.max(dim) reports it
                best = a;
                bj = j;
            }
        }
        out[gr * out_stride + out_offset + ch] = best;
        arg[e] = (uint8_t)bj;
    }
}

// ---- the same pooling over ALL k rows of a group (group_all), k unbounded: warp <-> (group, 32 channels, row range) --------
// Lanes along channels (coalesced z rows); a warp keeps the largest activation and its first row over its range, then the
// ranges of a group are combined by a 64-bit atomicMax on key = (value bits << 32) | ~row: the values are non-negative
// (ReLU; -0 is stored as +0), so the bits order like the values, and on equal values the smaller row has the larger ~row.
// Exact and independent of the order of the CTAs.  keys (groups, c) start at 0, below every real key.
__global__ void __launch_bounds__(256)
train_bn_relu_max_all_kernel(long long groups, long long k, int c, const float *__restrict__ z, const float *__restrict__ scale,
                             const float *__restrict__ shift, long long rows_per_range, unsigned long long *__restrict__ keys) {
    const int lane = threadIdx.x & 31;
    const int nchunks = (c + 31) / 32;
    const long long nranges = (k + rows_per_range - 1) / rows_per_range;
    const long long items = groups * nchunks * nranges;
    for (long long it = ((long long)blockIdx.x * 256 + threadIdx.x) / 32; it < items; it += (long long)gridDim.x * 8) {
        const long long gr = it / (nchunks * nranges);
        const long long rest = it - gr * nchunks * nranges;
        const int ch = (int)(rest / nranges) * 32 + lane;
        const long long j0 = (rest % nranges) * rows_per_range, j1 = min(k, j0 + rows_per_range);
        if (ch >= c) continue;
        const float sc = __ldg(scale + ch), sh = __ldg(shift + ch);
        const float *zr = z + gr * k * c + ch;
        float best = -1.f;
        long long bj = j0;
#pragma unroll 4
        for (long long j = j0; j < j1; ++j) {
            const float a = fmaxf(fmaf(__ldg(zr + j * c), sc, sh), 0.f);
            if (a > best) {  // strict: the first maximum wins, as torch.max(dim) reports it
                best = a;
                bj = j;
            }
        }
        const unsigned long long key = ((unsigned long long)(best > 0.f ? __float_as_uint(best) : 0u) << 32) | (unsigned)~(unsigned)bj;
        atomicMax(keys + gr * c + ch, key);
    }
}

__global__ void __launch_bounds__(256)
train_max_all_finalize_kernel(long long groups, int c, const unsigned long long *__restrict__ keys, float *__restrict__ out,
                              int out_stride, int out_offset, int32_t *__restrict__ arg) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < groups * c; e += (long long)gridDim.x * 256) {
        const long long gr = e / c;
        const unsigned long long key = keys[e];
        out[gr * out_stride + out_offset + (e - gr * c)] = __uint_as_float((unsigned)(key >> 32));
        arg[e] = (int32_t)~(unsigned)key;
    }
}

// ---- backward of either pooling: the pooled gradient on the winning row, 0 on the others; every element of g is written -------
template <class Arg>
__global__ void __launch_bounds__(256)
train_max_bwd_kernel(long long groups, long long k, int c, const float *__restrict__ gp, int gp_stride, int gp_offset,
                     const Arg *__restrict__ arg, float *__restrict__ g) {
    const long long total = groups * k * c;
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < total; e += (long long)gridDim.x * 256) {
        const long long row = e / c;
        const int ch = (int)(e - row * c);
        const long long gr = row / k;
        const long long j = row - gr * k;
        g[e] = (long long)__ldg(arg + gr * c + ch) == j ? __ldg(gp + gr * gp_stride + gp_offset + ch) : 0.f;
    }
}

// ---- per-channel coefficient kernels (one tiny launch instead of ~15 elementwise torch launches per layer and direction) ----
// forward: (sum z, sum z^2) -> mean, biased var, rstd (fp64 -> fp32 where stored), scale = gamma rstd, shift = beta - mean scale;
// running statistics updated like torch.nn.BatchNorm in training mode (momentum, UNBIASED variance).
__global__ void train_bn_finalize_kernel(int c, double rows, const double *__restrict__ stats, const float *__restrict__ gamma,
                                         const float *__restrict__ beta, double eps, double momentum, float *__restrict__ scale,
                                         float *__restrict__ shift, double *__restrict__ mean_rstd, float *__restrict__ running_mean,
                                         float *__restrict__ running_var) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= c) return;
    const double mean = stats[k] / rows;
    double var = stats[c + k] / rows - mean * mean;
    var = var > 0.0 ? var : 0.0;
    const double rstd = rsqrt(var + eps);
    const double g = (double)gamma[k];
    scale[k] = (float)(g * rstd);
    shift[k] = (float)((double)beta[k] - mean * g * rstd);
    mean_rstd[k] = mean;
    mean_rstd[c + k] = rstd;
    if (running_mean) {
        running_mean[k] = (float)((1.0 - momentum) * (double)running_mean[k] + momentum * (double)(float)mean);
        const double unbiased = (double)(float)var * (rows / (rows > 1.0 ? rows - 1.0 : 1.0));
        running_var[k] = (float)((1.0 - momentum) * (double)running_var[k] + momentum * unbiased);
    }
}

// backward: (S1 = sum dy, S2 = sum dy z) -> ca, cb, cc of dz = ca dy + cb + cc z; dgamma = rstd (S2 - mean S1), dbeta = S1
__global__ void train_bn_bwd_coeffs_kernel(int c, double rows, const double *__restrict__ sums, const double *__restrict__ mean_rstd,
                                           const float *__restrict__ gamma, float *__restrict__ coef, float *__restrict__ dgamma,
                                           float *__restrict__ dbeta) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= c) return;
    const double S1 = sums[k], S2 = sums[c + k], mean = mean_rstd[k], rstd = mean_rstd[c + k], g = (double)gamma[k];
    const double t = S2 - mean * S1;
    const double ca = g * rstd;
    const double cc = -g * rstd * rstd * rstd * t / rows;
    const double cb = -ca * S1 / rows - cc * mean;
    coef[k] = (float)ca;
    coef[c + k] = (float)cb;
    coef[2 * c + k] = (float)cc;
    dgamma[k] = (float)(rstd * t);
    dbeta[k] = (float)S1;
}

// ---- the same two coefficient kernels for a BatchNorm that normalises with its RUNNING statistics (eval mode: torch's
// rule is batch statistics iff bn.training or running_mean is None).  zhat = (z - rm) rstd with constant rm, rstd, so
// dL/dz = gamma rstd dy: ca = scale, cb = cc = 0.  Nothing but the outputs is written (the running statistics stay as they are).
__global__ void train_bn_running_kernel(int c, const float *__restrict__ running_mean, const float *__restrict__ running_var,
                                        const float *__restrict__ gamma, const float *__restrict__ beta, double eps,
                                        float *__restrict__ scale, float *__restrict__ shift, double *__restrict__ mean_rstd) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= c) return;
    const double rm = (double)running_mean[k];
    const double rstd = rsqrt((double)running_var[k] + eps);
    const double g = (double)gamma[k];
    scale[k] = (float)(g * rstd);
    shift[k] = (float)((double)beta[k] - rm * g * rstd);
    mean_rstd[k] = rm;
    mean_rstd[c + k] = rstd;
}

// (S1 = sum dy, S2 = sum dy z) -> coef = (scale, 0, 0); dgamma = rstd (S2 - rm S1), dbeta = S1, and the conv bias gradient
// dbias = sum dz = scale S1 (not zero here: nothing subtracts the batch mean)
__global__ void train_bn_running_bwd_coeffs_kernel(int c, const double *__restrict__ sums, const double *__restrict__ mean_rstd,
                                                   const float *__restrict__ scale, float *__restrict__ coef,
                                                   float *__restrict__ dgamma, float *__restrict__ dbeta, float *__restrict__ dbias) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= c) return;
    const double S1 = sums[k], S2 = sums[c + k], rm = mean_rstd[k], rstd = mean_rstd[c + k];
    const float sc = scale[k];
    coef[k] = sc;
    coef[c + k] = 0.f;
    coef[2 * c + k] = 0.f;
    dgamma[k] = (float)(rstd * (S2 - rm * S1));
    dbeta[k] = (float)S1;
    dbias[k] = (float)((double)sc * S1);
}

int pick_nt(int n) { return n <= 32 ? 32 : (n <= 64 ? 64 : 128); }

template <int NT>
size_t tile_smem() { return TileShape<NT>::smem_floats * sizeof(float); }


template <class LX>
int launch_fwd(const LX &a, const WeightIn &b, const float *bias, float *z, double *stats, cudaStream_t s) {
    const long long rows = a.rows;
    const int cout = b.n_total;
    const long long tiles = (rows + TG_M - 1) / TG_M;
    const int nt = pick_nt(cout);
    const long long work = tiles * ((cout + nt - 1) / nt);
    const unsigned grid = (unsigned)(work < 2ll * sm_count() ? work : 2ll * sm_count());
#define PN2_FW(NTV, ST) train_linear_fwd_kernel<NTV, LX, ST><<<grid, TG_THREADS, tile_smem<NTV>(), s>>>(a, b, bias, z, stats, tiles)
    if (stats) {
        if (nt == 32) PN2_FW(32, true); else if (nt == 64) PN2_FW(64, true); else PN2_FW(128, true);
    } else {
        if (nt == 32) PN2_FW(32, false); else if (nt == 64) PN2_FW(64, false); else PN2_FW(128, false);
    }
#undef PN2_FW
    PN2_LAUNCH_OK("train_linear_fwd_kernel");
    return PN2_OK;
}

// g_in = dz W (split: see train_linear_bwd_input_kernel), then dW += dz^T x
template <class LX>
int launch_bwd(const DzIn &dz, const LX &a, const float *wt, float *g_in, float *g_skip, int split, float *dw, cudaStream_t s) {
    const long long rows = dz.rows;
    const int cin = a.c, cout = dz.c;
    const long long tiles = (rows + TG_M - 1) / TG_M;
    if (g_in || g_skip) {
        WeightIn b = {wt, cin, cout};
        const int nt = pick_nt(cin);
        const long long work = tiles * ((cin + nt - 1) / nt);
        const unsigned grid = (unsigned)(work < 2ll * sm_count() ? work : 2ll * sm_count());
#define PN2_BI(NTV, SPL) train_linear_bwd_input_kernel<NTV, SPL><<<grid, TG_THREADS, tile_smem<NTV>(), s>>>(dz, b, g_in, g_skip, split, tiles)
        if (split > 0) {
            if (nt == 32) PN2_BI(32, true); else if (nt == 64) PN2_BI(64, true); else PN2_BI(128, true);
        } else {
            if (nt == 32) PN2_BI(32, false); else if (nt == 64) PN2_BI(64, false); else PN2_BI(128, false);
        }
#undef PN2_BI
        PN2_LAUNCH_OK("train_linear_bwd_input_kernel");
    }
    {
        // grid = (row ranges, output tiles): about four CTAs per SM in total, at least 128 rows per range (the partial sums
        // go to dW with atomics)
        // output tile (cout x cin) = mt x nt: no padded FMAs for narrow layers.  The interpolated operand stages three source
        // rows per element: its 128 x 128 tile spilled (412 bytes), so it stays at 64 input channels per tile.
        constexpr bool wide_ok = !std::is_same<LX, InterpIn>::value;
        const int nt = wide_ok ? pick_nt(cin) : min(pick_nt(cin), 64), mt = pick_nt(cout);
        const long long out_tiles = (long long)((cout + mt - 1) / mt) * ((cin + nt - 1) / nt);
        PN2_REQUIRE(out_tiles <= 65535, "train_linear_bwd: too many output tiles");
        long long ranges = (4ll * sm_count() + out_tiles - 1) / out_tiles;
        long long per = (rows + ranges - 1) / ranges;
        if (per < 128) per = 128;
        per = (per + TG_KC - 1) / TG_KC * TG_KC;
        ranges = (rows + per - 1) / per;
        const dim3 grid((unsigned)ranges, (unsigned)out_tiles);
#define PN2_WG(NTV, MTV) train_linear_bwd_weight_kernel<NTV, MTV><<<grid, TG_THREADS, TileShape<NTV, MTV>::smem_floats * sizeof(float), s>>>(dz, a, dw, per)
        if (mt == 32) {
            if (nt == 32) PN2_WG(32, 32); else if (nt == 64) PN2_WG(64, 32); else if constexpr (wide_ok) PN2_WG(128, 32);
        } else if (mt == 64) {
            if (nt == 32) PN2_WG(32, 64); else if (nt == 64) PN2_WG(64, 64); else if constexpr (wide_ok) PN2_WG(128, 64);
        } else {
            if (nt == 32) PN2_WG(32, 128); else if (nt == 64) PN2_WG(64, 128); else if constexpr (wide_ok) PN2_WG(128, 128);
        }
#undef PN2_WG
        PN2_LAUNCH_OK("train_linear_bwd_weight_kernel");
    }
    return PN2_OK;
}

bool aligned16(const void *p) { return ((uintptr_t)p & 15) == 0; }

// Validates a pn2_rows against (rows, cin) and builds its loader.  Returns PN2_OK or the error status.
int rows_loader(const char *who, long long rows, int cin, const pn2_rows *src, GroupIn &gi, InterpIn &ii, AllIn &ai) {
    PN2_REQUIRE(src, "%s: null row source", who);
    PN2_REQUIRE(src->kind == PN2_ROWS_GROUPED || src->kind == PN2_ROWS_INTERP || src->kind == PN2_ROWS_ALL,
                "%s: unknown row source kind %d", who, src->kind);
    PN2_REQUIRE(rows < (1ll << 31), "%s: more than 2^31 rows", who);
    const pn2_rows &r = *src;
    if (r.kind == PN2_ROWS_GROUPED) {
        PN2_REQUIRE(r.b >= 1 && r.n >= 1 && r.m >= 1 && r.k >= 1 && r.d >= 0 && (r.order == PN2_ORDER_XYZ_FIRST || r.order == PN2_ORDER_FEAT_FIRST),
                    "%s: bad grouped source b=%d n=%d m=%d k=%d d=%d order=%d", who, r.b, r.n, r.m, r.k, r.d, r.order);
        PN2_REQUIRE(rows == (long long)r.b * r.m * r.k && cin == 3 + r.d, "%s: rows=%lld cin=%d do not match the grouped source", who, rows, cin);
        PN2_REQUIRE(r.xyz && r.new_xyz && r.idx && ((r.feat == nullptr) == (r.d == 0)), "%s: null pointer", who);
        const bool xyz_first = r.order == PN2_ORDER_XYZ_FIRST;
        gi = {r.xyz, r.new_xyz, r.feat, r.idx, rows, cin, r.n, r.m, r.k, r.d, xyz_first ? 0 : r.d, xyz_first ? 3 : 0,
              r.d > 0 && (r.d & 3) == 0 && aligned16(r.feat)};
    } else if (r.kind == PN2_ROWS_ALL) {
        PN2_REQUIRE(r.b >= 1 && r.n >= 1 && r.d >= 0, "%s: bad group_all source b=%d n=%d d=%d", who, r.b, r.n, r.d);
        PN2_REQUIRE(rows == (long long)r.b * r.n && cin == 3 + r.d, "%s: rows=%lld cin=%d do not match the group_all source", who, rows, cin);
        PN2_REQUIRE(r.xyz && ((r.feat == nullptr) == (r.d == 0)), "%s: null pointer", who);
        ai = {r.xyz, r.feat, rows, cin, r.d};
    } else {
        PN2_REQUIRE(r.b >= 1 && r.n >= 1 && r.m >= 1 && r.d >= 1 && r.d_skip >= 0, "%s: bad interpolated source b=%d n=%d m=%d d=%d d_skip=%d",
                    who, r.b, r.n, r.m, r.d, r.d_skip);
        PN2_REQUIRE(rows == (long long)r.b * r.n && cin == r.d_skip + r.d, "%s: rows=%lld cin=%d do not match the interpolated source", who,
                    rows, cin);
        PN2_REQUIRE(r.feat && ((r.skip == nullptr) == (r.d_skip == 0)) && (r.m == 1 || (r.idx && r.weight)), "%s: null pointer", who);
        ii = {r.skip, r.feat, r.weight, r.m == 1 ? nullptr : r.idx, rows, cin, r.n, r.m, r.d, r.d_skip,
              r.d_skip > 0 && (r.d_skip & 3) == 0 && aligned16(r.skip), (r.d & 3) == 0 && aligned16(r.feat)};
    }
    return PN2_OK;
}

}  // namespace
}  // namespace pn2

using namespace pn2;

extern "C" int pn2_train_linear_fwd(long long rows, int cin, int cout, const float *x, const float *in_scale, const float *in_shift,
                                    const float *w, const float *bias, float *z, double *stats, void *stream) {
    PN2_REQUIRE(rows >= 0 && cin >= 1 && cout >= 1, "train_linear_fwd: bad dims rows=%lld cin=%d cout=%d", rows, cin, cout);
    if (rows == 0) return PN2_OK;
    PN2_REQUIRE(x && w && bias && z && ((in_scale == nullptr) == (in_shift == nullptr)), "train_linear_fwd: null pointer");
    PN2_REQUIRE((((uintptr_t)x | (uintptr_t)w | (uintptr_t)z | (uintptr_t)in_scale | (uintptr_t)in_shift) & 15) == 0, "train_linear_fwd: 16-byte alignment");
    ActIn a = {x, in_scale, in_shift, rows, cin};
    return launch_fwd(a, WeightIn{w, cout, cin}, bias, z, stats, (cudaStream_t)stream);
}

extern "C" int pn2_train_linear_fwd_rows(long long rows, int cin, int cout, const pn2_rows *src, const float *w, const float *bias,
                                         float *z, double *stats, void *stream) {
    PN2_REQUIRE(rows >= 0 && cin >= 1 && cout >= 1, "train_linear_fwd_rows: bad dims rows=%lld cin=%d cout=%d", rows, cin, cout);
    if (rows == 0) return PN2_OK;
    GroupIn gi;
    InterpIn ii;
    AllIn ai;
    if (int st = rows_loader("train_linear_fwd_rows", rows, cin, src, gi, ii, ai)) return st;
    PN2_REQUIRE(w && bias && z, "train_linear_fwd_rows: null pointer");
    PN2_REQUIRE((((uintptr_t)w | (uintptr_t)z) & 15) == 0, "train_linear_fwd_rows: 16-byte alignment");
    const WeightIn b = {w, cout, cin};
    cudaStream_t s = (cudaStream_t)stream;
    if (src->kind == PN2_ROWS_ALL) return launch_fwd(ai, b, bias, z, stats, s);
    return src->kind == PN2_ROWS_GROUPED ? launch_fwd(gi, b, bias, z, stats, s) : launch_fwd(ii, b, bias, z, stats, s);
}

extern "C" int pn2_train_bn_bwd_reduce(long long rows, int c, const float *g, const float *z, const float *scale, const float *shift,
                                       double *sums, void *stream) {
    PN2_REQUIRE(rows >= 0 && c >= 1, "train_bn_bwd_reduce: bad dims");
    if (rows == 0) return PN2_OK;
    PN2_REQUIRE(g && z && scale && shift && sums, "train_bn_bwd_reduce: null pointer");
    long long want = (rows + 63) / 64;
    const unsigned grid = (unsigned)(want < 4ll * sm_count() ? (want < 1 ? 1 : want) : 4ll * sm_count());
    train_bn_bwd_reduce_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rows, c, g, z, scale, shift, sums);
    PN2_LAUNCH_OK("train_bn_bwd_reduce_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_linear_bwd(long long rows, int cin, int cout, const float *x, const float *in_scale, const float *in_shift,
                                    const float *wt, const float *g, const float *z, const float *scale, const float *shift,
                                    const float *ca, const float *cb, const float *cc, float *g_in, float *dw, void *stream) {
    PN2_REQUIRE(rows >= 0 && cin >= 1 && cout >= 1, "train_linear_bwd: bad dims rows=%lld cin=%d cout=%d", rows, cin, cout);
    if (rows == 0) return PN2_OK;
    PN2_REQUIRE(x && wt && g && z && scale && shift && ca && cb && cc && dw && ((in_scale == nullptr) == (in_shift == nullptr)),
                "train_linear_bwd: null pointer");
    // 128-bit loads are only used for widths that are multiples of 4: those tensors must then be 16-byte aligned
    PN2_REQUIRE((((uintptr_t)x | (uintptr_t)wt | (uintptr_t)g | (uintptr_t)z | (uintptr_t)g_in | (uintptr_t)in_scale | (uintptr_t)in_shift) & 15) == 0,
                "train_linear_bwd: 16-byte alignment");
    PN2_REQUIRE((cout & 3) != 0 || (((uintptr_t)scale | (uintptr_t)shift | (uintptr_t)ca | (uintptr_t)cb | (uintptr_t)cc) & 15) == 0,
                "train_linear_bwd: 16-byte alignment of the per-channel vectors");
    DzIn dz = {g, z, scale, shift, ca, cb, cc, rows, cout};
    ActIn a = {x, in_scale, in_shift, rows, cin};
    return launch_bwd(dz, a, wt, g_in, nullptr, 0, dw, (cudaStream_t)stream);
}

extern "C" int pn2_train_linear_bwd_rows(long long rows, int cin, int cout, const pn2_rows *src, const float *wt, const float *g,
                                         const float *z, const float *scale, const float *shift, const float *ca, const float *cb,
                                         const float *cc, float *g_in, float *g_skip, float *dw, void *stream) {
    PN2_REQUIRE(rows >= 0 && cin >= 1 && cout >= 1, "train_linear_bwd_rows: bad dims rows=%lld cin=%d cout=%d", rows, cin, cout);
    if (rows == 0) return PN2_OK;
    GroupIn gi;
    InterpIn ii;
    AllIn ai;
    if (int st = rows_loader("train_linear_bwd_rows", rows, cin, src, gi, ii, ai)) return st;
    PN2_REQUIRE(wt && g && z && scale && shift && ca && cb && cc && dw, "train_linear_bwd_rows: null pointer");
    PN2_REQUIRE(g_skip == nullptr || (src->kind == PN2_ROWS_INTERP && src->d_skip > 0),
                "train_linear_bwd_rows: g_skip needs an interpolated source with skip columns (d_skip > 0)");
    PN2_REQUIRE(g_in == nullptr || src->kind != PN2_ROWS_ALL || src->d > 0,
                "train_linear_bwd_rows: a group_all source without features (d == 0) has no input gradient");
    PN2_REQUIRE((((uintptr_t)wt | (uintptr_t)g | (uintptr_t)z | (uintptr_t)g_in) & 15) == 0, "train_linear_bwd_rows: 16-byte alignment");
    PN2_REQUIRE((cout & 3) != 0 || (((uintptr_t)scale | (uintptr_t)shift | (uintptr_t)ca | (uintptr_t)cb | (uintptr_t)cc) & 15) == 0,
                "train_linear_bwd_rows: 16-byte alignment of the per-channel vectors");
    DzIn dz = {g, z, scale, shift, ca, cb, cc, rows, cout};
    cudaStream_t s = (cudaStream_t)stream;
    if (src->kind == PN2_ROWS_GROUPED) return launch_bwd(dz, gi, wt, g_in, nullptr, 0, dw, s);
    // group_all: a row is a point, so the feature columns go straight to g_in = (b, n, d); the 3 xyz columns are dropped
    if (src->kind == PN2_ROWS_ALL) return launch_bwd(dz, ai, wt, g_in, nullptr, 3, dw, s);
    // an FP block's skip columns come first: split them off into g_skip (without skip columns g_in is (rows, cin))
    return launch_bwd(dz, ii, wt, g_in, g_skip, src->d_skip, dw, s);
}

extern "C" int pn2_train_bn_relu(long long rows, int c, const float *z, const float *scale, const float *shift, float *a, void *stream) {
    PN2_REQUIRE(rows >= 0 && c >= 1, "train_bn_relu: bad dims");
    if (rows == 0) return PN2_OK;
    PN2_REQUIRE(z && scale && shift && a, "train_bn_relu: null pointer");
    const long long total = rows * c;
    cudaStream_t s = (cudaStream_t)stream;
    if ((c & 3) == 0 && (((uintptr_t)z | (uintptr_t)a | (uintptr_t)scale | (uintptr_t)shift) & 15) == 0) {
        const long long t4 = total / 4;
        const unsigned grid = (unsigned)((t4 + 255) / 256 < 8ll * sm_count() ? (t4 + 255) / 256 : 8ll * sm_count());
        train_bn_relu_kernel<<<grid, 256, 0, s>>>(t4, c, z, scale, shift, a);
    } else {
        const unsigned grid = (unsigned)((total + 255) / 256 < 8ll * sm_count() ? (total + 255) / 256 : 8ll * sm_count());
        train_bn_relu_scalar_kernel<<<grid, 256, 0, s>>>(total, c, z, scale, shift, a);
    }
    PN2_LAUNCH_OK("train_bn_relu_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_bn_finalize(long long rows, int c, const double *stats, const float *gamma, const float *beta, double eps,
                                     double momentum, float *scale, float *shift, double *mean_rstd, float *running_mean,
                                     float *running_var, void *stream) {
    PN2_REQUIRE(rows >= 1 && c >= 1, "train_bn_finalize: bad dims");
    PN2_REQUIRE(stats && gamma && beta && scale && shift && mean_rstd && ((running_mean == nullptr) == (running_var == nullptr)),
                "train_bn_finalize: null pointer");
    train_bn_finalize_kernel<<<(c + 127) / 128, 128, 0, (cudaStream_t)stream>>>(c, (double)rows, stats, gamma, beta, eps, momentum, scale,
                                                                                shift, mean_rstd, running_mean, running_var);
    PN2_LAUNCH_OK("train_bn_finalize_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_bn_bwd_coeffs(long long rows, int c, const double *sums, const double *mean_rstd, const float *gamma, float *coef,
                                       float *dgamma, float *dbeta, void *stream) {
    PN2_REQUIRE(rows >= 1 && c >= 1, "train_bn_bwd_coeffs: bad dims");
    PN2_REQUIRE(sums && mean_rstd && gamma && coef && dgamma && dbeta, "train_bn_bwd_coeffs: null pointer");
    train_bn_bwd_coeffs_kernel<<<(c + 127) / 128, 128, 0, (cudaStream_t)stream>>>(c, (double)rows, sums, mean_rstd, gamma, coef, dgamma, dbeta);
    PN2_LAUNCH_OK("train_bn_bwd_coeffs_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_bn_running(int c, const float *running_mean, const float *running_var, const float *gamma, const float *beta,
                                    double eps, float *scale, float *shift, double *mean_rstd, void *stream) {
    PN2_REQUIRE(c >= 1 && eps >= 0.0, "train_bn_running: bad dims c=%d eps=%g", c, eps);
    PN2_REQUIRE(running_mean && running_var && gamma && beta && scale && shift && mean_rstd, "train_bn_running: null pointer");
    train_bn_running_kernel<<<(c + 127) / 128, 128, 0, (cudaStream_t)stream>>>(c, running_mean, running_var, gamma, beta, eps, scale,
                                                                               shift, mean_rstd);
    PN2_LAUNCH_OK("train_bn_running_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_bn_running_bwd_coeffs(int c, const double *sums, const double *mean_rstd, const float *scale, float *coef,
                                               float *dgamma, float *dbeta, float *dbias, void *stream) {
    PN2_REQUIRE(c >= 1, "train_bn_running_bwd_coeffs: bad dims c=%d", c);
    PN2_REQUIRE(sums && mean_rstd && scale && coef && dgamma && dbeta && dbias, "train_bn_running_bwd_coeffs: null pointer");
    train_bn_running_bwd_coeffs_kernel<<<(c + 127) / 128, 128, 0, (cudaStream_t)stream>>>(c, sums, mean_rstd, scale, coef, dgamma,
                                                                                          dbeta, dbias);
    PN2_LAUNCH_OK("train_bn_running_bwd_coeffs_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_bn_relu_max(long long groups, int k, int c, const float *z, const float *scale, const float *shift, float *out,
                                     int out_stride, int out_offset, uint8_t *arg, void *stream) {
    PN2_REQUIRE(groups >= 0 && k >= 1 && k <= 256 && c >= 1, "train_bn_relu_max: bad dims groups=%lld k=%d c=%d (k <= 256)", groups, k, c);
    PN2_REQUIRE(out_offset >= 0 && out_stride >= out_offset + c, "train_bn_relu_max: out_stride=%d out_offset=%d c=%d", out_stride, out_offset, c);
    if (groups == 0) return PN2_OK;
    PN2_REQUIRE(z && scale && shift && out && arg, "train_bn_relu_max: null pointer");
    const long long total = groups * c;
    const unsigned grid = (unsigned)((total + 255) / 256 < 8ll * sm_count() ? (total + 255) / 256 : 8ll * sm_count());
    train_bn_relu_max_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(groups, k, c, z, scale, shift, out, out_stride, out_offset, arg);
    PN2_LAUNCH_OK("train_bn_relu_max_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_max_bwd(long long groups, int k, int c, const float *gp, int gp_stride, int gp_offset, const uint8_t *arg,
                                 float *g, void *stream) {
    PN2_REQUIRE(groups >= 0 && k >= 1 && k <= 256 && c >= 1, "train_max_bwd: bad dims groups=%lld k=%d c=%d (k <= 256)", groups, k, c);
    PN2_REQUIRE(gp_offset >= 0 && gp_stride >= gp_offset + c, "train_max_bwd: gp_stride=%d gp_offset=%d c=%d", gp_stride, gp_offset, c);
    if (groups == 0) return PN2_OK;
    PN2_REQUIRE(gp && arg && g, "train_max_bwd: null pointer");
    const long long total = groups * k * c;
    const unsigned grid = (unsigned)((total + 255) / 256 < 8ll * sm_count() ? (total + 255) / 256 : 8ll * sm_count());
    train_max_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(groups, k, c, gp, gp_stride, gp_offset, arg, g);
    PN2_LAUNCH_OK("train_max_bwd_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_bn_relu_max_all(long long groups, long long k, int c, const float *z, const float *scale, const float *shift,
                                         float *out, int out_stride, int out_offset, int32_t *arg, void *stream) {
    PN2_REQUIRE(groups >= 0 && k >= 1 && k < (1ll << 31) && c >= 1, "train_bn_relu_max_all: bad dims groups=%lld k=%lld c=%d (1 <= k < 2^31)",
                groups, k, c);
    PN2_REQUIRE(out_offset >= 0 && out_stride >= out_offset + c, "train_bn_relu_max_all: out_stride=%d out_offset=%d c=%d", out_stride,
                out_offset, c);
    if (groups == 0) return PN2_OK;
    PN2_REQUIRE(z && scale && shift && out && arg, "train_bn_relu_max_all: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    Scratch keys(s);
    PN2_CUDA(keys.alloc((size_t)groups * c * sizeof(unsigned long long)));
    PN2_CUDA(cudaMemsetAsync(keys.ptr, 0, (size_t)groups * c * sizeof(unsigned long long), s));
    // row ranges: about 64 warps per SM in total, at least 128 rows each (one atomic per lane and range)
    const long long nchunks = (c + 31) / 32;
    const long long warps = 64ll * sm_count();
    long long per = (groups * nchunks * k + warps - 1) / warps;
    if (per < 128) per = 128;
    const long long items = groups * nchunks * ((k + per - 1) / per);
    const long long want = (items + 7) / 8;
    const unsigned grid = (unsigned)(want < 8ll * sm_count() ? want : 8ll * sm_count());
    train_bn_relu_max_all_kernel<<<grid, 256, 0, s>>>(groups, k, c, z, scale, shift, per, (unsigned long long *)keys.ptr);
    PN2_LAUNCH_OK("train_bn_relu_max_all_kernel");
    const long long total = groups * c;
    const unsigned fgrid = (unsigned)((total + 255) / 256 < 8ll * sm_count() ? (total + 255) / 256 : 8ll * sm_count());
    train_max_all_finalize_kernel<<<fgrid, 256, 0, s>>>(groups, c, (const unsigned long long *)keys.ptr, out, out_stride, out_offset, arg);
    PN2_LAUNCH_OK("train_max_all_finalize_kernel");
    return PN2_OK;
}

extern "C" int pn2_train_max_bwd_all(long long groups, long long k, int c, const float *gp, int gp_stride, int gp_offset,
                                     const int32_t *arg, float *g, void *stream) {
    PN2_REQUIRE(groups >= 0 && k >= 1 && k < (1ll << 31) && c >= 1, "train_max_bwd_all: bad dims groups=%lld k=%lld c=%d (1 <= k < 2^31)",
                groups, k, c);
    PN2_REQUIRE(gp_offset >= 0 && gp_stride >= gp_offset + c, "train_max_bwd_all: gp_stride=%d gp_offset=%d c=%d", gp_stride, gp_offset, c);
    if (groups == 0) return PN2_OK;
    PN2_REQUIRE(gp && arg && g, "train_max_bwd_all: null pointer");
    const long long total = groups * k * c;
    const unsigned grid = (unsigned)((total + 255) / 256 < 8ll * sm_count() ? (total + 255) / 256 : 8ll * sm_count());
    train_max_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(groups, k, c, gp, gp_stride, gp_offset, arg, g);
    PN2_LAUNCH_OK("train_max_bwd_kernel");
    return PN2_OK;
}
