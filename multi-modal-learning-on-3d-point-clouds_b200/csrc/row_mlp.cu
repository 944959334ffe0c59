// row_mlp.cu -- fused "gather -> shared MLP -> pool/store" blocks, fp32.
//
// Replaces, per set-abstraction scale (model/pointnet_util.py:37-41,101-109 / 152-166):
//     grouping_operation(xyz) + centre subtraction + grouping_operation(feat) + concat + permutes
//     + L x (Conv2d 1x1 -> BatchNorm2d(eval) -> ReLU) + max over nsample
// and per feature-propagation block (model/pointnet_util.py:209-220, model/pointnet2.py:158-159):
//     three_interpolate + concat + permutes + L x (Conv1d 1x1 -> BatchNorm1d(eval) -> ReLU)
//     (+ the head's conv1/bn1/relu/conv2 appended as two more layers)
// and per group_all SA layer (model/pointnet_util.py:50-67, 101-109):
//     concat [xyz | feat] + L x (Conv2d 1x1 -> BatchNorm2d(eval) -> ReLU) + max over all N points of a cloud
// which the reference runs as ~5 custom launches + ~8 layout copies + 3 x (cuDNN conv, BN, ReLU) +
// max, writing every intermediate activation to HBM (~100 MB per scene in sa1, SURVEY.md 8a A9).
//
// Here one CTA owns a tile of TR rows (a row = one (centroid, sample) pair, or one point).  The
// gathered input, every intermediate activation and the pooled result stay in shared memory; the
// only HBM traffic is the gathered input rows, the weights (L2 resident) and the final output.
// Activations are stored k-major ([channel][row], row stride TR+4) so that a thread's A fragment
// is one or two LDS.128 and its 8 interleaved output columns land conflict-free; weight k-chunks
// are staged through a double-buffered tile with their columns permuted to match.
// BatchNorm is folded into (W, bias) by the caller (eval mode), see pn2_b200/pointnet_util.py.
//
// fp32 FFMA throughout (the 1e-5 parity path).  The bf16 tcgen05 variant lives in row_mlp_tc.cu.
#include "common.cuh"
#include "row_mlp_tile.cuh"

namespace pn2 {
namespace {

enum { MODE_SA = 0, MODE_FP = 1, MODE_ALL = 2 };

struct RowMlpParams {
    int mode;
    int num_layers;
    int cin[PN2_MAX_LAYERS], cout[PN2_MAX_LAYERS], relu[PN2_MAX_LAYERS];
    const float *w[PN2_MAX_LAYERS];
    const float *bias[PN2_MAX_LAYERS];
    int buf_a_floats, buf_b_floats;  // ping / pong activation buffers (floats)
    // SA
    int n, m, k, d, order;
    long long groups;  // B*M
    const float *xyz, *feat, *new_xyz;
    const int32_t *idx;
    float *out;
    int out_stride, out_offset;
    // FP, ALL
    long long rows;  // B*n
    int d1, d2, fp_m;
    const float *feat1, *feat2, *weight;
};

template <int TR>
__device__ __forceinline__ void gather_sa(const RowMlpParams &p, float *x0, long long tile) {
    constexpr int TRP = TR + 4;
    const int K = p.k, D = p.d, C0 = 3 + D;
    const int gpt = TR / K;  // groups per tile
    const int xyz_off = p.order == PN2_ORDER_XYZ_FIRST ? 0 : D;
    const int feat_off = p.order == PN2_ORDER_XYZ_FIRST ? 3 : 0;
    const int cpad = round_up(C0, KC);
    if (C0 <= 16) {
        // few channels: consecutive threads take consecutive rows (conflict-free stores)
        for (int e = threadIdx.x; e < cpad * TR; e += RM_THREADS) {
            const int r = e % TR, c = e / TR;
            const long long g = tile * gpt + r / K;
            float v = 0.f;
            if (g < p.groups && c < C0) {
                const int b = (int)(g / p.m);
                const int pt = __ldg(p.idx + g * K + (r % K));
                const size_t src = (size_t)b * p.n + pt;
                if (c >= xyz_off && c < xyz_off + 3) {
                    const int a = c - xyz_off;
                    v = __fsub_rn(__ldg(p.xyz + src * 3 + a), __ldg(p.new_xyz + g * 3 + a));
                } else {
                    v = __ldg(p.feat + src * D + (c - feat_off));
                }
            }
            x0[(size_t)c * TRP + r] = v;
        }
    } else {
        // wide rows: one warp per row, lanes along the (contiguous, channel-last) feature row.  Lane i first loads the
        // sample index of row warp + NW * i (one round trip for the warp's rows); the row loop gets it by shuffle
        constexpr int NW = RM_THREADS / 32, RPW = TR / NW;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        long long m_src = -1;
        if (lane < RPW) {
            const int r = warp + NW * lane;
            const long long g = tile * gpt + r / K;
            if (g < p.groups) m_src = (g / p.m) * p.n + __ldg(p.idx + g * K + (r % K));
        }
#pragma unroll 2
        for (int i = 0; i < RPW; ++i) {
            const int r = warp + NW * i;
            const long long g = tile * gpt + r / K;
            const long long src_or = __shfl_sync(0xffffffffu, m_src, i);
            const bool ok = src_or >= 0;
            const size_t src = ok ? (size_t)src_or : 0;
            if (lane < 3)
                x0[(size_t)(xyz_off + lane) * TRP + r] =
                    ok ? __fsub_rn(__ldg(p.xyz + src * 3 + lane), __ldg(p.new_xyz + g * 3 + lane)) : 0.f;
            const float *f = p.feat + src * D;
#pragma unroll 4
            for (int c = lane; c < D; c += 32) x0[(size_t)(feat_off + c) * TRP + r] = ok ? __ldg(f + c) : 0.f;
            for (int c = C0 + lane; c < cpad; c += 32) x0[(size_t)c * TRP + r] = 0.f;
        }
    }
}

template <int TR>
__device__ __forceinline__ void gather_fp(const RowMlpParams &p, float *x0, long long tile) {
    constexpr int TRP = TR + 4;
    constexpr int NW = RM_THREADS / 32;
    constexpr int RPW = TR / NW;  // rows per warp: r = warp + NW * i
    static_assert(RPW >= 1 && RPW <= 32, "rows per warp");
    const int D1 = p.d1, D2 = p.d2, C0 = D1 + D2;
    const int cpad = round_up(C0, KC);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = p.n;
    const bool single = p.fp_m == 1;
    // index phase: lane i loads what row warp + NW * i needs (its three coarse rows and weights), so the whole warp pays
    // ONE round trip for its RPW rows; the row loop below gets them by shuffle and its feature loads depend on registers only
    // (one dependent index -> feature chain per row kept 16 round trips per warp on the critical path of the tile)
    long long m_row = -1;
    long long m_s0 = 0, m_s1 = 0, m_s2 = 0;  // element offsets of the coarse rows in feat2
    float m_w0 = 0.f, m_w1 = 0.f, m_w2 = 0.f;
    if (lane < RPW) {
        const long long row = tile * TR + warp + NW * lane;
        if (row < p.rows) {
            m_row = row;
            const long long b = row / n;
            if (single) {
                m_s0 = b * D2;  // S == 1: the single coarse feature row is repeated (model/pointnet_util.py:202-203)
            } else {
                const int32_t *id = p.idx + (size_t)row * 3;
                const float *w = p.weight + (size_t)row * 3;
                const long long base = b * p.fp_m;
                m_s0 = (base + __ldg(id)) * D2; m_s1 = (base + __ldg(id + 1)) * D2; m_s2 = (base + __ldg(id + 2)) * D2;
                m_w0 = __ldg(w); m_w1 = __ldg(w + 1); m_w2 = __ldg(w + 2);
            }
        }
    }
#pragma unroll 2
    for (int i = 0; i < RPW; ++i) {
        const int r = warp + NW * i;
        const long long row = __shfl_sync(0xffffffffu, m_row, i);
        const bool ok = row >= 0;
        if (D1 > 0) {
            const float *f1 = p.feat1 + (size_t)(ok ? row : 0) * D1;
            for (int c = lane; c < D1; c += 32) x0[(size_t)c * TRP + r] = ok ? __ldg(f1 + c) : 0.f;
        }
        const float *r0 = p.feat2 + __shfl_sync(0xffffffffu, m_s0, i);
        if (single) {
            for (int c = lane; c < D2; c += 32) x0[(size_t)(D1 + c) * TRP + r] = ok ? __ldg(r0 + c) : 0.f;
        } else {
            const float *r1 = p.feat2 + __shfl_sync(0xffffffffu, m_s1, i), *r2 = p.feat2 + __shfl_sync(0xffffffffu, m_s2, i);
            const float w0 = __shfl_sync(0xffffffffu, m_w0, i), w1 = __shfl_sync(0xffffffffu, m_w1, i), w2 = __shfl_sync(0xffffffffu, m_w2, i);
            // rows past the end carry offset 0 and weight 0: they read a valid row and store zeros
#pragma unroll 4
            for (int c = lane; c < D2; c += 32) {
                // same rounding sequence as three_interpolate (interpolate.cu)
                const float v = __fmaf_rn(w2, __ldg(r2 + c), __fmaf_rn(w0, __ldg(r0 + c), __fmul_rn(w1, __ldg(r1 + c))));
                x0[(size_t)(D1 + c) * TRP + r] = ok ? v : 0.f;
            }
        }
        for (int c = C0 + lane; c < cpad; c += 32) x0[(size_t)c * TRP + r] = 0.f;
    }
}

// group_all: row bb*n + i = [xyz[bb, i] | feat[bb, i]], read as it lies (no index list, no centring)
template <int TR>
__device__ __forceinline__ void gather_all(const RowMlpParams &p, float *x0, long long tile) {
    constexpr int TRP = TR + 4;
    const int D = p.d, C0 = 3 + D;
    const int cpad = round_up(C0, KC);
    if (C0 <= 16) {
        // few channels: consecutive threads take consecutive rows (conflict-free stores)
        for (int e = threadIdx.x; e < cpad * TR; e += RM_THREADS) {
            const int r = e % TR, c = e / TR;
            const long long row = tile * TR + r;
            float v = 0.f;
            if (row < p.rows && c < C0) v = c < 3 ? __ldg(p.xyz + row * 3 + c) : __ldg(p.feat + row * D + (c - 3));
            x0[(size_t)c * TRP + r] = v;
        }
    } else {
        // wide rows: one warp per row, lanes along the (contiguous, channel-last) feature row
        constexpr int NW = RM_THREADS / 32, RPW = TR / NW;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll 2
        for (int i = 0; i < RPW; ++i) {
            const int r = warp + NW * i;
            const long long row = tile * TR + r;
            const bool ok = row < p.rows;
            if (lane < 3) x0[(size_t)lane * TRP + r] = ok ? __ldg(p.xyz + row * 3 + lane) : 0.f;
            const float *f = p.feat + (ok ? row : 0) * D;
#pragma unroll 4
            for (int c = lane; c < D; c += 32) x0[(size_t)(3 + c) * TRP + r] = ok ? __ldg(f + c) : 0.f;
            for (int c = C0 + lane; c < cpad; c += 32) x0[(size_t)c * TRP + r] = 0.f;
        }
    }
}

template <int TR>
#ifndef PN2_RM_MINB
#define PN2_RM_MINB 2
#endif
__global__ void __launch_bounds__(RM_THREADS, PN2_RM_MINB) row_mlp_kernel(const __grid_constant__ RowMlpParams p) {
    constexpr int TRP = TR + 4;
    // shared memory layout: [ping: buf_a_floats][pong: buf_b_floats][weight tiles: 2*KC*WSP]
    extern __shared__ __align__(16) float smem[];
    // (the ping / pong pointers are computed as offsets from `smem`, not picked from a pointer array: an indexed
    // array of pointers lives in local memory and hides the address space, and every activation access of the layer
    // tiles became a generic LD.E / ST.E instead of LDS / STS)
    float *ws = smem + p.buf_a_floats + p.buf_b_floats;
    const long long tile = blockIdx.x;

    if (p.mode == MODE_SA)
        gather_sa<TR>(p, smem, tile);
    else if (p.mode == MODE_FP)
        gather_fp<TR>(p, smem, tile);
    else
        gather_all<TR>(p, smem, tile);
    __syncthreads();

    int cur = 0;  // which buffer holds the current layer's input
    for (int l = 0; l < p.num_layers; ++l) {
        const bool last = (l == p.num_layers - 1);
        const int cin = p.cin[l], cout = p.cout[l];
        const int nt = pick_nt(cout, TR);
        // A layer of ONE n-tile writes its output over its input: every read of the input is behind the barrier that ends
        // the tile's k loop, and the epilogue stores come after it.  Stacks of such layers (fp1 + head, sa1, sa2) need no
        // pong buffer, which is what lets two CTAs share an SM.  Wider layers write to the other buffer (make_layout).
        const bool in_place = cout <= nt;
        const float *xin = smem + (cur ? p.buf_a_floats : 0);
        float *xout = smem + ((cur != 0) == in_place ? p.buf_a_floats : 0);
        if (!in_place) cur ^= 1;
        for (int n0 = 0; n0 < cout; n0 += nt) {
            const int ch0 = last ? 0 : n0;
            if (nt == 128)
                layer_tile<TR, 128>(xin, xout, ch0, p.w[l], p.bias[l], cin, cout, n0, p.relu[l], ws);
            else if (nt == 64)
                layer_tile<TR, 64>(xin, xout, ch0, p.w[l], p.bias[l], cin, cout, n0, p.relu[l], ws);
            else if constexpr (TR != 16)
                layer_tile<TR, 32>(xin, xout, ch0, p.w[l], p.bias[l], cin, cout, n0, p.relu[l], ws);
            if (!last) continue;
            __syncthreads();
            const int nv = min(nt, cout - n0);  // valid columns of this n-tile
            if (p.mode == MODE_SA) {
                // max over the K rows of each group (torch.max(new_points, 2)[0], pointnet_util.py:109)
                const int K = p.k, gpt = TR / K;
                for (int e = threadIdx.x; e < gpt * nv; e += RM_THREADS) {
                    const int col = e % nv, gl = e / nv;
                    const long long g = tile * gpt + gl;
                    if (g >= p.groups) continue;
                    const float *src = xout + (size_t)col * TRP + gl * K;
                    float mx = src[0];
                    for (int s = 1; s < K; ++s) mx = fmaxf(mx, src[s]);
                    p.out[(size_t)g * p.out_stride + p.out_offset + n0 + col] = mx;
                }
            } else if (p.mode == MODE_ALL) {
                // max over the rows of each cloud in this tile (a tile may end one cloud and start the next, or hold
                // many clouds when n < TR), combined across tiles by an integer atomicMax on the bits: the last layer
                // has a ReLU, so every value is a non-negative float whose bit pattern orders like the value (out was
                // zeroed first; -0 has the sign bit and loses to +0).  Max is exact: the result does not depend on the
                // order in which the CTAs finish.
                const long long r0 = tile * TR, r1 = min(r0 + TR, p.rows);
                const long long cl0 = r0 / p.n;
                const int ncl = (int)((r1 - 1) / p.n - cl0) + 1;
                for (int e = threadIdx.x; e < ncl * nv; e += RM_THREADS) {
                    const int col = e % nv;
                    const long long cl = cl0 + e / nv;
                    const int lo = (int)(max(cl * p.n, r0) - r0), hi = (int)(min((cl + 1) * p.n, r1) - r0);
                    const float *src = xout + (size_t)col * TRP;
                    float mx = src[lo];
                    for (int s = lo + 1; s < hi; ++s) mx = fmaxf(mx, src[s]);
                    atomicMax(reinterpret_cast<int *>(p.out) + (size_t)cl * p.out_stride + p.out_offset + n0 + col, __float_as_int(mx));
                }
            } else {
                for (int e = threadIdx.x; e < TR * nv; e += RM_THREADS) {
                    const int col = e % nv, r = e / nv;
                    const long long row = tile * TR + r;
                    if (row >= p.rows) continue;
                    p.out[(size_t)row * cout + n0 + col] = xout[(size_t)col * TRP + r];
                }
            }
            __syncthreads();
        }
        // layer_tile ends with a barrier after its last chunk, but its epilogue stores come after
        // that barrier: make them visible before the next layer reads them.
        __syncthreads();
    }
}

// out[r*stride + offset + ch] = 0 for r < rows, ch < c: the start value of the group_all pooling's atomicMax
__global__ void __launch_bounds__(256) zero_cols_kernel(long long rows, int c, float *out, int stride, int offset) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < rows * c; e += (long long)gridDim.x * 256) {
        const long long r = e / c;
        out[r * stride + offset + (e - r * c)] = 0.f;
    }
}

struct Layout {
    int buf_a, buf_b;  // floats
    size_t bytes;
};

Layout make_layout(int tr, int c0, const pn2_mlp *mlp) {
    // mirrors the buffer walk of row_mlp_kernel: single-n-tile layers run in place, wider ones flip buffers
    const int trp = tr + 4;
    int need[2] = {round_up(c0, KC) * trp, 0};
    int cur = 0;
    for (int l = 0; l < mlp->num_layers; ++l) {
        const int nt = pick_nt(mlp->cout[l], tr);
        const bool in_place = mlp->cout[l] <= nt;
        // the last layer hands one n-tile at a time to the pool / store step
        const int ch = (l == mlp->num_layers - 1) ? nt : round_up(mlp->cout[l], nt);
        if (!in_place) cur ^= 1;
        need[cur] = need[cur] > ch * trp ? need[cur] : ch * trp;
        // inputs are read up to round_up(cin, KC) channels only through kk_end, no extra space needed
    }
    Layout L;
    L.buf_a = need[0];
    L.buf_b = need[1];
    L.bytes = (size_t)(need[0] + need[1] + 2 * KC * WSP) * sizeof(float);
    return L;
}

constexpr size_t SMEM_LIMIT = 227 * 1024;

int check_mlp(const char *op, const pn2_mlp *mlp, int c0) {
    PN2_REQUIRE(mlp, "%s: null mlp", op);
    PN2_REQUIRE(mlp->num_layers >= 1 && mlp->num_layers <= PN2_MAX_LAYERS, "%s: num_layers %d outside 1..%d", op,
                mlp->num_layers, PN2_MAX_LAYERS);
    int c = c0;
    for (int l = 0; l < mlp->num_layers; ++l) {
        PN2_REQUIRE(mlp->cin[l] == c, "%s: layer %d expects cin=%d but the previous stage produces %d", op, l, mlp->cin[l], c);
        PN2_REQUIRE(mlp->cout[l] >= 1, "%s: layer %d has cout=%d", op, l, mlp->cout[l]);
        PN2_REQUIRE(mlp->weight[l] && mlp->bias[l], "%s: layer %d has a null weight or bias", op, l);
        c = mlp->cout[l];
    }
    return PN2_OK;
}

template <int TR>
int launch(const RowMlpParams &p, const Layout &L, long long tiles, cudaStream_t s) {
    PN2_REQUIRE(tiles <= 2147483647ll, "row_mlp: too many tiles");
    PN2_CUDA(cudaFuncSetAttribute(row_mlp_kernel<TR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.bytes));
    row_mlp_kernel<TR><<<(unsigned)tiles, RM_THREADS, L.bytes, s>>>(p);
    PN2_LAUNCH_OK("row_mlp_kernel");
    return PN2_OK;
}

// Picks the largest row tile whose buffers fit in shared memory, then shrinks it while the grid
// would leave SMs idle.
int dispatch(RowMlpParams &p, const pn2_mlp *mlp, int c0, long long total_rows, int min_tr, cudaStream_t s) {
    const int cands[4] = {128, 64, 32, 16};
    int chosen = -1;
    for (int i = 0; i < 4; ++i) {
        const int tr = cands[i];
        if (tr < min_tr || tr % min_tr) continue;
        if (make_layout(tr, c0, mlp).bytes > SMEM_LIMIT) continue;
        chosen = tr;
        const long long tiles = (total_rows + tr - 1) / tr;
        if (tiles >= 2ll * sm_count() || tr <= 32) break;  // enough CTAs; otherwise try a smaller tile (16 only if nothing else fits)
    }
    if (chosen < 0)
        return set_error(PN2_ERR_UNSUPPORTED, "row_mlp: channel widths need more than %zu bytes of shared memory", SMEM_LIMIT);
    const Layout L = make_layout(chosen, c0, mlp);
    p.buf_a_floats = L.buf_a;
    p.buf_b_floats = L.buf_b;
    const long long tiles = (total_rows + chosen - 1) / chosen;
    switch (chosen) {
        case 128: return launch<128>(p, L, tiles, s);
        case 64: return launch<64>(p, L, tiles, s);
        case 32: return launch<32>(p, L, tiles, s);
        default: return launch<16>(p, L, tiles, s);
    }
}

void copy_mlp(RowMlpParams &p, const pn2_mlp *mlp) {
    p.num_layers = mlp->num_layers;
    for (int l = 0; l < mlp->num_layers; ++l) {
        p.cin[l] = mlp->cin[l];
        p.cout[l] = mlp->cout[l];
        p.relu[l] = mlp->relu[l];
        p.w[l] = mlp->weight[l];
        p.bias[l] = mlp->bias[l];
    }
}

}  // namespace
}  // namespace pn2

// 1 when pn2_sa_mlp_max (nsample > 0) / pn2_fp_mlp and pn2_sa_all_mlp_max (nsample == 0: the same row tiles and shared
// memory layout; pn2_sa_all_mlp_max also needs a ReLU on the last layer) can run this stack with `c0` input channels: the
// callers (pn2_b200/pointnet_util.py::_fusable) use the reference's operator composition otherwise, so a module that
// trains on the composed path never fails at eval time for its shape alone.
extern "C" int pn2_mlp_fp32_supported(const pn2_mlp *mlp, int c0, int nsample) {
    using namespace pn2;
    if (!mlp || mlp->num_layers < 1 || mlp->num_layers > PN2_MAX_LAYERS || c0 < 1 || mlp->cin[0] != c0) return 0;
    const int k = nsample;
    if (k < 0 || (k > 0 && !(k == 1 || k == 2 || k == 4 || k == 8 || k == 16 || k == 32 || k == 64 || k == 128))) return 0;
    const int min_tr = k < 16 ? 16 : k;
    const int cands[4] = {128, 64, 32, 16};
    for (int i = 0; i < 4; ++i)
        if (cands[i] >= min_tr && cands[i] % min_tr == 0 && make_layout(cands[i], c0, mlp).bytes <= SMEM_LIMIT) return 1;
    return 0;
}

extern "C" int pn2_sa_mlp_max(int b, int n, int m, int k, int d, const float *xyz, const float *feat, const float *new_xyz,
                              const int32_t *idx, int order, const pn2_mlp *mlp, float *out, int out_stride,
                              int out_offset, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && n >= 1 && m >= 0 && k >= 1 && d >= 0, "sa_mlp_max: bad dims b=%d n=%d m=%d k=%d d=%d", b, n, m, k, d);
    PN2_REQUIRE(order == PN2_ORDER_XYZ_FIRST || order == PN2_ORDER_FEAT_FIRST, "sa_mlp_max: unknown concat order %d", order);
    if (int st = check_mlp("sa_mlp_max", mlp, 3 + d)) return st;
    if (b == 0 || m == 0) return PN2_OK;
    PN2_REQUIRE(xyz && new_xyz && idx && out && (feat || d == 0), "sa_mlp_max: null pointer");
    const int cl = mlp->cout[mlp->num_layers - 1];
    PN2_REQUIRE(out_offset >= 0 && out_stride >= out_offset + cl, "sa_mlp_max: out_stride/out_offset do not hold %d channels", cl);
    if (!(k == 1 || k == 2 || k == 4 || k == 8 || k == 16 || k == 32 || k == 64 || k == 128))
        return set_error(PN2_ERR_UNSUPPORTED, "sa_mlp_max: nsample must be a power of two <= 128 (got %d)", k);
    RowMlpParams p = {};
    p.mode = MODE_SA;
    copy_mlp(p, mlp);
    p.n = n; p.m = m; p.k = k; p.d = d; p.order = order;
    p.groups = (long long)b * m;
    p.xyz = xyz; p.feat = feat; p.new_xyz = new_xyz; p.idx = idx;
    p.out = out; p.out_stride = out_stride; p.out_offset = out_offset;
    return dispatch(p, mlp, 3 + d, p.groups * k, k < 16 ? 16 : k, (cudaStream_t)stream);
}

extern "C" int pn2_fp_mlp(int b, int n, int m, int d1, int d2, const float *feat1, const float *feat2, const int32_t *idx,
                          const float *weight, const pn2_mlp *mlp, float *out, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && n >= 0 && m >= 1 && d1 >= 0 && d2 >= 1, "fp_mlp: bad dims b=%d n=%d m=%d d1=%d d2=%d", b, n, m, d1, d2);
    if (int st = check_mlp("fp_mlp", mlp, d1 + d2)) return st;
    if (b == 0 || n == 0) return PN2_OK;
    PN2_REQUIRE(feat2 && out && (feat1 || d1 == 0) && (m == 1 || (idx && weight)), "fp_mlp: null pointer");
    RowMlpParams p = {};
    p.mode = MODE_FP;
    copy_mlp(p, mlp);
    p.n = n; p.fp_m = m; p.d1 = d1; p.d2 = d2;
    p.rows = (long long)b * n;
    p.feat1 = feat1; p.feat2 = feat2; p.idx = idx; p.weight = weight;
    p.out = out;
    return dispatch(p, mlp, d1 + d2, p.rows, 16, (cudaStream_t)stream);
}

extern "C" int pn2_sa_all_mlp_max(int b, int n, int d, const float *xyz, const float *feat, const pn2_mlp *mlp, float *out,
                                  int out_stride, int out_offset, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && n >= 1 && d >= 0, "sa_all_mlp_max: bad dims b=%d n=%d d=%d", b, n, d);
    if (int st = check_mlp("sa_all_mlp_max", mlp, 3 + d)) return st;
    const int cl = mlp->cout[mlp->num_layers - 1];
    PN2_REQUIRE(out_offset >= 0 && out_stride >= out_offset + cl, "sa_all_mlp_max: out_stride/out_offset do not hold %d channels", cl);
    if (!mlp->relu[mlp->num_layers - 1])
        return set_error(PN2_ERR_UNSUPPORTED, "sa_all_mlp_max: the last layer needs a ReLU (the pooling combines non-negative values)");
    if (b == 0) return PN2_OK;
    PN2_REQUIRE(xyz && out && (feat || d == 0), "sa_all_mlp_max: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    const long long total = (long long)b * cl;
    const unsigned zgrid = (unsigned)((total + 255) / 256 < 8ll * sm_count() ? (total + 255) / 256 : 8ll * sm_count());
    zero_cols_kernel<<<zgrid, 256, 0, s>>>(b, cl, out, out_stride, out_offset);
    PN2_LAUNCH_OK("zero_cols_kernel");
    RowMlpParams p = {};
    p.mode = MODE_ALL;
    copy_mlp(p, mlp);
    p.n = n; p.d = d;
    p.rows = (long long)b * n;
    p.xyz = xyz; p.feat = feat;
    p.out = out; p.out_stride = out_stride; p.out_offset = out_offset;
    return dispatch(p, mlp, 3 + d, p.rows, 16, s);
}
