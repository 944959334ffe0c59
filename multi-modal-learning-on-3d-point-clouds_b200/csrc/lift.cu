// lift.cu -- multi-view 2D->3D feature lifting in one launch per batch.
//
// Replaces, per (cloud, view): ProjectionHelper.compute_projection (utils/projection.py:166-230,
// ~25 small torch ops and >= 4 host<->device round trips), Projection.forward (:237-256) and the
// per-sample view reduction of PointNet2Multiview* (model/pointnet2multiview.py:30-43, 83-102).
//
// Per point and view (SURVEY.md A.8/A.9): six frustum planes with round(100*s)/100 < 0; camera
// transform; pinhole projection (multiply, divide, add); round-half-even to the NEAREST pixel (no
// interpolation, utils/projection.py:204); bounds; depth-range and |depth - z| <= accuracy tests;
// then the C-channel feature column of that pixel is fetched and reduced over views (max with
// zeros for invisible views, or first view whose column is not all-zero).
//
// fp32 evaluation order (the reference leaves it to BLAS): dot products are
// fma(c, z, fma(b, y, rn(a*x))) (+ rn add of the translation); identical in oracle/pn2_oracle.c.
#include "common.cuh"

namespace pn2 {
namespace {

constexpr int LV_THREADS = 256;
constexpr int LV_MAXV = 8;

struct CamCorners {
    float p[8][3];  // depth_to_skeleton of the four image corners at depth_min (0-3) and depth_max (4-7), utils/projection.py:37-44
};

struct ViewParams {  // 38 floats per view, staged in shared memory
    float w2c[12];   // rows 0..2 of world_to_camera
    float c2[3], c4[3];
    float nrm[18];
};

// Geometry half of the per-(point, view) test: frustum planes, projection, nearest pixel.  Returns the pixel or -1 and the
// camera-space depth; the depth-map test (project_depth_ok) needs one dependent random load and is kept apart so that a
// caller can put the loads of all views in flight before the first comparison.
__device__ __forceinline__ int project_pixel(float px, float py, float pz, const ViewParams &vp, float fx, float fy, float cx,
                                             float cy, int W, int H, float &cam_z) {
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const float *c = k < 3 ? vp.c2 : vp.c4;
        const float dx = __fsub_rn(px, c[0]), dy = __fsub_rn(py, c[1]), dz = __fsub_rn(pz, c[2]);
        const float s = __fmaf_rn(dz, vp.nrm[3 * k + 2], __fmaf_rn(dy, vp.nrm[3 * k + 1], __fmul_rn(dx, vp.nrm[3 * k])));
        // round(100 s) / 100 < 0 (utils/projection.py:115): dividing the integer-valued k = rint(100 s) by +100 keeps its
        // sign (-0.0 / 100 = -0.0, NaN stays NaN, |k| >= 1 cannot underflow), so the test is exactly k < 0 -- no IEEE division
        const float r = rintf(__fmul_rn(s, 100.0f));
        if (!(r < 0.0f)) return -1;
    }
    float cam[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float *m = vp.w2c + 4 * r;
        cam[r] = __fadd_rn(__fmaf_rn(m[2], pz, __fmaf_rn(m[1], py, __fmul_rn(m[0], px))), m[3]);
    }
    const float u = __fadd_rn(__fdiv_rn(__fmul_rn(cam[0], fx), cam[2]), cx);
    const float v = __fadd_rn(__fdiv_rn(__fmul_rn(cam[1], fy), cam[2]), cy);
    const float ur = rintf(u), vr = rintf(v);
    if (!(ur >= 0.0f && vr >= 0.0f && ur < (float)W && vr < (float)H)) return -1;
    cam_z = cam[2];
    return (int)vr * W + (int)ur;
}
__device__ __forceinline__ bool project_depth_ok(float z, float cam_z, float dmin, float dmax, float acc) {
    return z >= dmin && z <= dmax && fabsf(__fsub_rn(z, cam_z)) <= acc;
}
__device__ __forceinline__ int project_point(float px, float py, float pz, const ViewParams &vp, float fx, float fy,
                                             float cx, float cy, int W, int H, const float *__restrict__ depth,
                                             float dmin, float dmax, float acc) {
    float cam_z = 0.f;
    const int pix = project_pixel(px, py, pz, vp, fx, fy, cx, cy, W, H, cam_z);
    if (pix < 0) return -1;
    return project_depth_ok(__ldg(depth + pix), cam_z, dmin, dmax, acc) ? pix : -1;
}

__global__ void __launch_bounds__(LV_THREADS)
lift_views_kernel(int n, int nv, int c, int h, int w, const float *__restrict__ points, const float *__restrict__ feats,
                  const float *__restrict__ depth, const float *__restrict__ w2c, const float *__restrict__ corner2,
                  const float *__restrict__ corner4, const float *__restrict__ normals, float fx, float fy, float cx,
                  float cy, float dmin, float dmax, float acc, int reduce, float *__restrict__ out,
                  int32_t *__restrict__ pix_out, int32_t *__restrict__ count) {
    __shared__ ViewParams vps[LV_MAXV];
    __shared__ int vcount[LV_MAXV];
    const int b = blockIdx.y;
    const int hw = h * w;
    if (threadIdx.x < nv) {
        const size_t bv = (size_t)b * nv + threadIdx.x;
        ViewParams &vp = vps[threadIdx.x];
        for (int k = 0; k < 12; ++k) vp.w2c[k] = w2c[bv * 16 + k];
        for (int k = 0; k < 3; ++k) {
            vp.c2[k] = corner2[bv * 3 + k];
            vp.c4[k] = corner4[bv * 3 + k];
        }
        for (int k = 0; k < 18; ++k) vp.nrm[k] = normals[bv * 18 + k];
        vcount[threadIdx.x] = 0;
    }
    __syncthreads();
    const int i = blockIdx.x * LV_THREADS + threadIdx.x;
    const bool live = i < n;
    int pix[LV_MAXV];
    if (live) {
        const float *p = points + ((size_t)b * n + i) * 3;
        const float px = p[0], py = p[1], pz = p[2];
#pragma unroll
        for (int v = 0; v < LV_MAXV; ++v) {
            pix[v] = -1;
            if (v < nv) {
                const size_t bv = (size_t)b * nv + v;
                pix[v] = project_point(px, py, pz, vps[v], fx, fy, cx, cy, w, h, depth + bv * hw, dmin, dmax, acc);
                if (pix_out) pix_out[bv * n + i] = pix[v];
                if (count && pix[v] >= 0) atomicAdd(&vcount[v], 1);
            }
        }
    }
    if (count) {
        __syncthreads();
        if (threadIdx.x < nv && vcount[threadIdx.x]) atomicAdd(count + (size_t)b * nv + threadIdx.x, vcount[threadIdx.x]);
    }
    if (!live) return;
    float *o = out + (size_t)b * c * n + i;
    if (reduce == PN2_REDUCE_MAX) {
        // F.max_pool1d over the stacked per-view maps: invisible views contribute zeros
        for (int ch = 0; ch < c; ++ch) {
            float best = 0.f;
            bool any = false;
#pragma unroll
            for (int v = 0; v < LV_MAXV; ++v) {
                if (v < nv) {
                    const float f = pix[v] >= 0 ? __ldg(feats + (((size_t)b * nv + v) * c + ch) * hw + pix[v]) : 0.f;
                    best = any ? fmaxf(best, f) : f;
                    any = true;
                }
            }
            __stcs(o + (size_t)ch * n, best);
        }
    } else {
        bool have = false;
#pragma unroll
        for (int v = 0; v < LV_MAXV; ++v) {
            if (v < nv && !have && pix[v] >= 0) {
                const float *f = feats + ((size_t)b * nv + v) * c * hw + pix[v];
                bool nz = false;
                for (int ch = 0; ch < c; ++ch) {
                    const float val = __ldg(f + (size_t)ch * hw);
                    nz = nz || (val != 0.f);
                    o[(size_t)ch * n] = val;
                }
                have = nz;
                // a visible but all-zero column stays replaceable by a later view (pointnet2multiview.py:97)
                if (!nz) have = false;
            }
        }
        bool wrote = false;
#pragma unroll
        for (int v = 0; v < LV_MAXV; ++v) wrote = wrote || (v < nv && pix[v] >= 0);
        if (!wrote)
            for (int ch = 0; ch < c; ++ch) o[(size_t)ch * n] = 0.f;
    }
}

// ---- per-view parameters in one launch ------------------------------------------------------------------------
// The reference derives them per (scene, view) with ~25 small torch ops (utils/projection.py:25-95, 178): inverse of the
// pose, eight frustum corners = pose x camera-space corners, six plane normals = cross products of corner differences.
// One thread per view here.  The inverse is evaluated in fp64 (adjugate) and rounded once -- torch.inverse is an fp32 LU
// whose low bits depend on the backend, so agreement is to ~1 ulp, not bitwise; corners and normals are fp32 with one
// rounding per operation.

// One view: pose (16 floats, row-major) -> world_to_camera (16), frustum corners 2 and 4 (3 each), six plane normals (18).
__device__ __forceinline__ void compute_view_params(const float *__restrict__ m, const CamCorners &cam, float *__restrict__ w,
                                                    float *__restrict__ corner2, float *__restrict__ corner4, float *__restrict__ normals) {
    double a[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = (double)m[k];
    // general 4x4 inverse by the adjugate (2x2 sub-determinants)
    const double s0 = a[0] * a[5] - a[4] * a[1], s1 = a[0] * a[6] - a[4] * a[2], s2 = a[0] * a[7] - a[4] * a[3];
    const double s3 = a[1] * a[6] - a[5] * a[2], s4 = a[1] * a[7] - a[5] * a[3], s5 = a[2] * a[7] - a[6] * a[3];
    const double c5 = a[10] * a[15] - a[14] * a[11], c4 = a[9] * a[15] - a[13] * a[11], c3 = a[9] * a[14] - a[13] * a[10];
    const double c2 = a[8] * a[15] - a[12] * a[11], c1 = a[8] * a[14] - a[12] * a[10], c0 = a[8] * a[13] - a[12] * a[9];
    const double inv = 1.0 / (s0 * c5 - s1 * c4 + s2 * c3 + s3 * c2 - s4 * c1 + s5 * c0);
    w[0] = (float)((a[5] * c5 - a[6] * c4 + a[7] * c3) * inv);
    w[1] = (float)((-a[1] * c5 + a[2] * c4 - a[3] * c3) * inv);
    w[2] = (float)((a[13] * s5 - a[14] * s4 + a[15] * s3) * inv);
    w[3] = (float)((-a[9] * s5 + a[10] * s4 - a[11] * s3) * inv);
    w[4] = (float)((-a[4] * c5 + a[6] * c2 - a[7] * c1) * inv);
    w[5] = (float)((a[0] * c5 - a[2] * c2 + a[3] * c1) * inv);
    w[6] = (float)((-a[12] * s5 + a[14] * s2 - a[15] * s1) * inv);
    w[7] = (float)((a[8] * s5 - a[10] * s2 + a[11] * s1) * inv);
    w[8] = (float)((a[4] * c4 - a[5] * c2 + a[7] * c0) * inv);
    w[9] = (float)((-a[0] * c4 + a[1] * c2 - a[3] * c0) * inv);
    w[10] = (float)((a[12] * s4 - a[13] * s2 + a[15] * s0) * inv);
    w[11] = (float)((-a[8] * s4 + a[9] * s2 - a[11] * s0) * inv);
    w[12] = (float)((-a[4] * c3 + a[5] * c1 - a[6] * c0) * inv);
    w[13] = (float)((a[0] * c3 - a[1] * c1 + a[2] * c0) * inv);
    w[14] = (float)((-a[12] * s3 + a[13] * s1 - a[14] * s0) * inv);
    w[15] = (float)((a[8] * s3 - a[9] * s1 + a[10] * s0) * inv);
    // world-space corners: rows 0..2 of pose x (x, y, z, 1)
    float cw[8][3];
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int r = 0; r < 3; ++r)
            cw[k][r] = __fadd_rn(__fmaf_rn(m[4 * r + 2], cam.p[k][2], __fmaf_rn(m[4 * r + 1], cam.p[k][1], __fmul_rn(m[4 * r], cam.p[k][0]))),
                                 m[4 * r + 3]);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        corner2[r] = cw[2][r];
        corner4[r] = cw[4][r];
    }
    // inward normals (utils/projection.py:66-93): cross(c[a1] - c[a0], c[b1] - c[b0])
    const int A0[6] = {0, 1, 2, 3, 0, 5}, A1[6] = {3, 2, 3, 0, 1, 6}, B0[6] = {0, 1, 2, 3, 0, 5}, B1[6] = {1, 5, 6, 7, 4, 4};
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        float u[3], v[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            u[r] = __fsub_rn(cw[A1[k]][r], cw[A0[k]][r]);
            v[r] = __fsub_rn(cw[B1[k]][r], cw[B0[k]][r]);
        }
        float *nk = normals + 3 * k;
        nk[0] = __fsub_rn(__fmul_rn(u[1], v[2]), __fmul_rn(u[2], v[1]));
        nk[1] = __fsub_rn(__fmul_rn(u[2], v[0]), __fmul_rn(u[0], v[2]));
        nk[2] = __fsub_rn(__fmul_rn(u[0], v[1]), __fmul_rn(u[1], v[0]));
    }
}

__global__ void lift_setup_kernel(int nviews, const float *__restrict__ c2w_all, CamCorners cam, float *__restrict__ w2c_all,
                                  float *__restrict__ corner2, float *__restrict__ corner4, float *__restrict__ normals) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nviews) return;
    compute_view_params(c2w_all + (size_t)t * 16, cam, w2c_all + (size_t)t * 16, corner2 + (size_t)t * 3, corner4 + (size_t)t * 3,
                        normals + (size_t)t * 18);
}

// ---- staged path (the default): project once, then stream the feature maps through shared memory ----------------
// The single-kernel form above fetches every (point, view, channel) value as its own 32-byte sector from a channel-major
// map (stride H*W floats between channels): 8x read amplification and, measured, 4 % of the HBM roofline.  Staged:
//   lift_nonzero_kernel  (REDUCE_FIRST only) flags, per (cloud, view, pixel), whether the C-channel column is non-zero;
//   lift_project_kernel  projects every point into every view once -> pix (b,v,n), count, and for REDUCE_FIRST the view
//                        each point takes its column from (first visible view with a non-zero column);
//   lift_gather_kernel   one CTA per (cloud, chunk of CH channels): the chunk's slab of ALL views (V x CH x H*W floats,
//                        contiguous per view) is copied to shared memory with coalesced 128-bit loads, then every point
//                        reads its pixels from the slab and the warp writes 32 consecutive points per channel.
// Feature maps are read once (twice for REDUCE_FIRST), the output is written once, both coalesced.
__global__ void __launch_bounds__(256)
lift_nonzero_kernel(int c, int hw, const float *__restrict__ feats, unsigned char *__restrict__ nz) {
    const int px = blockIdx.x * 256 + threadIdx.x;
    if (px >= hw) return;
    const size_t bv = blockIdx.y;
    const float *f = feats + bv * c * hw + px;
    bool any = false;
    for (int ch = 0; ch < c; ++ch) any = any || (__ldg(f + (size_t)ch * hw) != 0.f);
    nz[bv * hw + px] = any ? 1 : 0;
}

__global__ void __launch_bounds__(LV_THREADS, 4)  // 64 registers: the dependent round trip per point is hidden by resident warps
lift_project_kernel(int n, int nv, int h, int w, const float *__restrict__ points, const float *__restrict__ depth,
                    const float *__restrict__ w2c, const float *__restrict__ corner2, const float *__restrict__ corner4,
                    const float *__restrict__ normals, const float *__restrict__ c2w, CamCorners cam, float fx, float fy, float cx,
                    float cy, float dmin, float dmax, float acc, const unsigned char *__restrict__ nz, int32_t *__restrict__ pix_out,
                    int16_t *__restrict__ pix16, signed char *__restrict__ sel, int32_t *__restrict__ count) {
    __shared__ ViewParams vps[LV_MAXV];
    __shared__ int vcount[LV_MAXV];
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the gather kernel may start its (independent) slab fill
    const int b = blockIdx.y;
    const int hw = h * w;
    if (threadIdx.x < nv) {
        const size_t bv = (size_t)b * nv + threadIdx.x;
        ViewParams &vp = vps[threadIdx.x];
        if (c2w) {
            // per-view parameters straight from the poses (what pn2_lift_setup computes, same device function -> same bits):
            // saves a launch in front of every lifting call
            float wfull[16];
            compute_view_params(c2w + bv * 16, cam, wfull, vp.c2, vp.c4, vp.nrm);
            for (int k = 0; k < 12; ++k) vp.w2c[k] = wfull[k];
        } else {
            for (int k = 0; k < 12; ++k) vp.w2c[k] = w2c[bv * 16 + k];
            for (int k = 0; k < 3; ++k) {
                vp.c2[k] = corner2[bv * 3 + k];
                vp.c4[k] = corner4[bv * 3 + k];
            }
            for (int k = 0; k < 18; ++k) vp.nrm[k] = normals[bv * 18 + k];
        }
        vcount[threadIdx.x] = 0;
    }
    __syncthreads();
    const int i = blockIdx.x * LV_THREADS + threadIdx.x;
    const bool live = i < n;
    // phase 1: geometry of every view; phase 2: the depth values of all candidate pixels are loaded together (one
    // dependent round trip per point instead of one per view -- the kernel is bound by that latency: ncu showed the depth
    // comparison as its largest stall); phase 3: depth tests, outputs
    int cand[LV_MAXV];
    float camz[LV_MAXV], zv[LV_MAXV];
    float px = 0.f, py = 0.f, pz = 0.f;
    if (live) {
        const float *p = points + ((size_t)b * n + i) * 3;
        px = p[0]; py = p[1]; pz = p[2];
    }
#pragma unroll
    for (int v = 0; v < LV_MAXV; ++v) {
        cand[v] = -1;
        camz[v] = 0.f;
        if (v < nv && live) cand[v] = project_pixel(px, py, pz, vps[v], fx, fy, cx, cy, w, h, camz[v]);
    }
#pragma unroll
    for (int v = 0; v < LV_MAXV; ++v) {
        zv[v] = 0.f;
        if (v < nv && cand[v] >= 0) zv[v] = __ldg(depth + ((size_t)b * nv + v) * hw + cand[v]);
    }
    int chosen = -1;
#pragma unroll
    for (int v = 0; v < LV_MAXV; ++v) {
        if (v < nv) {
            const size_t bv = (size_t)b * nv + v;
            const int pix = (cand[v] >= 0 && project_depth_ok(zv[v], camz[v], dmin, dmax, acc)) ? cand[v] : -1;
            if (live) {
                if (pix_out) pix_out[bv * n + i] = pix;
                if (pix16) pix16[bv * n + i] = (int16_t)pix;  // what the gather kernel reads: half the index traffic (hw < 32768)
            }
            if (count) {  // one shared-memory atomic per warp and view
                const unsigned m = __ballot_sync(0xffffffffu, pix >= 0);
                if ((threadIdx.x & 31) == 0 && m) atomicAdd(&vcount[v], __popc(m));
            }
            // first view, then only views that fill an all-zero column (model/pointnet2multiview.py:93-98)
            if (sel && chosen < 0 && pix >= 0 && nz[bv * hw + pix]) chosen = v;
        }
    }
    if (live && sel) sel[(size_t)b * n + i] = (signed char)chosen;
    if (count) {
        __syncthreads();
        if (threadIdx.x < nv && vcount[threadIdx.x]) atomicAdd(count + (size_t)b * nv + threadIdx.x, vcount[threadIdx.x]);
    }
}

constexpr int LG_THREADS = 512;

template <int CH>
__global__ void __launch_bounds__(LG_THREADS)
lift_gather_kernel(int n, int nv, int c, int hw, const float *__restrict__ feats, const int32_t *__restrict__ pix,
                   const signed char *__restrict__ sel, float *__restrict__ out) {
    extern __shared__ __align__(16) float slab[];  // [nv][CH][hw]
    const int b = blockIdx.y;
    const int c0 = blockIdx.x * CH;
    const int cc = min(CH, c - c0);
    for (int v = 0; v < nv; ++v) {
        const float *src = feats + (((size_t)b * nv + v) * c + c0) * hw;  // cc * hw contiguous floats
        float *dst = slab + (size_t)v * CH * hw;
        const int total = cc * hw;
        if (((uintptr_t)src & 15) == 0 && (total & 3) == 0 && ((CH * hw) & 3) == 0) {
            for (int e = threadIdx.x; e < total / 4; e += LG_THREADS)
                reinterpret_cast<float4 *>(dst)[e] = __ldcs(reinterpret_cast<const float4 *>(src) + e);
        } else {
            for (int e = threadIdx.x; e < total; e += LG_THREADS) dst[e] = __ldcs(src + e);
        }
    }
    __syncthreads();
    float *o = out + ((size_t)b * c + c0) * n;
    const int32_t *pb = pix + (size_t)b * nv * n;
    if ((n & 3) == 0 && ((uintptr_t)o & 15) == 0 && ((uintptr_t)pb & 15) == 0) {
        // four consecutive points per thread: 128-bit pixel-index loads and 128-bit streaming stores per channel
        const int n4 = n >> 2;
        for (int i4 = threadIdx.x; i4 < n4; i4 += LG_THREADS) {
            float r[CH][4];
#pragma unroll
            for (int q = 0; q < CH; ++q) r[q][0] = r[q][1] = r[q][2] = r[q][3] = 0.f;
            if (sel) {
                const char4 sv = *reinterpret_cast<const char4 *>(sel + (size_t)b * n + 4 * i4);
                const int vs[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (vs[k] >= 0) {
                        const float *f = slab + (size_t)vs[k] * CH * hw + pb[(size_t)vs[k] * n + 4 * i4 + k];
#pragma unroll
                        for (int q = 0; q < CH; ++q) r[q][k] = f[q * hw];
                    }
            } else {
                // F.max_pool1d over the stacked per-view maps: invisible views contribute zeros
                for (int v = 0; v < nv; ++v) {
                    const int4 pv = *(reinterpret_cast<const int4 *>(pb + (size_t)v * n) + i4);
                    const int ps[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float *f = slab + (size_t)v * CH * hw + (ps[k] >= 0 ? ps[k] : 0);
#pragma unroll
                        for (int q = 0; q < CH; ++q) {
                            const float x = ps[k] >= 0 ? f[q * hw] : 0.f;
                            r[q][k] = v == 0 ? x : fmaxf(r[q][k], x);
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < CH; ++q)
                if (q < cc) __stcs(reinterpret_cast<float4 *>(o + (size_t)q * n) + i4, make_float4(r[q][0], r[q][1], r[q][2], r[q][3]));
        }
        return;
    }
    for (int i = threadIdx.x; i < n; i += LG_THREADS) {
        float r[CH];
#pragma unroll
        for (int q = 0; q < CH; ++q) r[q] = 0.f;
        if (sel) {
            const int v = sel[(size_t)b * n + i];
            if (v >= 0) {
                const float *f = slab + (size_t)v * CH * hw + pb[(size_t)v * n + i];
#pragma unroll
                for (int q = 0; q < CH; ++q) r[q] = f[q * hw];
            }
        } else {
            for (int v = 0; v < nv; ++v) {
                const int p = pb[(size_t)v * n + i];
                const float *f = slab + (size_t)v * CH * hw + (p >= 0 ? p : 0);
#pragma unroll
                for (int q = 0; q < CH; ++q) {
                    const float x = p >= 0 ? f[q * hw] : 0.f;
                    r[q] = v == 0 ? x : fmaxf(r[q], x);
                }
            }
        }
#pragma unroll
        for (int q = 0; q < CH; ++q)
            if (q < cc) __stcs(o + (size_t)q * n + i, r[q]);
    }
}

// Pixel-major variant (the default when n % 4 == 0): the slab holds, per view and pixel, the FOUR channels of this CTA as
// one float4, so a (point, view) fetch is ONE 128-bit shared-memory load instead of four 32-bit ones, a lane that does not
// see the point issues no load at all, and the four points of a thread leave as one 128-bit streaming store per channel
// (a warp writes 512 contiguous bytes).  The fill transposes on the fly: a thread reads its pixel from the four channel
// rows (four coalesced 32-bit loads per warp) and writes one float4.

__device__ __forceinline__ void cp_async4(float *smem_dst, const float *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}

// NV = number of views at compile time (0 = run-time loop): with the views unrolled, the pixel indices of ALL views are
// loaded before the first shared-memory access (one L2 round trip per 4 points instead of one per view), and the fill
// is a burst of asynchronous 4-byte copies (cp.async: no registers, every load of the CTA in flight at once).
// (A persistent one-CTA-per-SM variant that fills a second slab while gathering from the first measured SLOWER: 78 vs
// 68 us for 32 scenes x 3 views; two independent 512-thread CTAs per SM overlap their phases better.)
constexpr int LP_THREADS = 512;

template <bool kFirst, int NV>
__global__ void __launch_bounds__(LP_THREADS, 2)
lift_gather_pm_kernel(int n, int nv_rt, int c, int hw, const float *__restrict__ feats, const int16_t *__restrict__ pix,
                      const signed char *__restrict__ sel, float *__restrict__ out) {
    extern __shared__ __align__(16) float4 slab4[];  // [nv][hw]
    const int nv = NV > 0 ? NV : nv_rt;
    const int b = blockIdx.y;
    const int c0 = blockIdx.x * 4;
    const int cc = min(4, c - c0);
    {
        // a warp instruction copies 32 consecutive pixels of one channel row: one 128-byte line on the global side, a 16-byte
        // stride (four wavefronts) on the shared side.  The opposite mapping (8 pixels x 4 channels per instruction: four
        // 32-byte global segments, 32 consecutive shared words) measured SLOWER: 78 vs 68 us for 32 scenes x 3 views.
        float *sl = reinterpret_cast<float *>(slab4);
        const int total = nv * hw;
        for (int e = threadIdx.x; e < total; e += LP_THREADS) {
            const int v = e / hw, p = e - v * hw;
            const float *src = feats + (((size_t)b * nv + v) * c + c0) * hw + p;
            float *dst = sl + (size_t)e * 4;
            cp_async4(dst, src);
            if (cc > 1) cp_async4(dst + 1, src + hw); else dst[1] = 0.f;
            if (cc > 2) cp_async4(dst + 2, src + 2 * (size_t)hw); else dst[2] = 0.f;
            if (cc > 3) cp_async4(dst + 3, src + 3 * (size_t)hw); else dst[3] = 0.f;
        }
        // Programmatic dependent launch: this grid may start while lift_project_kernel is still running (the fill above does
        // not depend on it); the pixel indices / view selection are only read after the projection grid has completed.
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("cp.async.wait_all;" ::: "memory");
    }
    __syncthreads();
    float *o = out + ((size_t)b * c + c0) * n;
    const int16_t *pb = pix + (size_t)b * nv * n;
    const int n4 = n >> 2;
    for (int i4 = threadIdx.x; i4 < n4; i4 += LP_THREADS) {
        float4 r[4];
        if (kFirst) {
#pragma unroll
            for (int k = 0; k < 4; ++k) r[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            // the view each point takes its column from was chosen by lift_project_kernel (first view with a non-zero column)
            const char4 sv = *reinterpret_cast<const char4 *>(sel + (size_t)b * n + 4 * i4);
            const int vs[4] = {sv.x, sv.y, sv.z, sv.w};
            int px[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) px[k] = vs[k] >= 0 ? (int)__ldg(pb + (size_t)vs[k] * n + 4 * i4 + k) : 0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (vs[k] >= 0) r[k] = slab4[(size_t)vs[k] * hw + px[k]];
        } else {
            // F.max_pool1d over the stacked per-view maps: invisible views contribute zeros.  max over {x_v} with -inf as the
            // neutral start value: every view, visible or not, contributes a finite value, so -inf never survives.
#pragma unroll
            for (int k = 0; k < 4; ++k) r[k] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
            if (NV > 0) {
                uint2 pv[NV > 0 ? NV : 1];
#pragma unroll
                for (int v = 0; v < NV; ++v) pv[v] = __ldg(reinterpret_cast<const uint2 *>(pb + (size_t)v * n) + i4);
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    const int ps[4] = {(int)(short)(pv[v].x & 0xffffu), (int)(short)(pv[v].x >> 16), (int)(short)(pv[v].y & 0xffffu),
                                       (int)(short)(pv[v].y >> 16)};
                    const float4 *sl = slab4 + (size_t)v * hw;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ps[k] >= 0) x = sl[ps[k]];
                        r[k].x = fmaxf(r[k].x, x.x);
                        r[k].y = fmaxf(r[k].y, x.y);
                        r[k].z = fmaxf(r[k].z, x.z);
                        r[k].w = fmaxf(r[k].w, x.w);
                    }
                }
            } else {
                for (int v = 0; v < nv; ++v) {
                    const uint2 pv = __ldg(reinterpret_cast<const uint2 *>(pb + (size_t)v * n) + i4);
                    const int ps[4] = {(int)(short)(pv.x & 0xffffu), (int)(short)(pv.x >> 16), (int)(short)(pv.y & 0xffffu), (int)(short)(pv.y >> 16)};
                    const float4 *sl = slab4 + (size_t)v * hw;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ps[k] >= 0) x = sl[ps[k]];
                        r[k].x = fmaxf(r[k].x, x.x);
                        r[k].y = fmaxf(r[k].y, x.y);
                        r[k].z = fmaxf(r[k].z, x.z);
                        r[k].w = fmaxf(r[k].w, x.w);
                    }
                }
            }
        }
        __stcs(reinterpret_cast<float4 *>(o) + i4, make_float4(r[0].x, r[1].x, r[2].x, r[3].x));
        if (cc > 1) __stcs(reinterpret_cast<float4 *>(o + (size_t)n) + i4, make_float4(r[0].y, r[1].y, r[2].y, r[3].y));
        if (cc > 2) __stcs(reinterpret_cast<float4 *>(o + 2 * (size_t)n) + i4, make_float4(r[0].z, r[1].z, r[2].z, r[3].z));
        if (cc > 3) __stcs(reinterpret_cast<float4 *>(o + 3 * (size_t)n) + i4, make_float4(r[0].w, r[1].w, r[2].w, r[3].w));
    }
}

template <bool kFirst, int NV>
int launch_lift_gather_pm_t(int b, int n, int nv, int c, int hw, const float *feats, const int16_t *pix, const signed char *sel, float *out,
                            cudaStream_t s) {
    const size_t smem = (size_t)nv * hw * sizeof(float4);
    PN2_CUDA(cudaFuncSetAttribute(lift_gather_pm_kernel<kFirst, NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ceil_div(c, 4), b);
    cfg.blockDim = dim3(LP_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // overlap the slab fill with the projection kernel
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    PN2_CUDA(cudaLaunchKernelEx(&cfg, lift_gather_pm_kernel<kFirst, NV>, n, nv, c, hw, feats, pix, sel, out));
    count_launch();
    return PN2_OK;
}

int launch_lift_gather_pm(int b, int n, int nv, int c, int hw, const float *feats, const int16_t *pix, const signed char *sel, float *out,
                          cudaStream_t s) {
    if (sel) return launch_lift_gather_pm_t<true, 0>(b, n, nv, c, hw, feats, pix, sel, out, s);
    switch (nv) {  // the view counts of the reference's multi-view training (3 in the script, 5 the class default) and their neighbours
        case 1: return launch_lift_gather_pm_t<false, 1>(b, n, nv, c, hw, feats, pix, sel, out, s);
        case 2: return launch_lift_gather_pm_t<false, 2>(b, n, nv, c, hw, feats, pix, sel, out, s);
        case 3: return launch_lift_gather_pm_t<false, 3>(b, n, nv, c, hw, feats, pix, sel, out, s);
        case 4: return launch_lift_gather_pm_t<false, 4>(b, n, nv, c, hw, feats, pix, sel, out, s);
        case 5: return launch_lift_gather_pm_t<false, 5>(b, n, nv, c, hw, feats, pix, sel, out, s);
        default: return launch_lift_gather_pm_t<false, 0>(b, n, nv, c, hw, feats, pix, sel, out, s);
    }
}

template <int CH>
int launch_lift_gather(int b, int n, int nv, int c, int hw, const float *feats, const int32_t *pix, const signed char *sel, float *out,
                       cudaStream_t s) {
    const size_t smem = (size_t)nv * CH * hw * sizeof(float);
    PN2_CUDA(cudaFuncSetAttribute(lift_gather_kernel<CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(ceil_div(c, CH), b);
    lift_gather_kernel<CH><<<grid, LG_THREADS, smem, s>>>(n, nv, c, hw, feats, pix, sel, out);
    PN2_LAUNCH_OK("lift_gather_kernel");
    return PN2_OK;
}

// Best-view selection of the ScanNet loader (data_utils/ScanNetDataLoader.py:87-105, 260-278): how many of the N crop
// points fall inside the frustum of EACH of the scene's P camera poses.  The reference calls points_in_frustum_cpu
// (utils/projection.py:132-164) once per pose file on the CPU in fp64; here all P x N tests are one launch, in fp64
// like the reference (same predicate as the lifting: round(100 * s) / 100 < 0 for the six planes).
constexpr int FC_THREADS = 256;
constexpr int FC_POSES = 32;  // poses per CTA (shared-memory tile)

__global__ void __launch_bounds__(FC_THREADS)
frustum_count_kernel(int n, int np, const float *__restrict__ points, const float *__restrict__ corner2,
                     const float *__restrict__ corner4, const float *__restrict__ normals, int32_t *__restrict__ counts) {
    __shared__ double sc2[FC_POSES][3], sc4[FC_POSES][3], sn[FC_POSES][18];
    __shared__ int cnt[FC_POSES];
    const int p0 = blockIdx.y * FC_POSES;
    const int pc = min(FC_POSES, np - p0);
    for (int e = threadIdx.x; e < pc * 18; e += FC_THREADS) sn[e / 18][e % 18] = (double)normals[(size_t)p0 * 18 + e];
    for (int e = threadIdx.x; e < pc * 3; e += FC_THREADS) {
        sc2[e / 3][e % 3] = (double)corner2[(size_t)p0 * 3 + e];
        sc4[e / 3][e % 3] = (double)corner4[(size_t)p0 * 3 + e];
    }
    if (threadIdx.x < FC_POSES) cnt[threadIdx.x] = 0;
    __syncthreads();
    const int i = blockIdx.x * FC_THREADS + threadIdx.x;
    const bool live = i < n;
    double px = 0, py = 0, pz = 0;
    if (live) {
        px = (double)points[3 * (size_t)i];
        py = (double)points[3 * (size_t)i + 1];
        pz = (double)points[3 * (size_t)i + 2];
    }
    for (int q = 0; q < pc; ++q) {
        bool inside = live;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const double *c = k < 3 ? sc2[q] : sc4[q];
            const double s = (px - c[0]) * sn[q][3 * k] + (py - c[1]) * sn[q][3 * k + 1] + (pz - c[2]) * sn[q][3 * k + 2];
            inside = inside && (rint(s * 100.0) < 0.0);  // == rint(100 s) / 100 < 0, see project_point
        }
        const unsigned m = __ballot_sync(0xffffffffu, inside);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&cnt[q], __popc(m));
    }
    __syncthreads();
    if (threadIdx.x < pc && cnt[threadIdx.x]) atomicAdd(counts + p0 + threadIdx.x, cnt[threadIdx.x]);
}

// ---- backward of the lifting with respect to the feature maps (pn2_lift_views_grad) --------------------------------
// The gradient torch autograd computes for the reference's composition: per view Projection (a scatter of the maps onto
// the points, zero for points that are not lifted; its backward is the transposed scatter), then the view reduction:
//   max   (F.max_pool1d over the stacked views, invisible views = 0): grad_out[b, c, i] goes to the FIRST view holding the
//         maximum of channel c (the pooling takes a new maximum only on a strict >), if that view sees the point;
//   first (in-place fill loop, model/pointnet2multiview.py:93-98): the whole column goes to the first visible view whose
//         C-channel column is not all zero, else to view V-1 (the loop's last assignment) if it sees the point.
// Deterministic by construction: the (view, pixel) keys of all contributions are inverted once per call (segment_sort,
// stable: ascending point index inside a segment), then every output element sums its segment in that order, fp32, with
// no atomics.  Every element of grad_feats is written.
//   lift_grad_keys_kernel  key per contribution: cloud * (V*HW + 1) + view * HW + pixel, or the cloud's last bucket (V*HW)
//                          for a point the view does not see / whose gradient is dropped; payload = the point index.
//                          max: one key per (view, point); first: one per point (the selected view, nz flags as in the forward)
//   lift_grad_kernel       one CTA per (cloud, 4 channels), output-stationary: a thread owns (view, pixel) outputs and
//                          walks their segments.  grad_out rows of the 4 channels are staged point-major (one float4 per
//                          point) and, for max, the feature slab of all views pixel-major as in lift_gather_pm_kernel, from
//                          which the per-channel winner of every contribution is recomputed.  Either falls back to global
//                          reads when it does not fit shared memory (large maps / clouds).  Writes are coalesced along pixels.
__global__ void __launch_bounds__(256)
lift_grad_keys_kernel(long long total, int n, int nv, int hw, int first, const int32_t *__restrict__ pix,
                      const unsigned char *__restrict__ nz, uint32_t *__restrict__ keys, int32_t *__restrict__ pos) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= total) return;
    const int nout = nv * hw;
    if (first) {  // e = b * n + i
        const long long b = e / n;
        const int i = (int)(e - b * n);
        const int32_t *pb = pix + (size_t)b * nv * n + i;
        int j = nv - 1;  // no view with a non-zero column: the fill loop's last assignment is view V-1
        for (int u = 0; u < nv; ++u) {
            const int p = pb[(size_t)u * n];
            if (p >= 0 && nz[((size_t)b * nv + u) * hw + p]) {
                j = u;
                break;
            }
        }
        const int p = pb[(size_t)j * n];
        keys[e] = (uint32_t)(b * (nout + 1) + (p >= 0 ? j * hw + p : nout));
        pos[e] = i;
    } else {  // e = (b * nv + u) * n + i
        const long long bu = e / n;
        const int i = (int)(e - bu * n);
        const long long b = bu / nv;
        const int u = (int)(bu - b * nv);
        const int p = pix[e];
        keys[e] = (uint32_t)(b * (nout + 1) + (p >= 0 ? u * hw + p : nout));
        pos[e] = i;
    }
}

// four channels of one (view, pixel) / one point, zero beyond the last channel; `stride` floats between channels
__device__ __forceinline__ float4 load_ch4(const float *__restrict__ src, size_t stride, int cc) {
    float4 x = make_float4(__ldg(src), 0.f, 0.f, 0.f);
    if (cc > 1) x.y = __ldg(src + stride);
    if (cc > 2) x.z = __ldg(src + 2 * stride);
    if (cc > 3) x.w = __ldg(src + 3 * stride);
    return x;
}

__device__ __forceinline__ void cp_async_ch4(float *dst, const float *src, size_t stride, int cc) {
    cp_async4(dst, src);
    if (cc > 1) cp_async4(dst + 1, src + stride); else dst[1] = 0.f;
    if (cc > 2) cp_async4(dst + 2, src + 2 * stride); else dst[2] = 0.f;
    if (cc > 3) cp_async4(dst + 3, src + 3 * stride); else dst[3] = 0.f;
}

constexpr int LGR_THREADS = 512;

template <bool kFirst, bool kSlab, bool kGrad>
__global__ void __launch_bounds__(LGR_THREADS)
lift_grad_kernel(int n, int nv, int c, int hw, const float *__restrict__ feats, const int32_t *__restrict__ pix,
                 const int32_t *__restrict__ seg_start, const int32_t *__restrict__ pos, const float *__restrict__ grad_out,
                 float *__restrict__ grad_feats) {
    extern __shared__ __align__(16) float4 sm4[];
    const int b = blockIdx.y;
    const int c0 = blockIdx.x * 4;
    const int cc = min(4, c - c0);
    const int nout = nv * hw;
    float4 *slab = sm4;                        // [nv][hw], kSlab
    float4 *gs = sm4 + (kSlab ? nout : 0);     // [n], kGrad
    const float *fb = feats + ((size_t)b * nv * c + c0) * hw;  // view u, channel c0 + q: fb + (u * c + q) * hw
    const float *gb = grad_out + ((size_t)b * c + c0) * n;     // channel c0 + q, point i: gb + q * n + i
    // fills: asynchronous 4-byte copies (every load of the CTA in flight at once), channel rows read coalesced
    if (kSlab)
        for (int e = threadIdx.x; e < nout; e += LGR_THREADS) {
            const int u = e / hw, p = e - u * hw;
            cp_async_ch4(reinterpret_cast<float *>(slab + e), fb + (size_t)u * c * hw + p, hw, cc);
        }
    if (kGrad)
        for (int i = threadIdx.x; i < n; i += LGR_THREADS) cp_async_ch4(reinterpret_cast<float *>(gs + i), gb + i, n, cc);
    if (kSlab || kGrad) {
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();
    }
    const int32_t *sb = seg_start + (size_t)b * (nout + 1);
    const int32_t *pb = pix + (size_t)b * nv * n;
    for (int o = threadIdx.x; o < nout; o += LGR_THREADS) {
        const int vv = o / hw, p = o - vv * hw;
        const int s0 = sb[o], s1 = sb[o + 1];
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int s = s0; s < s1; ++s) {
            const int i = __ldg(pos + s);
            const float4 g = kGrad ? gs[i] : load_ch4(gb + i, n, cc);
            if (kFirst) {
                acc.x = __fadd_rn(acc.x, g.x);
                acc.y = __fadd_rn(acc.y, g.y);
                acc.z = __fadd_rn(acc.z, g.z);
                acc.w = __fadd_rn(acc.w, g.w);
                continue;
            }
            // winner of each channel: the first view holding the maximum, invisible views taking part with 0.  The pixel
            // indices of all views are loaded before the first use (one dependent round trip per contribution, not V-1).
            int pu[LV_MAXV];
#pragma unroll
            for (int u = 0; u < LV_MAXV; ++u) pu[u] = u < nv && u != vv ? __ldg(pb + (size_t)u * n + i) : p;
            float4 best = make_float4(0.f, 0.f, 0.f, 0.f);
            int wx = 0, wy = 0, wz = 0, ww = 0;
#pragma unroll
            for (int u = 0; u < LV_MAXV; ++u) {
                if (u >= nv) break;
                float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pu[u] >= 0) x = kSlab ? slab[(size_t)u * hw + pu[u]] : load_ch4(fb + (size_t)u * c * hw + pu[u], hw, cc);
                if (u == 0) {
                    best = x;
                    continue;
                }
                if (x.x > best.x) { best.x = x.x; wx = u; }
                if (x.y > best.y) { best.y = x.y; wy = u; }
                if (x.z > best.z) { best.z = x.z; wz = u; }
                if (x.w > best.w) { best.w = x.w; ww = u; }
            }
            if (wx == vv) acc.x = __fadd_rn(acc.x, g.x);
            if (wy == vv) acc.y = __fadd_rn(acc.y, g.y);
            if (wz == vv) acc.z = __fadd_rn(acc.z, g.z);
            if (ww == vv) acc.w = __fadd_rn(acc.w, g.w);
        }
        float *dst = grad_feats + (((size_t)b * nv + vv) * c + c0) * hw + p;
        __stcs(dst, acc.x);
        if (cc > 1) __stcs(dst + hw, acc.y);
        if (cc > 2) __stcs(dst + 2 * (size_t)hw, acc.z);
        if (cc > 3) __stcs(dst + 3 * (size_t)hw, acc.w);
    }
}

template <bool kFirst, bool kSlab, bool kGrad>
int launch_lift_grad_t(int b, int n, int nv, int c, int hw, const float *feats, const int32_t *pix, const int32_t *seg_start,
                       const int32_t *pos, const float *grad_out, float *grad_feats, size_t smem, cudaStream_t s) {
    PN2_CUDA(cudaFuncSetAttribute(lift_grad_kernel<kFirst, kSlab, kGrad>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lift_grad_kernel<kFirst, kSlab, kGrad><<<dim3(ceil_div(c, 4), b), LGR_THREADS, smem, s>>>(n, nv, c, hw, feats, pix, seg_start, pos,
                                                                                            grad_out, grad_feats);
    PN2_LAUNCH_OK("lift_grad_kernel");
    return PN2_OK;
}

}  // namespace
}  // namespace pn2

extern "C" int pn2_frustum_count(int n, int num_poses, const float *points, const float *corner2, const float *corner4,
                                 const float *normals, int32_t *counts, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(n >= 0 && num_poses >= 0, "frustum_count: bad dims");
    if (n == 0 || num_poses == 0) return PN2_OK;
    PN2_REQUIRE(points && corner2 && corner4 && normals && counts, "frustum_count: null pointer");
    PN2_REQUIRE(ceil_div(num_poses, FC_POSES) <= 65535, "frustum_count: too many poses");
    dim3 grid(ceil_div(n, FC_THREADS), ceil_div(num_poses, FC_POSES));
    frustum_count_kernel<<<grid, FC_THREADS, 0, (cudaStream_t)stream>>>(n, num_poses, points, corner2, corner4, normals, counts);
    PN2_LAUNCH_OK("frustum_count");
    return PN2_OK;
}

extern "C" int pn2_lift_setup(int num_views, const float *c2w, const float *cam_corners, float *w2c, float *corner2, float *corner4,
                              float *normals, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(num_views >= 0, "lift_setup: bad dims");
    if (num_views == 0) return PN2_OK;
    PN2_REQUIRE(c2w && cam_corners && w2c && corner2 && corner4 && normals, "lift_setup: null pointer");
    CamCorners cam;
    for (int k = 0; k < 8; ++k)
        for (int r = 0; r < 3; ++r) cam.p[k][r] = cam_corners[3 * k + r];
    lift_setup_kernel<<<ceil_div(num_views, 128), 128, 0, (cudaStream_t)stream>>>(num_views, c2w, cam, w2c, corner2, corner4, normals);
    PN2_LAUNCH_OK("lift_setup_kernel");
    return PN2_OK;
}

static int lift_views_impl(int b, int n, int v, int c, int h, int w, const float *points, const float *feats,
                           const float *depth, const float *w2c, const float *corner2, const float *corner4,
                           const float *normals, const float *c2w, const float *cam_corners, const float *intr, float depth_min,
                           float depth_max, float accuracy, int reduce, float *out, int32_t *pix, int32_t *count, void *stream) {
    using namespace pn2;
    CamCorners cam = {};
    if (c2w)
        for (int k = 0; k < 8; ++k)
            for (int r = 0; r < 3; ++r) cam.p[k][r] = cam_corners[3 * k + r];
    PN2_REQUIRE(b >= 0 && n >= 0 && v >= 1 && c >= 0 && h >= 1 && w >= 1, "lift_views: bad dims");
    if (v > LV_MAXV) return set_error(PN2_ERR_UNSUPPORTED, "lift_views: at most %d views per cloud (got %d)", LV_MAXV, v);
    PN2_REQUIRE(reduce == PN2_REDUCE_MAX || reduce == PN2_REDUCE_FIRST, "lift_views: unknown reduce %d", reduce);
    if (b == 0 || n == 0) return PN2_OK;
    PN2_REQUIRE(points && depth && ((w2c && corner2 && corner4 && normals) || (c2w && cam_corners)) && intr && ((feats && out) || c == 0),
                "lift_views: null pointer");
    PN2_REQUIRE(b <= 65535, "lift_views: b exceeds the grid limit");
    cudaStream_t s = (cudaStream_t)stream;
    const int hw = h * w;
    // staged path when a slab of all views fits shared memory for at least one channel (ENet-sized maps: 4-8 channels)
    const size_t per_ch = (size_t)v * hw * sizeof(float);
    const int chunk = c == 0 ? 0 : (8 * per_ch <= 100 * 1024 ? 8 : 4 * per_ch <= 100 * 1024 ? 4 : 2 * per_ch <= 200 * 1024 ? 2 : per_ch <= 200 * 1024 ? 1 : -1);
    if (chunk >= 0 && ceil_div(c, chunk > 0 ? chunk : 1) <= 65535) {
        const bool first = reduce == PN2_REDUCE_FIRST && c > 0;
        // the pixel-major gather reads 16-bit pixel indices (half the index traffic: every 4-channel CTA re-reads them)
        const bool pm_ok = c > 0 && (n & 3) == 0 && (((uintptr_t)out) & 15) == 0 && (size_t)v * hw * 16 <= 200 * 1024 && hw < 32768 &&
                           ceil_div(c, 4) <= 65535;
        const bool need32 = !pix && !pm_ok;
        const size_t pix_bytes = need32 ? ((size_t)b * v * n * sizeof(int32_t) + 255) / 256 * 256 : 0;
        const size_t pix16_bytes = pm_ok ? ((size_t)b * v * n * sizeof(int16_t) + 255) / 256 * 256 : 0;
        const size_t sel_bytes = first ? ((size_t)b * n + 255) / 256 * 256 : 0;
        const size_t nz_bytes = first ? ((size_t)b * v * hw + 255) / 256 * 256 : 0;
        Scratch scratch_mem(s);  // released on every return below
        PN2_CUDA(scratch_mem.alloc(pix_bytes + pix16_bytes + sel_bytes + nz_bytes + 256));
        unsigned char *scratch = (unsigned char *)scratch_mem.ptr;
        unsigned char *cur = scratch;
        int32_t *pixbuf = pix;
        if (need32) {
            pixbuf = (int32_t *)cur;
            cur += pix_bytes;
        }
        int16_t *pix16 = pm_ok ? (int16_t *)cur : nullptr;
        cur += pix16_bytes;
        signed char *sel = first ? (signed char *)cur : nullptr;
        cur += sel_bytes;
        unsigned char *nz = first ? cur : nullptr;
        if (first) {
            lift_nonzero_kernel<<<dim3(ceil_div(hw, 256), b * v), 256, 0, s>>>(c, hw, feats, nz);
            PN2_LAUNCH_OK("lift_nonzero_kernel");
        }
        lift_project_kernel<<<dim3(ceil_div(n, LV_THREADS), b), LV_THREADS, 0, s>>>(n, v, h, w, points, depth, w2c, corner2, corner4, normals,
                                                                                  c2w, cam, intr[0], intr[1], intr[2], intr[3], depth_min,
                                                                                  depth_max, accuracy, nz, pixbuf, pix16, sel, count);
        PN2_LAUNCH_OK("lift_project_kernel");
        int st = PN2_OK;
        if (pm_ok) st = launch_lift_gather_pm(b, n, v, c, hw, feats, pix16, sel, out, s);
        else if (chunk == 8) st = launch_lift_gather<8>(b, n, v, c, hw, feats, pixbuf, sel, out, s);
        else if (chunk == 4) st = launch_lift_gather<4>(b, n, v, c, hw, feats, pixbuf, sel, out, s);
        else if (chunk == 2) st = launch_lift_gather<2>(b, n, v, c, hw, feats, pixbuf, sel, out, s);
        else if (chunk == 1) st = launch_lift_gather<1>(b, n, v, c, hw, feats, pixbuf, sel, out, s);
        return st;
    }
    // feature maps too large for a shared-memory slab: one kernel, per-element gathers
    if (!w2c) return set_error(PN2_ERR_UNSUPPORTED, "lift_views_poses: feature maps too large for the staged path; call pn2_lift_setup + pn2_lift_views");
    dim3 grid(ceil_div(n, LV_THREADS), b);
    lift_views_kernel<<<grid, LV_THREADS, 0, s>>>(n, v, c, h, w, points, feats, depth, w2c, corner2, corner4,
                                                                     normals, intr[0], intr[1], intr[2], intr[3], depth_min,
                                                                     depth_max, accuracy, reduce, out, pix, count);
    PN2_LAUNCH_OK("lift_views");
    return PN2_OK;
}

extern "C" int pn2_lift_views(int b, int n, int v, int c, int h, int w, const float *points, const float *feats,
                              const float *depth, const float *w2c, const float *corner2, const float *corner4,
                              const float *normals, const float *intr, float depth_min, float depth_max,
                              float accuracy, int reduce, float *out, int32_t *pix, int32_t *count, void *stream) {
    return lift_views_impl(b, n, v, c, h, w, points, feats, depth, w2c, corner2, corner4, normals, nullptr, nullptr, intr, depth_min,
                           depth_max, accuracy, reduce, out, pix, count, stream);
}

extern "C" int pn2_lift_views_poses(int b, int n, int v, int c, int h, int w, const float *points, const float *feats,
                                    const float *depth, const float *c2w, const float *cam_corners, const float *intr,
                                    float depth_min, float depth_max, float accuracy, int reduce, float *out, int32_t *pix,
                                    int32_t *count, void *stream) {
    return lift_views_impl(b, n, v, c, h, w, points, feats, depth, nullptr, nullptr, nullptr, nullptr, c2w, cam_corners, intr, depth_min,
                           depth_max, accuracy, reduce, out, pix, count, stream);
}

extern "C" int pn2_lift_views_grad(int b, int n, int v, int c, int h, int w, const float *feats, const int32_t *pix, int reduce,
                                   const float *grad_out, float *grad_feats, void *stream) {
    using namespace pn2;
    PN2_REQUIRE(b >= 0 && n >= 0 && v >= 1 && c >= 0 && h >= 1 && w >= 1, "lift_views_grad: bad dims");
    if (v > LV_MAXV) return set_error(PN2_ERR_UNSUPPORTED, "lift_views_grad: at most %d views per cloud (got %d)", LV_MAXV, v);
    PN2_REQUIRE(reduce == PN2_REDUCE_MAX || reduce == PN2_REDUCE_FIRST, "lift_views_grad: unknown reduce %d", reduce);
    if (b == 0 || c == 0) return PN2_OK;
    PN2_REQUIRE(grad_feats && (n == 0 || (feats && pix && grad_out)), "lift_views_grad: null pointer");
    PN2_REQUIRE(b <= 65535 && ceil_div(c, 4) <= 65535 && (reduce != PN2_REDUCE_FIRST || b * v <= 65535),
                "lift_views_grad: b, c/4 and (for reduce first) b*v must be <= 65535");
    const int hw = h * w;
    const long long nkeys = (long long)b * ((long long)v * hw + 1);
    PN2_REQUIRE(nkeys < (1ll << 31) && (long long)b * v * n < (1ll << 31) && (long long)b * v * c * hw < (1ll << 31),
                "lift_views_grad: more than 2^31 elements");
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0) {  // no point: nothing reaches the maps
        PN2_CUDA(cudaMemsetAsync(grad_feats, 0, (size_t)b * v * c * hw * sizeof(float), s));
        return PN2_OK;
    }
    const bool first = reduce == PN2_REDUCE_FIRST;
    const long long total = first ? (long long)b * n : (long long)b * v * n;  // one contribution per point / per (view, point)
    const size_t key_bytes = ((size_t)total * sizeof(uint32_t) + 255) / 256 * 256;
    const size_t seg_bytes = ((size_t)(nkeys + 1) * sizeof(int32_t) + 255) / 256 * 256;
    const size_t nz_bytes = first ? ((size_t)b * v * hw + 255) / 256 * 256 : 0;
    Scratch scratch_mem(s);  // [keys | payloads in | payloads sorted | segment starts | nz flags | segment_sort scratch]
    PN2_CUDA(scratch_mem.alloc(3 * key_bytes + seg_bytes + nz_bytes + segment_sort_scratch_bytes(total, nkeys)));
    unsigned char *cur = (unsigned char *)scratch_mem.ptr;
    uint32_t *keys = (uint32_t *)cur;
    int32_t *pos_in = (int32_t *)(cur + key_bytes);
    int32_t *pos = (int32_t *)(cur + 2 * key_bytes);
    int32_t *seg_start = (int32_t *)(cur + 3 * key_bytes);
    unsigned char *nz = cur + 3 * key_bytes + seg_bytes;
    void *sort_scratch = cur + 3 * key_bytes + seg_bytes + nz_bytes;
    if (first) {
        lift_nonzero_kernel<<<dim3(ceil_div(hw, 256), b * v), 256, 0, s>>>(c, hw, feats, nz);
        PN2_LAUNCH_OK("lift_nonzero_kernel");
    }
    lift_grad_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(total, n, v, hw, first ? 1 : 0, pix, nz, keys, pos_in);
    PN2_LAUNCH_OK("lift_grad_keys_kernel");
    const int st = segment_sort(total, nkeys, keys, pos_in, sort_scratch, seg_start, pos, s);
    if (st != PN2_OK) return st;
    // shared memory: the feature slab of all views (max only), then the grad_out rows, each only while it fits
    const size_t budget = 200 * 1024;
    const size_t slab_bytes = !first && (size_t)v * hw * sizeof(float4) <= budget ? (size_t)v * hw * sizeof(float4) : 0;
    const size_t grad_bytes = slab_bytes + (size_t)n * sizeof(float4) <= budget ? (size_t)n * sizeof(float4) : 0;
    const size_t smem = slab_bytes + grad_bytes;
    if (first)
        return grad_bytes ? launch_lift_grad_t<true, false, true>(b, n, v, c, hw, feats, pix, seg_start, pos, grad_out, grad_feats, smem, s)
                          : launch_lift_grad_t<true, false, false>(b, n, v, c, hw, feats, pix, seg_start, pos, grad_out, grad_feats, smem, s);
    if (slab_bytes)
        return grad_bytes ? launch_lift_grad_t<false, true, true>(b, n, v, c, hw, feats, pix, seg_start, pos, grad_out, grad_feats, smem, s)
                          : launch_lift_grad_t<false, true, false>(b, n, v, c, hw, feats, pix, seg_start, pos, grad_out, grad_feats, smem, s);
    return grad_bytes ? launch_lift_grad_t<false, false, true>(b, n, v, c, hw, feats, pix, seg_start, pos, grad_out, grad_feats, smem, s)
                      : launch_lift_grad_t<false, false, false>(b, n, v, c, hw, feats, pix, seg_start, pos, grad_out, grad_feats, smem, s);
}
