// fps.cu -- furthest point sampling for sm_100a.
//
// Replaces furthest_point_sampling_kernel / _launcher of the reference
// (utils/src/sampling_gpu.cu:93-253).  Result contract (SURVEY.md A.1): idx[0] = 0, and round j
// picks the point maximising temp[k] = min over previous picks of D(k, pick) under the total order
//     (temp desc, bitrev_{log2 bs}(k mod bs) asc, k asc),   bs = largest pow2 <= min(N, 1024),
// which is what the reference's per-thread strict-max scan + tree reduction produce.
//
// Design (not the reference's): the cloud lives ON CHIP for the whole kernel.  Each thread owns
// P points (coordinates and running minimum in registers), so a round touches no global or L2
// memory at all.  The arg-max is a single 64-bit key  (float bits of temp | ~tie key)  reduced with
// two CREDUX.MAX per warp, one shared-memory hop and ONE block barrier per round (slots are
// double-buffered by round parity); the reference spends 10 barriers and 20*N bytes of L2 traffic
// per round.  Clouds of 1024 < N <= 8192 points run on 256 threads with 8-32 points each (fps_few_kernel:
// the per-warp cost of a round is paid by 8 warps, 0.53 us per round at N = 8192).  With few clouds in
// flight (4*B <= #SMs) or clouds larger than one CTA's registers (8192 < N <= 49152) each cloud is split
// over a 4-CTA thread-block cluster whose warps exchange their winners through distributed shared memory
// with st.async + mbarrier complete_tx (fps_cluster_kernel): 0.44 us per round at N = 8192.
#include "common.cuh"

namespace pn2 {
namespace {

constexpr int QB = 22;  // low bits of the tie key hold q = k / bs; high bits hold bitrev(k mod bs)
constexpr uint32_t QMASK = (1u << QB) - 1u;

__device__ __forceinline__ void warp_argmax(uint32_t &hi, uint32_t &lo) {
    const uint32_t mh = __reduce_max_sync(0xffffffffu, hi);
    const uint32_t l2 = (hi == mh) ? lo : 0u;
    lo = __reduce_max_sync(0xffffffffu, l2);
    hi = mh;
}

// Running-minimum update of a thread's P points against the newest pick.  Pairs of points go through the packed
// f32x2 pipe (FADD2 / FMUL2 / FFMA2: half the issue slots of the scalar sequence); every lane performs exactly the
// IEEE operations of dist_ref -- x - c is x + (-c), then rn(dy*dy), fma(dx,dx,.), fma(dz,dz,.) -- so the result is
// bit-identical.
template <int P>
__device__ __forceinline__ void update_min(const float (&x)[P], const float (&y)[P], const float (&z)[P], float (&tm)[P],
                                           float cx, float cy, float cz) {
    if constexpr (P % 2 == 0) {
        const float2 nx = make_float2(-cx, -cx), ny = make_float2(-cy, -cy), nz = make_float2(-cz, -cz);
#pragma unroll
        for (int i = 0; i < P; i += 2) {
            const float2 dx = __fadd2_rn(make_float2(x[i], x[i + 1]), nx);
            const float2 dy = __fadd2_rn(make_float2(y[i], y[i + 1]), ny);
            const float2 dz = __fadd2_rn(make_float2(z[i], z[i + 1]), nz);
            const float2 d = __ffma2_rn(dz, dz, __ffma2_rn(dx, dx, __fmul2_rn(dy, dy)));
            tm[i] = fminf(d.x, tm[i]);
            tm[i + 1] = fminf(d.y, tm[i + 1]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < P; ++i) tm[i] = fminf(dist_ref(x[i], y[i], z[i], cx, cy, cz), tm[i]);
    }
}

template <int T>
struct Log2 {
    static constexpr int value = 1 + Log2<T / 2>::value;
};
template <>
struct Log2<1> {
    static constexpr int value = 0;
};

// One CTA per cloud, T == the reference block size for this N, N <= T*P.
// Thread t owns points k = t + i*T (i < P): all share r = k mod bs = t, so the tie key of point i is
// (bitrev(t) << QB) | i and "first strict maximum in ascending i" is the correct in-thread order.
template <int T, int P>
__global__ void __launch_bounds__(T, 1)
fps_reg_kernel(int n, int m, const float *__restrict__ xyz_all, int32_t *__restrict__ idx_all,
               float *__restrict__ new_xyz_all) {
    constexpr int NW = T / 32;
    constexpr int LG = Log2<T>::value;
    extern __shared__ float smem[];
    float *sx = smem, *sy = smem + T * P, *sz = smem + 2 * T * P;
    __shared__ unsigned long long slot[2][32];

    const float *xyz = xyz_all + (size_t)blockIdx.x * n * 3;
    int32_t *idx = idx_all + (size_t)blockIdx.x * m;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;

    float x[P], y[P], z[P], tm[P];
#pragma unroll
    for (int i = 0; i < P; ++i) {
        const int k = t + i * T;
        const bool ok = k < n;
        x[i] = ok ? xyz[3 * k + 0] : 0.f;
        y[i] = ok ? xyz[3 * k + 1] : 0.f;
        z[i] = ok ? xyz[3 * k + 2] : 0.f;
        // padding points carry temp = 0: they can only tie when every real temp is 0, and then
        // point 0 (tie key 0) wins anyway.  Real points start at 1e10 (model/pointnet2_utils.py:26).
        tm[i] = ok ? 1e10f : 0.f;
        sx[k] = x[i];
        sy[k] = y[i];
        sz[k] = z[i];
    }
    const uint32_t rank = __brev((uint32_t)t) >> (32 - LG);
    const uint32_t inv_base = 0xFFFFFFFFu - (rank << QB);
    float *new_xyz = new_xyz_all ? new_xyz_all + (size_t)blockIdx.x * m * 3 : nullptr;
    if (t == 0) idx[0] = 0;
    __syncthreads();
    float x1 = sx[0], y1 = sy[0], z1 = sz[0];
    if (t == 0 && new_xyz) {
        new_xyz[0] = x1; new_xyz[1] = y1; new_xyz[2] = z1;
    }

    for (int j = 1; j < m; ++j) {
        update_min<P>(x, y, z, tm, x1, y1, z1);
        float best = tm[0];
        int besti = 0;
#pragma unroll
        for (int i = 1; i < P; ++i) {
            if (tm[i] > best) {
                best = tm[i];
                besti = i;
            }
        }
        uint32_t hi = __float_as_uint(best), lo = inv_base - (uint32_t)besti;
        warp_argmax(hi, lo);
        if (NW > 1) {
            if (lane == 0) slot[j & 1][warp] = ((unsigned long long)hi << 32) | lo;
            __syncthreads();
            const unsigned long long v = lane < NW ? slot[j & 1][lane] : 0ull;
            hi = (uint32_t)(v >> 32);
            lo = (uint32_t)v;
            warp_argmax(hi, lo);
        }
        const uint32_t tie = 0xFFFFFFFFu - lo;
        const int k = (int)(tie & QMASK) * T + (int)(__brev(tie >> QB) >> (32 - LG));
        x1 = sx[k];
        y1 = sy[k];
        z1 = sz[k];
        if (t == 0) {
            idx[j] = k;
            if (new_xyz) {
                new_xyz[3 * j] = x1; new_xyz[3 * j + 1] = y1; new_xyz[3 * j + 2] = z1;
            }
        }
    }
}

// One CTA per cloud with FEWER THREADS than the reference block size (bs = 1024): T = 256 threads own P = 4Q points
// each (Q = capacity / 1024).  The fixed per-warp cost of a round (two CREDUX pairs, slot exchange, barrier, decode) is
// paid by 8 warps instead of 32, so a round issues ~30 % fewer instructions and the CTA holds fewer registers -- the
// variant for several batches in flight, where SM time, not latency, is what FPS costs.
// Thread t owns k = t + 256*(4q + s), q < Q, s < 4.  Its tie key is (bitrev10(k mod 1024) << QB) | q with
// bitrev10(t + 256 s) = bitrev10(t) + bitrev2(s), so the in-thread tie order is "s in bit-reversed order, then q
// ascending": the points are held in that order (slot j = bitrev2(s)*Q + q) and the first strict maximum in ascending j
// is the reference's winner.
// A value-first round (reduce only the maximum's value, then the threads holding it resolve the tie key by an atomic
// minimum in shared memory) was slower: 0.571 vs 0.529 us per round at 8192 points (32 clouds) -- it saves issue slots
// but adds a block barrier to the round's dependent chain, and that chain, not issue, is what a round costs.
template <int Q>
__global__ void __launch_bounds__(256, 1)
fps_few_kernel(int n, int m, const float *__restrict__ xyz_all, int32_t *__restrict__ idx_all,
               float *__restrict__ new_xyz_all) {
    constexpr int T = 256, SUB = 4, LS = 2, P = SUB * Q, NW = T / 32;
    extern __shared__ float smem[];
    float *sx = smem, *sy = smem + 1024 * Q, *sz = smem + 2 * 1024 * Q;
    __shared__ unsigned long long slot[2][32];

    const float *xyz = xyz_all + (size_t)blockIdx.x * n * 3;
    int32_t *idx = idx_all + (size_t)blockIdx.x * m;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;

    float x[P], y[P], z[P], tm[P];
#pragma unroll
    for (int j = 0; j < P; ++j) {
        const int sr = j / Q, q = j % Q;                               // sr = bit-reversed s
        const int sb = (int)(__brev((unsigned)sr) >> (32 - LS));
        const int k = t + T * (SUB * q + sb);
        const bool ok = k < n;
        x[j] = ok ? xyz[3 * k + 0] : 0.f;
        y[j] = ok ? xyz[3 * k + 1] : 0.f;
        z[j] = ok ? xyz[3 * k + 2] : 0.f;
        tm[j] = ok ? 1e10f : 0.f;  // padding never wins: see fps_reg_kernel
        sx[k] = x[j];
        sy[k] = y[j];
        sz[k] = z[j];
    }
    const uint32_t rank0 = __brev((uint32_t)t) >> 22;  // bitrev10(t); t < T so its low log2(SUB) bits are free
    const uint32_t inv_base = 0xFFFFFFFFu - (rank0 << QB);
    float *new_xyz = new_xyz_all ? new_xyz_all + (size_t)blockIdx.x * m * 3 : nullptr;
    if (t == 0) idx[0] = 0;
    __syncthreads();
    float x1 = sx[0], y1 = sy[0], z1 = sz[0];
    if (t == 0 && new_xyz) {
        new_xyz[0] = x1; new_xyz[1] = y1; new_xyz[2] = z1;
    }

    for (int r = 1; r < m; ++r) {
        update_min<P>(x, y, z, tm, x1, y1, z1);
        // pairwise (log-depth) arg-max; on ties the lower slot wins
        float bv[P];
        int bi[P];
#pragma unroll
        for (int j = 0; j < P; ++j) {
            bv[j] = tm[j];
            bi[j] = j;
        }
#pragma unroll
        for (int s2 = 1; s2 < P; s2 *= 2) {
#pragma unroll
            for (int j = 0; j + s2 < P; j += 2 * s2) {
                const bool take = bv[j + s2] > bv[j];
                bv[j] = take ? bv[j + s2] : bv[j];
                bi[j] = take ? bi[j + s2] : bi[j];
            }
        }
        const int bj = bi[0];
        uint32_t hi = __float_as_uint(bv[0]);
        uint32_t lo = inv_base - ((((uint32_t)bj / Q) << QB) | ((uint32_t)bj % Q));
        warp_argmax(hi, lo);
        if (lane == 0) slot[r & 1][warp] = ((unsigned long long)hi << 32) | lo;
        __syncthreads();
        const unsigned long long v = lane < NW ? slot[r & 1][lane] : 0ull;
        hi = (uint32_t)(v >> 32);
        lo = (uint32_t)v;
        warp_argmax(hi, lo);
        const uint32_t tie = 0xFFFFFFFFu - lo;
        const int k = (int)(tie & QMASK) * 1024 + (int)(__brev(tie >> QB) >> 22);
        x1 = sx[k];
        y1 = sy[k];
        z1 = sz[k];
        if (t == 0) {
            idx[r] = k;
            if (new_xyz) {
                new_xyz[3 * r] = x1; new_xyz[3 * r + 1] = y1; new_xyz[3 * r + 2] = z1;
            }
        }
    }
}

// ---- one CTA per cloud, warps own spatial slabs and SKIP rounds that provably change nothing -------------------------
// Same round as fps_few_kernel (T = 256 threads, P = 4Q points per thread in registers), but a warp's 32P points are a
// spatial slab of the cloud -- the points are bucketed along the cloud's longest axis when the kernel starts (counting
// sort over 256 bins) -- instead of the index-interleaved set k = t (mod 256).  Per round a warp first tests the distance
// from the newest pick to its slab's bounding box against the largest running minimum it holds: if
// d_box^2 * (1 - 1e-4) > max_j temp[j]  no temp[j] of the warp can decrease (every distance the update would compute is
// >= d_box^2 up to a few ulp), so the warp keeps its cached (max, tie key) and contributes it to the block reduction
// without touching its points.  Once a few dozen points are picked most warps skip most rounds (2.1 of 8 slabs active on
// average over the 1023 rounds of a ScanNet-shaped scene) and the one or two warps near the pick run alone on their
// schedulers.  The result is bit-identical: a skipped update is an update that changes no value.
// Measured (32 clouds, 8192 -> 1024): 0.492 ms against 0.543 ms for fps_few_kernel; the round is bound by its latency
// chain (two dependent warp reductions, one shared-memory hop, one barrier, the decode and the coordinate fetch), not
// by issue slots.  A finer variant -- every thread holds a share of all eight slabs, lane g tests slab g, a ballot gives
// the slabs to update, so the remaining work is spread over all warps -- measured NO faster (0.543 ms: the per-group
// bookkeeping costs what the skipped updates save) and 30 % slower at 4096 points.
// Tie order: ownership is spatial, so a point's tie key (bitrev10(k mod 1024) << QB | k / 1024) is explicit.  Each warp
// sorts its slab by tie key once (bitonic sort in shared memory) and deals the sorted points to (slot, lane) slot-major,
// so inside a thread "first strict maximum in ascending slot" is again "smallest tie key among equal maxima"; the key of
// a thread's winner is read from shared memory (one LDS per round).
template <int Q>
__global__ void __maxnreg__(184)  // leaves the registers of one tensor-core MLP CTA (192 x 96) on the SM, like fps_few_kernel
fps_slab_kernel(int n, int m, const float *__restrict__ xyz_all, int32_t *__restrict__ idx_all, float *__restrict__ new_xyz_all) {
    constexpr int T = 256, P = 4 * Q, NPT = T * P, S = 32 * P, NW = T / 32;
    extern __shared__ float smem[];
    float *sx = smem, *sy = smem + NPT, *sz = smem + 2 * NPT;                 // coordinates by ORIGINAL index
    uint32_t *skey = reinterpret_cast<uint32_t *>(smem + 3 * NPT);             // tie key by slab position
    unsigned long long *scratch = reinterpret_cast<unsigned long long *>(smem);  // set-up only: aliases sx / sy
    __shared__ unsigned long long slot[2][32];
    __shared__ int hist[256];
    __shared__ float red[6][NW];
    __shared__ int wsum[NW];

    const float *xyz = xyz_all + (size_t)blockIdx.x * n * 3;
    int32_t *idx = idx_all + (size_t)blockIdx.x * m;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const float INF = __int_as_float(0x7f800000);

    // ---- set-up 1: bounding box of the cloud, longest axis ----
    float lo0 = INF, lo1 = INF, lo2 = INF, hi0 = -INF, hi1 = -INF, hi2 = -INF;
    for (int i = 0; i < P; ++i) {
        const int k = t + T * i;
        if (k < n) {
            const float vx = xyz[3 * k], vy = xyz[3 * k + 1], vz = xyz[3 * k + 2];
            lo0 = fminf(lo0, vx); hi0 = fmaxf(hi0, vx);
            lo1 = fminf(lo1, vy); hi1 = fmaxf(hi1, vy);
            lo2 = fminf(lo2, vz); hi2 = fmaxf(hi2, vz);
        }
    }
    for (int o = 16; o; o >>= 1) {
        lo0 = fminf(lo0, __shfl_xor_sync(0xffffffffu, lo0, o)); hi0 = fmaxf(hi0, __shfl_xor_sync(0xffffffffu, hi0, o));
        lo1 = fminf(lo1, __shfl_xor_sync(0xffffffffu, lo1, o)); hi1 = fmaxf(hi1, __shfl_xor_sync(0xffffffffu, hi1, o));
        lo2 = fminf(lo2, __shfl_xor_sync(0xffffffffu, lo2, o)); hi2 = fmaxf(hi2, __shfl_xor_sync(0xffffffffu, hi2, o));
    }
    if (lane == 0) {
        red[0][warp] = lo0; red[1][warp] = lo1; red[2][warp] = lo2;
        red[3][warp] = hi0; red[4][warp] = hi1; red[5][warp] = hi2;
    }
    hist[t] = 0;
    __syncthreads();
    for (int w = 0; w < NW; ++w) {
        lo0 = fminf(lo0, red[0][w]); lo1 = fminf(lo1, red[1][w]); lo2 = fminf(lo2, red[2][w]);
        hi0 = fmaxf(hi0, red[3][w]); hi1 = fmaxf(hi1, red[4][w]); hi2 = fmaxf(hi2, red[5][w]);
    }
    int axis = 0;
    float c0 = lo0, ext = hi0 - lo0;
    if (hi1 - lo1 > ext) { axis = 1; c0 = lo1; ext = hi1 - lo1; }
    if (hi2 - lo2 > ext) { axis = 2; c0 = lo2; ext = hi2 - lo2; }
    const float scale = ext > 0.f ? 256.0f / ext : 0.f;
    // ---- set-up 2: counting sort of the points into 256 bins along that axis (slab = S consecutive positions) ----
    for (int i = 0; i < P; ++i) {
        const int k = t + T * i;
        if (k < n) atomicAdd(&hist[min(255, max(0, (int)((xyz[3 * k + axis] - c0) * scale)))], 1);
    }
    __syncthreads();
    {
        const int v = hist[t];
        int inc = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        int base = 0;
        for (int w = 0; w < warp; ++w) base += wsum[w];
        hist[t] = base + inc - v;  // exclusive prefix = first position of the bin; doubles as its cursor below
    }
    __syncthreads();
    for (int i = 0; i < P; ++i) {
        const int k = t + T * i;
        if (k < n) {
            const int pos = atomicAdd(&hist[min(255, max(0, (int)((xyz[3 * k + axis] - c0) * scale)))], 1);
            const uint32_t tie = ((__brev((uint32_t)k) >> 22) << QB) | ((uint32_t)k >> 10);
            scratch[pos] = ((unsigned long long)tie << 16) | (unsigned long long)k;
        }
    }
    for (int pos = n + t; pos < NPT; pos += T) scratch[pos] = ~0ull;  // padding: sorts last, never wins
    __syncthreads();
    // ---- set-up 3: every warp sorts its slab by tie key (ascending) ----
    {
        unsigned long long *base = scratch + warp * S;
        for (int size = 2; size <= S; size <<= 1)
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int e = lane; e < S / 2; e += 32) {
                    const int i = ((e & ~(stride - 1)) << 1) | (e & (stride - 1)), j = i + stride;  // stride is a power of two
                    const bool up = (i & size) == 0;
                    const unsigned long long a = base[i], b = base[j];
                    if ((a > b) == up) {
                        base[i] = b;
                        base[j] = a;
                    }
                }
                __syncwarp();
            }
    }
    __syncthreads();
    // ---- set-up 4: the thread's points (slot-major deal: position = slot * 32 + lane) into registers ----
    float x[P], y[P], z[P], tm[P];
    float bl0 = INF, bl1 = INF, bl2 = INF, bh0 = -INF, bh1 = -INF, bh2 = -INF;  // bounding box of the warp's slab
    {
        int kk[P];
#pragma unroll
        for (int j = 0; j < P; ++j) {
            const unsigned long long v = scratch[warp * S + j * 32 + lane];
            kk[j] = v == ~0ull ? -1 : (int)(v & 0xFFFFull);
        }
        __syncthreads();  // scratch is dead: tie keys and coordinates may be written (skey does not alias it, sx / sy do)
#pragma unroll
        for (int j = 0; j < P; ++j) {
            const bool ok = kk[j] >= 0;
            skey[warp * S + j * 32 + lane] = ok ? (((__brev((uint32_t)kk[j]) >> 22) << QB) | ((uint32_t)kk[j] >> 10)) : 0xFFFFFFFFu;
            x[j] = ok ? xyz[3 * kk[j] + 0] : 0.f;
            y[j] = ok ? xyz[3 * kk[j] + 1] : 0.f;
            z[j] = ok ? xyz[3 * kk[j] + 2] : 0.f;
            tm[j] = ok ? 1e10f : 0.f;  // padding never wins: see fps_reg_kernel
            if (ok) {
                bl0 = fminf(bl0, x[j]); bh0 = fmaxf(bh0, x[j]);
                bl1 = fminf(bl1, y[j]); bh1 = fmaxf(bh1, y[j]);
                bl2 = fminf(bl2, z[j]); bh2 = fmaxf(bh2, z[j]);
            }
        }
    }
    for (int o = 16; o; o >>= 1) {
        bl0 = fminf(bl0, __shfl_xor_sync(0xffffffffu, bl0, o)); bh0 = fmaxf(bh0, __shfl_xor_sync(0xffffffffu, bh0, o));
        bl1 = fminf(bl1, __shfl_xor_sync(0xffffffffu, bl1, o)); bh1 = fmaxf(bh1, __shfl_xor_sync(0xffffffffu, bh1, o));
        bl2 = fminf(bl2, __shfl_xor_sync(0xffffffffu, bl2, o)); bh2 = fmaxf(bh2, __shfl_xor_sync(0xffffffffu, bh2, o));
    }
    for (int i = 0; i < P; ++i) {
        const int k = t + T * i;
        const bool ok = k < n;
        sx[k] = ok ? xyz[3 * k + 0] : 0.f;
        sy[k] = ok ? xyz[3 * k + 1] : 0.f;
        sz[k] = ok ? xyz[3 * k + 2] : 0.f;
    }
    float *new_xyz = new_xyz_all ? new_xyz_all + (size_t)blockIdx.x * m * 3 : nullptr;
    if (t == 0) idx[0] = 0;
    __syncthreads();
    float x1 = sx[0], y1 = sy[0], z1 = sz[0];
    if (t == 0 && new_xyz) {
        new_xyz[0] = x1; new_xyz[1] = y1; new_xyz[2] = z1;
    }
    const uint32_t *mykeys = skey + warp * S + lane;
    uint32_t chi = 0x7f800000u, clo = 0u;  // the warp's cached winner; +inf forces the first update

    for (int r = 1; r < m; ++r) {
        // squared distance from the pick to the slab's box (zero inside); warp-uniform
        const float ex = fmaxf(fmaxf(bl0 - x1, x1 - bh0), 0.f);
        const float ey = fmaxf(fmaxf(bl1 - y1, y1 - bh1), 0.f);
        const float ez = fmaxf(fmaxf(bl2 - z1, z1 - bh2), 0.f);
        const float dbox = ex * ex + ey * ey + ez * ez;
        if (!(dbox * 0.9999f > __uint_as_float(chi))) {
            update_min<P>(x, y, z, tm, x1, y1, z1);
            // pairwise (log-depth) arg-max; on ties the lower slot (= the smaller tie key) wins
            float bv[P];
            int bi[P];
#pragma unroll
            for (int j = 0; j < P; ++j) {
                bv[j] = tm[j];
                bi[j] = j;
            }
#pragma unroll
            for (int s2 = 1; s2 < P; s2 *= 2) {
#pragma unroll
                for (int j = 0; j + s2 < P; j += 2 * s2) {
                    const bool take = bv[j + s2] > bv[j];
                    bv[j] = take ? bv[j + s2] : bv[j];
                    bi[j] = take ? bi[j + s2] : bi[j];
                }
            }
            chi = __float_as_uint(bv[0]);
            clo = 0xFFFFFFFFu - mykeys[bi[0] * 32];
            warp_argmax(chi, clo);
        }
        uint32_t hi = chi, lo = clo;
        if (lane == 0) slot[r & 1][warp] = ((unsigned long long)hi << 32) | lo;
        __syncthreads();
        const unsigned long long v = lane < NW ? slot[r & 1][lane] : 0ull;
        hi = (uint32_t)(v >> 32);
        lo = (uint32_t)v;
        warp_argmax(hi, lo);
        const uint32_t tie = 0xFFFFFFFFu - lo;
        const int k = (int)(tie & QMASK) * 1024 + (int)(__brev(tie >> QB) >> 22);
        x1 = sx[k];
        y1 = sy[k];
        z1 = sz[k];
        if (t == 0) {
            idx[r] = k;
            if (new_xyz) {
                new_xyz[3 * r] = x1; new_xyz[3 * r + 1] = y1; new_xyz[3 * r + 2] = z1;
            }
        }
    }
}

// ---- thread-block-cluster variant ---------------------------------------------------------------------
// One CLUSTER of C CTAs per cloud (C*T threads = 1024 = the reference block size, so the tie key of a thread's
// points is still (bitrev(g) << QB) | i with g the thread's rank in the cluster).  Each round costs one quarter
// (C = 4) of the single-CTA instruction issue; the CTAs exchange their warps' winners -- key and coordinates --
// through distributed shared memory: every warp pushes one 20-byte record into each CTA of the cluster with
// st.async, whose completion is counted (complete_tx) by that CTA's mbarrier; a CTA continues when all
// NW*C = 32 records of the round have landed.  There is NO block barrier in the round; records and barriers are double
// buffered by round parity.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta));
    return r;
}


template <int T, int P, int C>
__global__ void __launch_bounds__(T, 1)
fps_cluster_kernel(int n, int m, const float *__restrict__ xyz_all, int32_t *__restrict__ idx_all,
                   float *__restrict__ new_xyz_all) {
    constexpr int NW = T / 32;
    constexpr int G = T * C;          // threads per cloud: 1024 (C = 4) or 2048 (C = 8: large sweeps, half the points per thread)
    constexpr int NREC = NW * C;      // warp records per round
    constexpr int QS = G / 1024;      // thread g owns k = g + i*G: k mod 1024 = g mod 1024, k / 1024 = QS*i + g / 1024
    constexpr int SB = NREC == 32 ? 5 : 6;  // bits of the record slot below q in the tie key
    static_assert((G == 1024 || G == 2048) && (NREC == 32 || NREC == 64), "cluster FPS: 4 or 8 CTAs of 256 threads per cloud");
    extern __shared__ float smem[];
    float *sx = smem, *sy = smem + T * P, *sz = smem + 2 * T * P;
    __shared__ __align__(16) uint4 rec[2][NREC];   // {dist bits, ~tie key, x bits, y bits}
    __shared__ float rec_z[2][NREC];
    __shared__ __align__(8) unsigned long long mbar[2];

    const uint32_t rank = cluster_ctarank();
    const int cloud = blockIdx.x / C;
    const float *xyz = xyz_all + (size_t)cloud * n * 3;
    int32_t *idx = idx_all + (size_t)cloud * m;
    float *new_xyz = new_xyz_all ? new_xyz_all + (size_t)cloud * m * 3 : nullptr;
    const int tl = threadIdx.x, lane = tl & 31, warp = tl >> 5;
    const int g = (int)rank * T + tl;

    float x[P], y[P], z[P], tm[P];
#pragma unroll
    for (int i = 0; i < P; ++i) {
        const int k = g + i * G;
        const bool ok = k < n;
        x[i] = ok ? xyz[3 * k + 0] : 0.f;
        y[i] = ok ? xyz[3 * k + 1] : 0.f;
        z[i] = ok ? xyz[3 * k + 2] : 0.f;
        tm[i] = ok ? 1e10f : 0.f;
        sx[i * T + tl] = x[i];
        sy[i * T + tl] = y[i];
        sz[i * T + tl] = z[i];
    }
    // Tie key of the cluster kernel: (bitrev10(g mod 1024) << 22) | (q << SB) | slot with q = k / 1024 = QS*i + g / 1024.
    // The slot (= g / 32, the record index of this warp) is a function of g, so appending it below q does not change
    // the order; it lets the receiver find the winning record without a ballot.
    const int my_slot = (int)rank * NW + warp;
    const uint32_t inv_base =
        0xFFFFFFFFu - (((__brev((uint32_t)(g & 1023)) >> 22) << QB) | ((uint32_t)(g >> 10) << SB) | (uint32_t)my_slot);
    if (tl == 0) {
        const uint32_t b0 = (uint32_t)__cvta_generic_to_shared(&mbar[0]);
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b0), "r"(1));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b0 + 8), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    cluster_sync_all();  // every CTA's barriers exist before anyone stores remotely

    float x1 = __ldg(xyz), y1 = __ldg(xyz + 1), z1 = __ldg(xyz + 2);
    if (g == 0) {
        idx[0] = 0;
        if (new_xyz) {
            new_xyz[0] = x1; new_xyz[1] = y1; new_xyz[2] = z1;
        }
    }
    const uint32_t rec_base = (uint32_t)__cvta_generic_to_shared(&rec[0][0]);
    const uint32_t recz_base = (uint32_t)__cvta_generic_to_shared(&rec_z[0][0]);
    const uint32_t bar_base = (uint32_t)__cvta_generic_to_shared(&mbar[0]);
    // lane d < C delivers this warp's record to CTA d: remote addresses of the warp's record slot / z slot and of the
    // barrier in THAT CTA (parity 0).  All C deliveries of a round leave in one instruction instead of a 2C-store loop
    // in the winning lane.
    const uint32_t dest = (uint32_t)lane < (uint32_t)C ? (uint32_t)lane : 0u;
    const uint32_t my_ra = map_to_cta(rec_base + (uint32_t)my_slot * 16u, dest);
    const uint32_t my_rz = map_to_cta(recz_base + (uint32_t)my_slot * 4u, dest);
    const uint32_t my_rb = map_to_cta(bar_base, dest);

    for (int j = 1; j < m; ++j) {
        const int par = j & 1;
        // arm this round's barrier: one local arrival + NREC records x 20 bytes delivered by st.async
        if (tl == 0)
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_base + (uint32_t)par * 8u), "r"(NREC * 20)
                         : "memory");
        // update the running minima, then a pairwise (log-depth) in-thread arg-max; on ties the lower i wins
        update_min<P>(x, y, z, tm, x1, y1, z1);
        float bv[P];
        int bi[P];
#pragma unroll
        for (int i = 0; i < P; ++i) {
            bv[i] = tm[i];
            bi[i] = i;
        }
#pragma unroll
        for (int s2 = 1; s2 < P; s2 *= 2) {
#pragma unroll
            for (int i = 0; i + s2 < P; i += 2 * s2) {
                // ties keep the lower i: within a pair the left operand always covers the lower indices
                const bool take = bv[i + s2] > bv[i];
                bv[i] = take ? bv[i + s2] : bv[i];
                bi[i] = take ? bi[i + s2] : bi[i];
            }
        }
        const float best = bv[0];
        const int besti = bi[0];
        const uint32_t hi = __float_as_uint(best), lo = inv_base - ((uint32_t)(QS * besti) << SB);
        uint32_t whi = hi, wlo = lo;
        warp_argmax(whi, wlo);
        {
            // the winning lane's coordinates are broadcast, then lanes 0..C-1 deliver (key, coordinates) to one CTA each;
            // completion is counted on that CTA's barrier (st.async + complete_tx: no fences, no block barrier)
            const int wl = __ffs(__ballot_sync(0xffffffffu, hi == whi && lo == wlo)) - 1;
            const float cx = __shfl_sync(0xffffffffu, sx[besti * T + tl], wl);
            const float cy = __shfl_sync(0xffffffffu, sy[besti * T + tl], wl);
            const float cz = __shfl_sync(0xffffffffu, sz[besti * T + tl], wl);
            if (lane < C) {
                asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                                 my_ra + (uint32_t)par * (NREC * 16u)),
                             "r"(whi), "r"(wlo), "r"(__float_as_uint(cx)), "r"(__float_as_uint(cy)), "r"(my_rb + (uint32_t)par * 8u)
                             : "memory");
                asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(
                                 my_rz + (uint32_t)par * (NREC * 4u)),
                             "r"(__float_as_uint(cz)), "r"(my_rb + (uint32_t)par * 8u)
                             : "memory");
            }
        }
        // wait until all NREC records of this round are in OUR shared memory
        {
            const uint32_t bar = bar_base + (uint32_t)par * 8u;
            const uint32_t parity = (uint32_t)((j - 1) >> 1) & 1u;  // each barrier is used every other round
            asm volatile(
                "{\n\t"
                ".reg .pred p;\n\t"
                "CWAIT:\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                "@p bra CDONE;\n\t"
                "bra CWAIT;\n\t"
                "CDONE:\n\t"
                "}" ::"r"(bar), "r"(parity)
                : "memory");
        }
        const uint2 key = *reinterpret_cast<const uint2 *>(&rec[par][lane]);
        uint32_t ghi = key.x, glo = key.y;
        if (NREC == 64) {  // two records per lane: keep the larger (dist, ~tie key) pair
            const uint2 k2 = *reinterpret_cast<const uint2 *>(&rec[par][lane + 32]);
            if (k2.x > ghi || (k2.x == ghi && k2.y > glo)) {
                ghi = k2.x;
                glo = k2.y;
            }
        }
        warp_argmax(ghi, glo);
        const uint32_t tie = 0xFFFFFFFFu - glo;
        const int src = (int)(tie & (uint32_t)(NREC - 1));
        const uint4 win = rec[par][src];  // broadcast read of the winning record
        x1 = __uint_as_float(win.z);
        y1 = __uint_as_float(win.w);
        z1 = rec_z[par][src];
        if (g == 0) {
            const int k = (int)((tie & QMASK) >> SB) * 1024 + (int)(__brev(tie >> QB) >> 22);
            idx[j] = k;
            if (new_xyz) {
                new_xyz[3 * j] = x1; new_xyz[3 * j + 1] = y1; new_xyz[3 * j + 2] = z1;
            }
        }
    }
    cluster_sync_all();  // nobody leaves while a peer may still write into its shared memory
}

// Any N >= 1024 with the running minima in global memory (`temp`, caller scratch as in the
// reference).  Used only when the cloud exceeds what the on-chip kernels hold.
__global__ void __launch_bounds__(1024, 1)
fps_global_kernel(int n, int m, const float *__restrict__ xyz_all, float *__restrict__ temp_all,
                  int32_t *__restrict__ idx_all, float *__restrict__ new_xyz_all) {
    constexpr int T = 1024, LG = 10;
    __shared__ unsigned long long slot[2][32];
    const float *xyz = xyz_all + (size_t)blockIdx.x * n * 3;
    float *temp = temp_all + (size_t)blockIdx.x * n;
    int32_t *idx = idx_all + (size_t)blockIdx.x * m;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int k = t; k < n; k += T) temp[k] = 1e10f;
    const uint32_t rank = __brev((uint32_t)t) >> (32 - LG);
    const uint32_t inv_base = 0xFFFFFFFFu - (rank << QB);
    float *new_xyz = new_xyz_all ? new_xyz_all + (size_t)blockIdx.x * m * 3 : nullptr;
    float x1 = xyz[0], y1 = xyz[1], z1 = xyz[2];
    if (t == 0) {
        idx[0] = 0;
        if (new_xyz) {
            new_xyz[0] = x1; new_xyz[1] = y1; new_xyz[2] = z1;
        }
    }
    for (int j = 1; j < m; ++j) {
        float best = -1.f;
        int bestq = 0;
        for (int k = t, q = 0; k < n; k += T, ++q) {
            const float d = dist_ref(xyz[3 * k], xyz[3 * k + 1], xyz[3 * k + 2], x1, y1, z1);
            const float d2 = fminf(d, temp[k]);
            temp[k] = d2;
            if (d2 > best) {
                best = d2;
                bestq = q;
            }
        }
        uint32_t hi = __float_as_uint(best), lo = inv_base - (uint32_t)bestq;
        warp_argmax(hi, lo);
        if (lane == 0) slot[j & 1][warp] = ((unsigned long long)hi << 32) | lo;
        __syncthreads();
        const unsigned long long v = slot[j & 1][lane];
        hi = (uint32_t)(v >> 32);
        lo = (uint32_t)v;
        warp_argmax(hi, lo);
        const uint32_t tie = 0xFFFFFFFFu - lo;
        const int k = (int)(tie & QMASK) * T + (int)(__brev(tie >> QB) >> (32 - LG));
        x1 = xyz[3 * k];
        y1 = xyz[3 * k + 1];
        z1 = xyz[3 * k + 2];
        if (t == 0) {
            idx[j] = k;
            if (new_xyz) {
                new_xyz[3 * j] = x1; new_xyz[3 * j + 1] = y1; new_xyz[3 * j + 2] = z1;
            }
        }
    }
}

// N < 32: one thread per cloud walks the total order directly.
__global__ void fps_tiny_kernel(int b, int n, int m, int bs, int lg, const float *__restrict__ xyz_all,
                                int32_t *__restrict__ idx_all, float *__restrict__ new_xyz_all) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= b) return;
    const float *xyz = xyz_all + (size_t)c * n * 3;
    int32_t *idx = idx_all + (size_t)c * m;
    float tm[32];
    for (int k = 0; k < n; ++k) tm[k] = 1e10f;
    float *new_xyz = new_xyz_all ? new_xyz_all + (size_t)c * m * 3 : nullptr;
    int old = 0;
    idx[0] = 0;
    for (int j = 1; j <= m; ++j) {
        const float x1 = xyz[3 * old], y1 = xyz[3 * old + 1], z1 = xyz[3 * old + 2];
        if (new_xyz) {
            new_xyz[3 * (j - 1)] = x1; new_xyz[3 * (j - 1) + 1] = y1; new_xyz[3 * (j - 1) + 2] = z1;
        }
        if (j == m) break;
        float best = -1.f;
        uint32_t best_rank = 0;
        int besti = 0;
        for (int k = 0; k < n; ++k) {
            const float d2 = fminf(dist_ref(xyz[3 * k], xyz[3 * k + 1], xyz[3 * k + 2], x1, y1, z1), tm[k]);
            tm[k] = d2;
            const uint32_t rk = lg ? (__brev((uint32_t)(k & (bs - 1))) >> (32 - lg)) : 0u;
            if (d2 > best || (d2 == best && rk < best_rank)) {
                best = d2;
                best_rank = rk;
                besti = k;
            }
        }
        old = besti;
        idx[j] = old;
    }
}

template <int T, int P>
int launch_reg(int b, int n, int m, const float *xyz, int32_t *idx, float *new_xyz, cudaStream_t s) {
    const size_t smem = (size_t)3 * T * P * sizeof(float);
    if (smem > 40 * 1024)  // static shared memory (the reduction slots) counts against the 48 KB default too
        PN2_CUDA(cudaFuncSetAttribute(fps_reg_kernel<T, P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fps_reg_kernel<T, P><<<b, T, smem, s>>>(n, m, xyz, idx, new_xyz);
    PN2_LAUNCH_OK("fps_reg_kernel");
    return PN2_OK;
}

template <int Q>
int launch_few(int b, int n, int m, const float *xyz, int32_t *idx, float *new_xyz, cudaStream_t s) {
    const size_t smem = (size_t)3 * 1024 * Q * sizeof(float);
    PN2_CUDA(cudaFuncSetAttribute(fps_few_kernel<Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fps_few_kernel<Q><<<b, 256, smem, s>>>(n, m, xyz, idx, new_xyz);
    PN2_LAUNCH_OK("fps_few_kernel");
    return PN2_OK;
}

template <int Q>
int launch_slab(int b, int n, int m, const float *xyz, int32_t *idx, float *new_xyz, cudaStream_t s) {
    const size_t smem = (size_t)4 * 1024 * Q * sizeof(float);  // coordinates by index + tie keys by slab position
    PN2_CUDA(cudaFuncSetAttribute(fps_slab_kernel<Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fps_slab_kernel<Q><<<b, 256, smem, s>>>(n, m, xyz, idx, new_xyz);
    PN2_LAUNCH_OK("fps_slab_kernel");
    return PN2_OK;
}

template <int P, int C = 4, int T = 256>
int launch_cluster(int b, int n, int m, const float *xyz, int32_t *idx, float *new_xyz, cudaStream_t s) {
    const size_t smem = (size_t)3 * T * P * sizeof(float);
    if (smem > 40 * 1024)
        PN2_CUDA(cudaFuncSetAttribute(fps_cluster_kernel<T, P, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)b * C);
    cfg.blockDim = dim3(T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    PN2_CUDA(cudaLaunchKernelEx(&cfg, fps_cluster_kernel<T, P, C>, n, m, xyz, idx, new_xyz));
    count_launch();
    return PN2_OK;
}

template <int T>
int launch_reg_small(int b, int n, int m, const float *xyz, int32_t *idx, float *new_xyz, cudaStream_t s) {
    return n <= T ? launch_reg<T, 1>(b, n, m, xyz, idx, new_xyz, s) : launch_reg<T, 2>(b, n, m, xyz, idx, new_xyz, s);
}

}  // namespace
}  // namespace pn2

// PN2_FPS_AUTO / PN2_FPS_ONE_CTA / PN2_FPS_CLUSTER (see fps_impl)
static int g_fps_policy = PN2_FPS_AUTO;
extern "C" int pn2_set_fps_policy(int policy) {
    if (policy < PN2_FPS_AUTO || policy > PN2_FPS_CLUSTER) return -1;
    const int prev = g_fps_policy;
    g_fps_policy = policy;
    return prev;
}
extern "C" void pn2_debug_set_fps_mode(int mode) { pn2_set_fps_policy(mode); }

namespace pn2 {
namespace {
int fps_impl(int b, int n, int m, const float *xyz, float *temp, int32_t *idx, float *new_xyz, void *stream) {
    PN2_REQUIRE(b >= 0 && n >= 1, "fps: need b >= 0 and n >= 1 (got b=%d n=%d)", b, n);
    if (b == 0 || m <= 0) return PN2_OK;  // the reference kernel returns at once for m <= 0 (sampling_gpu.cu:101)
    PN2_REQUIRE(xyz && idx, "fps: null pointer");
    PN2_REQUIRE((long long)n < (1ll << 31) / 3, "fps: n too large");
    cudaStream_t s = (cudaStream_t)stream;
    const int T = ref_block_size(n);
    if (T < 32) {
        int lg = 0;
        while ((1 << lg) < T) ++lg;
        fps_tiny_kernel<<<ceil_div(b, 64), 64, 0, s>>>(b, n, m, T, lg, xyz, idx, new_xyz);
        PN2_LAUNCH_OK("fps_tiny_kernel");
        return PN2_OK;
    }
    switch (T) {
        case 32: return launch_reg_small<32>(b, n, m, xyz, idx, new_xyz, s);
        case 64: return launch_reg_small<64>(b, n, m, xyz, idx, new_xyz, s);
        case 128: return launch_reg_small<128>(b, n, m, xyz, idx, new_xyz, s);
        case 256: return launch_reg_small<256>(b, n, m, xyz, idx, new_xyz, s);
        case 512: return launch_reg_small<512>(b, n, m, xyz, idx, new_xyz, s);
        default: break;
    }
    if (n == 1024) return launch_few<1>(b, n, m, xyz, idx, new_xyz, s);  // 4 points per thread
    if (n <= 1024) return launch_reg<1024, 1>(b, n, m, xyz, idx, new_xyz, s);
    // 1024 < n <= 8192.  One CTA per cloud = the 256-thread kernel (fps_few_kernel): 0.12 / 0.17 / 0.54 ms for
    // 2048->512 / 4096->512 / 8192->1024, faster than both alternatives up to 4096 points.  At 4096 < n <= 8192 the
    // 4-CTA cluster is 17 % faster (0.45 ms) but occupies four SMs per cloud: chosen automatically only while the
    // clouds alone cannot fill the GPU; PN2_FPS_ONE_CTA keeps one SM per cloud (several batches in flight).
    const int policy = g_fps_policy;
    const bool cluster_ok = (long long)b * 4 <= sm_count();
    const bool use_cluster = n > 8192 || policy == PN2_FPS_CLUSTER || (policy == PN2_FPS_AUTO && n > 4096 && cluster_ok);
    if (use_cluster) {
        // large sweeps: 8 CTAs per cloud (half the points per thread) while the clusters still fit the GPU in one wave
        if (n <= 2048) return launch_cluster<2>(b, n, m, xyz, idx, new_xyz, s);
        if (n <= 4096) return launch_cluster<4>(b, n, m, xyz, idx, new_xyz, s);
        if (n <= 8192) return launch_cluster<8>(b, n, m, xyz, idx, new_xyz, s);
        if (n <= 16384) return launch_cluster<16>(b, n, m, xyz, idx, new_xyz, s);
        if (n <= 24576) return launch_cluster<24>(b, n, m, xyz, idx, new_xyz, s);
        if (n <= 32768) return launch_cluster<32>(b, n, m, xyz, idx, new_xyz, s);
        if (n <= 36864) return launch_cluster<36>(b, n, m, xyz, idx, new_xyz, s);  // a raw ~35k-point lidar sweep: no padded slots
        if (n <= 40960) return launch_cluster<40>(b, n, m, xyz, idx, new_xyz, s);
        if (n <= 49152) return launch_cluster<48>(b, n, m, xyz, idx, new_xyz, s);
        // 8 CTAs per cloud keep clouds of up to 65536 points on chip.  (For smaller clouds the 8-CTA exchange costs more
        // than the halved per-thread work saves: 16 sweeps x 34720 points 1789 -> 1483 sweeps/s, so 4 CTAs stay the default;
        // 512-thread CTAs -- 18 points per thread -- were no faster either: 0.80 vs 0.74 us per round.)
        if (n <= 65536) return launch_cluster<32, 8>(b, n, m, xyz, idx, new_xyz, s);
    } else {
        if (n <= 2048) return launch_few<2>(b, n, m, xyz, idx, new_xyz, s);
        // spatial slabs per warp + skipped rounds: pays once enough points are picked for the running minima to fall
        // below the slab distances (a few hundred picks)
        // (at 4096 points the slab kernel's set-up and per-round test cost more than the skipped rounds save)
        if (n <= 4096) return launch_few<4>(b, n, m, xyz, idx, new_xyz, s);
        return m >= 128 ? launch_slab<8>(b, n, m, xyz, idx, new_xyz, s) : launch_few<8>(b, n, m, xyz, idx, new_xyz, s);
    }
    if (!temp)
        return set_error(PN2_ERR_INVALID_ARGUMENT, "fps: n=%d exceeds the on-chip kernels; pass the (B,N) temp scratch", n);
    PN2_REQUIRE(n < (long long)(QMASK) * 1024ll, "fps: n too large for the tie key");
    fps_global_kernel<<<b, 1024, 0, s>>>(n, m, xyz, temp, idx, new_xyz);
    PN2_LAUNCH_OK("fps_global_kernel");
    return PN2_OK;
}
}  // namespace
}  // namespace pn2

extern "C" int pn2_furthest_point_sampling(int b, int n, int m, const float *xyz, float *temp, int32_t *idx,
                                           void *stream) {
    return pn2::fps_impl(b, n, m, xyz, temp, idx, nullptr, stream);
}

extern "C" int pn2_fps_gather(int b, int n, int m, const float *xyz, float *temp, int32_t *idx, float *new_xyz,
                              void *stream) {
    if (m > 0 && b > 0 && !new_xyz) return pn2::set_error(PN2_ERR_INVALID_ARGUMENT, "fps_gather: null new_xyz");
    return pn2::fps_impl(b, n, m, xyz, temp, idx, new_xyz, stream);
}
