// row_mlp_tc.cu -- fused "gather -> shared MLP -> pool/store" blocks on the 5th-gen tensor cores (bf16
// operands, fp32 accumulation in TMEM).  Same operator contract as row_mlp.cu (the fp32 path); outputs
// agree with it within bf16 rounding (2e-2 relative, BASELINE.json north_star; measured ~4e-3).
//
// PERSISTENT CTAs (2-4 per SM) walk tiles of 128 rows (= UMMA M); barriers, TMEM and biases are set up once.
// For every layer
//     D[128 x N] (TMEM, fp32) = A[128 x K] (smem, bf16, K-major, 128B swizzle) * W[N x K]^T (smem, same layout)
//   * A of layer 0 is written by the gather (grouped features + centred xyz, or 3-NN interpolation + skip rows),
//     in CHUNKS of whole 64-column k-blocks: the MMAs of a chunk accumulate into TMEM while the buffer is refilled,
//     so inputs of any width stream through a 32-64 KB operand buffer (fp4's 768 / 1536 channels included).  A last
//     k-block of only 16 columns (the xyz / colour tail) lives in its own 4 KB un-swizzled region and rides with the
//     last chunk.  bf16 feature rows are gathered warp-cooperatively (consecutive lanes = consecutive 16 bytes of one
//     source row); the index-level loads of tile i+1 are issued while the layers of tile i run;
//   * A of layer l+1 is written by the epilogue of layer l straight from TMEM (tcgen05.ld, bias, ReLU, bf16 pack --
//     packed f32x2 / bf16x2 math) into the SAME buffer: all MMAs of a layer are committed before its epilogue runs;
//   * W arrives as pre-swizzled tiles (packed once by pn2_mlp_pack_bf16; 64/128/256 rows chosen for residency)
//     through a 2-4-stage ring of bulk-async copies (cp.async.bulk = TMA unit, mbarrier complete_tx) that runs ahead
//     across layer AND tile boundaries;
//   * tcgen05.mma is issued by one elected lane of a warp that walks the schedule in uniform control flow;
//   * SA blocks compute their LAST layer transposed (D^T = W A^T: channels on TMEM lanes, the 128 samples on columns),
//     so the max over nsample is a register-local tree and bias + ReLU are applied once per group; FP blocks store rows
//     with 128-bit stores, or only the arg-max of the row (PN2_FLAG_OUT_ARGMAX);
//   * activations that only travel between such blocks are read / written as bf16 (PN2_FLAG_*), halving gather
//     traffic; FP rows can be processed in a spatially sorted order (row_perm) so neighbouring rows share their three
//     coarse rows in L1.
// Warp roles: 0-3 gather + epilogue (TMEM lanes 32w..32w+31), 4 weight producer, 5 TMEM alloc + MMA issue.
// Measured behaviour and the experiments behind these choices: profiles/README.md.
#include <cuda_bf16.h>

#include "common.cuh"

namespace pn2 {
namespace {

constexpr int TC_THREADS = 192;      // 4 worker warps + producer + issuer
constexpr int TC_THREADS_W8 = 320;   // 8 worker warps (two per TMEM lane quarter, splitting the columns) + producer + issuer
constexpr int TC_ROWS = 128;
constexpr int KBLK = 64;                       // bf16 elements per 128-byte swizzle row
constexpr int A_BLOCK_BYTES = TC_ROWS * 128;   // one k-block of A: 128 rows x 128 B
constexpr int MAX_STAGES = 4;
#ifndef PN2_FP_GATHER_U
#define PN2_FP_GATHER_U 2
#endif
// FP gather: 16-byte items per lane and batch (x3 neighbour rows in flight).  Measured, fp1+head: 2 -> 107 us, 4 -> 117 us
// (the 96-register budget of 3 CTAs x 6 warps spills inside the loop); weights shuffled before the loads: 125 us.
constexpr int FP_GATHER_U = PN2_FP_GATHER_U;

enum { MODE_SA = 0, MODE_FP = 1 };

struct TcLayer {
    int cin, cout;       // logical widths
    int kpad;            // cin rounded up to 16 (MMA K granularity)
    int npad;            // cout rounded up to 32 (MMA N, and the epilogue's 32-column loads)
    int nblk;            // rows of one weight tile: min(npad, 256)
    int nnb, nkb;        // npad / nblk weight tiles along N, ceil(kpad / 64) k-blocks (host-computed: no device divisions)
    int relu;
    const float *bias;
    long long w_off;     // byte offset of this layer's first tile in the packed buffer
    int bias_off;        // float offset of this layer's (zero padded) bias in the shared-memory copy
};

struct TcParams {
    int mode, num_layers;
    TcLayer layer[PN2_MAX_LAYERS];
    const unsigned char *packed;
    int stages, stage_bytes, a_bytes, tmem_cols, bias_floats;
    long long tiles;
    // SA
    int n, m, k, d;
    long long groups;
    const float *xyz, *feat, *new_xyz;
    const int32_t *idx;
    float *out;
    int out_stride, out_offset;
    // FP
    long long rows;
    int d1, d2, fp_m;
    const float *feat1, *feat2, *weight;
    int feat_aligned;  // gathered feature rows are 16-byte aligned (float4 loads allowed)
    const int32_t *row_perm;  // FP: optional (B, n) processing order (index within the cloud)
    int in_bf16;       // block0 features (SA feat / FP feat2) are stored as bf16
    int skip_bf16;     // FP skip features (feat1) are stored as bf16
    int out_bf16;      // write the result as bf16 (activations that only feed another tensor-core block)
    int out_argmax;    // FP: write one uint8 per row, the index of the largest output channel (first on ties)
    int kchunk;        // k-blocks of the first layer's operand produced per pass (see gather_chunk_tc)
    int pool_t;        // SA: the last layer is computed TRANSPOSED (channels on TMEM lanes, samples on columns; see kernel)
    int thin;          // the first layer's last k-block holds only 16 columns and lives in its own 4 KB region (see Plan)
    int pool_dup;      // SA, transposed last layer of <= 64 channels: its weight block is loaded 128 / npad times into the
                       // 128-row M operand, so every TMEM lane quarter holds real channels and each worker warp pools
                       // 128 / pool_dup of the tile's samples (otherwise only npad / 32 of the four warps would work)
    long long *dbg;    // optional phase timestamps of CTA 0 / warp 0 (developer profiling; NULL in production)
};

// ---- PTX helpers ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Blocking wait.  The suspend-time hint lets the hardware park the thread until the phase completes (or the hint
// expires) instead of spinning: without it the polling loops of the producer / MMA lanes and of the epilogue warps
// were ~40 % of all issued instructions (ncu, profiles/r1_tc_mlp_v2_*), stealing issue slots from the working warps.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(bar), "r"(parity), "r"(0x989680u)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// Issuer-warp variants: the WHOLE warp runs the schedule in uniform control flow and `leader` (one elected lane)
// predicates the instruction; the descriptors' high words are constant (SBO 1024 B, version 1, SWIZZLE_128B) and only
// the 14-bit start-address field of the low word moves, so a step along K is one 32-bit add.
constexpr uint32_t DESC_HI = 0x40004040u;        // SBO 1024 B | version 1 | SWIZZLE_128B
constexpr uint32_t DESC_HI_THIN = 0x00004010u;   // SBO 256 B | version 1 | no swizzle (core-matrix layout)
__device__ __forceinline__ uint32_t desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, q;\n\t"
        "}"
        : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void tc_mma_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                          uint32_t idesc, uint32_t accumulate, uint32_t leader) {
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        ".reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %7};\n\t"
        "mov.b64 db, {%2, %6};\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
        "}" ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(leader), "r"(b_hi), "r"(a_hi)
        : "memory");
}
__device__ __forceinline__ void tc_commit_if(uint32_t bar, uint32_t leader) {
    asm volatile(
        "{\n\t"
        ".reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
        "}" ::"r"(bar), "r"(leader)
        : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread t <-> lane base + t)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory descriptors (cute/arch/mma_sm100_desc.hpp): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout type [61,64).  Operands are K-major with 128-byte swizzle and 8-row groups 1024 B apart
// (desc_lo / DESC_HI above); the thin tail block is K-major without swizzle (DESC_HI_THIN).
// Instruction descriptor: D fp32, A/B bf16, both K-major, M = 128, N = n  (cute UMMA::InstrDescriptor)
__device__ __forceinline__ uint32_t umma_idesc(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TC_ROWS >> 4) << 24);
}

// two fp32 values -> packed bf16x2 (lo in the low half), optionally with ReLU in the same instruction
__device__ __forceinline__ uint32_t cvt_bf16x2(float lo, float hi, int relu) {
    uint32_t d;
    if (relu)
        asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    else
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// One 32-column chunk of a hidden layer's epilogue for one row: acc + bias -> (ReLU) -> bf16, written as four 16-byte
// slots of the next layer's swizzled operand (dst0 = row base + k-block, x0 = swizzle term of the chunk's first slot).
__device__ __forceinline__ void lds128(uint32_t addr, float4 &v) {
    asm("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4 &v) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
template <bool kRelu>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&acc)[32], uint32_t bsrc, uint32_t dst0, uint32_t x0) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float4 b0, b1;
        lds128(bsrc + 32u * q, b0);
        lds128(bsrc + 32u * q + 16u, b1);
        const float2 s0 = __fadd2_rn(make_float2(__uint_as_float(acc[8 * q + 0]), __uint_as_float(acc[8 * q + 1])), make_float2(b0.x, b0.y));
        const float2 s1 = __fadd2_rn(make_float2(__uint_as_float(acc[8 * q + 2]), __uint_as_float(acc[8 * q + 3])), make_float2(b0.z, b0.w));
        const float2 s2 = __fadd2_rn(make_float2(__uint_as_float(acc[8 * q + 4]), __uint_as_float(acc[8 * q + 5])), make_float2(b1.x, b1.y));
        const float2 s3 = __fadd2_rn(make_float2(__uint_as_float(acc[8 * q + 6]), __uint_as_float(acc[8 * q + 7])), make_float2(b1.z, b1.w));
        uint4 pk;
        pk.x = cvt_bf16x2(s0.x, s0.y, kRelu); pk.y = cvt_bf16x2(s1.x, s1.y, kRelu);
        pk.z = cvt_bf16x2(s2.x, s2.y, kRelu); pk.w = cvt_bf16x2(s3.x, s3.y, kRelu);
        sts128(dst0 + (x0 ^ (uint32_t)(q << 4)), pk);
    }
}

// 16-column TMEM loads with the wait split off, so the load of the NEXT piece is in flight while the current one is
// processed (tcgen05.wait::ld waits for every outstanding load of the thread: it is issued for piece i, then the load of
// piece i+1, then piece i is processed).  The wait takes the destination registers as in/out operands so that no use of
// them can be scheduled above it.
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16_wait(uint32_t (&r)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :
                 : "memory");
}
// One 16-column piece of a hidden layer's epilogue for one row (two 16-byte slots of the next layer's operand).
template <bool kRelu>
__device__ __forceinline__ void epilogue_piece(const uint32_t (&acc)[16], uint32_t bsrc, uint32_t dst0, uint32_t x0) {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        float4 b0, b1;
        lds128(bsrc + 32u * q, b0);
        lds128(bsrc + 32u * q + 16u, b1);
        const float2 s0 = __fadd2_rn(make_float2(__uint_as_float(acc[8 * q + 0]), __uint_as_float(acc[8 * q + 1])), make_float2(b0.x, b0.y));
        const float2 s1 = __fadd2_rn(make_float2(__uint_as_float(acc[8 * q + 2]), __uint_as_float(acc[8 * q + 3])), make_float2(b0.z, b0.w));
        const float2 s2 = __fadd2_rn(make_float2(__uint_as_float(acc[8 * q + 4]), __uint_as_float(acc[8 * q + 5])), make_float2(b1.x, b1.y));
        const float2 s3 = __fadd2_rn(make_float2(__uint_as_float(acc[8 * q + 6]), __uint_as_float(acc[8 * q + 7])), make_float2(b1.z, b1.w));
        uint4 pk;
        pk.x = cvt_bf16x2(s0.x, s0.y, kRelu); pk.y = cvt_bf16x2(s1.x, s1.y, kRelu);
        pk.z = cvt_bf16x2(s2.x, s2.y, kRelu); pk.w = cvt_bf16x2(s3.x, s3.y, kRelu);
        sts128(dst0 + (x0 ^ (uint32_t)(q << 4)), pk);
    }
}

// byte offset of the 16-byte chunk holding elements [8*c8, 8*c8+8) of row r in a [rows x K] operand
__device__ __forceinline__ uint32_t swz_chunk(int r, int c8, int rows) {
    const int kb = c8 >> 3, c = c8 & 7;
    return (uint32_t)(kb * rows * 128 + r * 128 + ((c ^ (r & 7)) << 4));
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&v);
}

// Where the gather puts the 8-column chunk c8 of row r.  Chunks of whole 64-column k-blocks go to the swizzled pass
// buffer (relative to the first chunk of the pass); the chunks of a THIN last k-block (16 columns: the xyz / colour
// tail of most layers) go to a separate 4 KB region in the un-swizzled K-major core-matrix layout
// (8 rows x 16 B contiguous, K step 128 B, 8-row groups 256 B apart), so the tail never costs a pass of its own.
struct ADst {
    unsigned char *a;
    int r, c8_begin, thin_c8;
    uint32_t thin_off;
    __device__ __forceinline__ unsigned char *operator()(int c8) const {
        if (c8 >= thin_c8) return a + thin_off + ((r >> 3) << 8) + ((c8 - thin_c8) << 7) + ((r & 7) << 4);
        return a + swz_chunk(r, c8 - c8_begin, TC_ROWS);
    }
};

__device__ __forceinline__ void st_chunk(unsigned char *dst, const float (&v)[8]) {
    uint4 q;
    q.x = pack_bf16(v[0], v[1]);
    q.y = pack_bf16(v[2], v[3]);
    q.z = pack_bf16(v[4], v[5]);
    q.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4 *>(dst) = q;
}

// ---- layer-0 operand: one thread per row, layout [block0 | block1 | zero pad] ---------------------------
// SA: block0 = grouped features (D), block1 = centred xyz (3).  FP: block0 = interpolated (D2), block1 = skip (D1).
// (pn2_mlp_pack_bf16 permutes the first layer's weight columns to this order.)
// The operand is produced in chunks of whole k-blocks [c8_begin, c8_end) (8-column units), written at the start of
// the A buffer, so arbitrarily wide inputs stream through a small buffer while the MMAs accumulate in TMEM.
struct RowCtx {
    bool ok;
    long long src0, src1, src2;  // element offsets of the gathered feature row(s): SA uses src0, FP all three
    // SA
    const float *f;
    float dx, dy, dz;
    // FP
    const float *r0, *r1, *r2, *f1;
    float w0, w1, w2;
    long long out_row;  // FP: destination row (after the optional permutation)
};

// What a row needs from "index" memory (sample index / 3-NN indices and weights, centred xyz): 9 registers, loaded for
// tile i+1 while the layers of tile i run, so the gather of a tile starts with its second-level loads.
struct RowPre {
    bool ok;
    int i0, i1, i2;     // SA: i0 = global source row (b*n + pt).  FP: global coarse rows (b*m + idx)
    float a, b, c;      // SA: centred xyz.  FP: interpolation weights
    long long row;      // FP: destination row (after the optional permutation)
};

template <int kMode>
__device__ __forceinline__ RowPre row_prefetch(const TcParams &p, long long tile, int r) {
    RowPre c = {};
    if (tile >= p.tiles) return c;
    if ((kMode == MODE_SA)) {
        const int K = p.k;
        const int lgK = 31 - __clz(K);  // nsample is a power of two
        const int gpt = TC_ROWS >> lgK;  // groups per tile
        const int g0 = (int)tile * gpt;
        const int g = g0 + (r >> lgK);
        c.ok = g < (int)p.groups;
        if (c.ok) {
            // the batch index of the tile's first group is uniform; a tile spans at most two clouds when gpt <= m
            int b = g0 / p.m;
            b = gpt <= p.m ? b + (g >= (b + 1) * p.m) : g / p.m;
            const int pt = __ldg(p.idx + (size_t)g * K + (r & (K - 1)));
            const int src = b * p.n + pt;
            c.i0 = src;
            c.a = __fsub_rn(__ldg(p.xyz + (size_t)src * 3 + 0), __ldg(p.new_xyz + (size_t)g * 3 + 0));
            c.b = __fsub_rn(__ldg(p.xyz + (size_t)src * 3 + 1), __ldg(p.new_xyz + (size_t)g * 3 + 1));
            c.c = __fsub_rn(__ldg(p.xyz + (size_t)src * 3 + 2), __ldg(p.new_xyz + (size_t)g * 3 + 2));
        }
    } else {
        const int row0 = (int)tile * TC_ROWS;
        int row = row0 + r;
        c.ok = row < (int)p.rows;
        if (c.ok) {
            int b = row0 / p.n;  // uniform; a tile spans at most two clouds when n >= 128
            b = TC_ROWS <= p.n ? b + (row >= (b + 1) * p.n) : row / p.n;
            if (p.row_perm) row = b * p.n + __ldg(p.row_perm + row);  // spatially coherent processing order
            if (p.fp_m == 1) {
                c.i0 = c.i1 = c.i2 = b;  // S == 1: the coarse row is repeated
                c.a = 1.f;
            } else {
                const int32_t *id = p.idx + (size_t)row * 3;
                const float *w = p.weight + (size_t)row * 3;
                c.i0 = b * p.fp_m + __ldg(id);
                c.i1 = b * p.fp_m + __ldg(id + 1);
                c.i2 = b * p.fp_m + __ldg(id + 2);
                c.a = __ldg(w); c.b = __ldg(w + 1); c.c = __ldg(w + 2);
            }
        }
        c.row = row;
    }
    return c;
}

template <int kMode>
__device__ __forceinline__ RowCtx row_expand(const TcParams &p, const RowPre &q) {
    RowCtx c = {};
    c.ok = q.ok;
    if ((kMode == MODE_SA)) {
        c.src0 = (long long)q.i0 * p.d;
        c.f = p.feat + c.src0;
        c.dx = q.a; c.dy = q.b; c.dz = q.c;
    } else {
        const long long D2 = p.d2;
        c.src0 = q.i0 * D2; c.src1 = q.i1 * D2; c.src2 = q.i2 * D2;
        c.r0 = p.feat2 + c.src0; c.r1 = p.feat2 + c.src1; c.r2 = p.feat2 + c.src2;
        c.w0 = q.a; c.w1 = q.b; c.w2 = q.c;
        c.f1 = p.feat1 + q.row * p.d1;
        c.out_row = q.row;
    }
    return c;
}

template <bool kInBf16, int kMode>
__device__ __forceinline__ void gather_tail_tc(const TcParams &p, const RowCtx &x, const ADst &dst, int c8_from, int c8_end,
                                               const float (&sk)[8], bool sk_valid) {
    const bool ok = x.ok;
    if constexpr (kInBf16) {
        // bf16 activations: a 16-byte load is a whole 8-column chunk.  SA: the chunk IS the operand chunk (pure copy,
        // bit-identical to converting fp32 features here); FP: three chunks are unpacked, interpolated in fp32, repacked.
        const int Dm = (kMode == MODE_SA) ? p.d : p.d2;
        const __nv_bfloat16 *b0 = reinterpret_cast<const __nv_bfloat16 *>((kMode == MODE_SA) ? (const void *)p.feat : (const void *)p.feat2);
        const bool fp3 = (kMode != MODE_SA) && p.fp_m != 1;
        int c8 = c8_from;
        const int c8_blk0 = min(c8_end, Dm / 8);
        for (; c8 < c8_blk0; c8 += 4) {
            const int nq = min(4, c8_blk0 - c8);
            uint4 q0[4], q1[4], q2[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                q0[q] = make_uint4(0u, 0u, 0u, 0u);
                q1[q] = q0[q];
                q2[q] = q0[q];
                if (q < nq && ok) {
                    q0[q] = __ldg(reinterpret_cast<const uint4 *>(b0 + x.src0) + c8 + q);
                    if (fp3) {
                        q1[q] = __ldg(reinterpret_cast<const uint4 *>(b0 + x.src1) + c8 + q);
                        q2[q] = __ldg(reinterpret_cast<const uint4 *>(b0 + x.src2) + c8 + q);
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (q >= nq) break;
                uint4 o = q0[q];
                if (fp3) {
                    const uint32_t *u0 = reinterpret_cast<const uint32_t *>(&q0[q]);
                    const uint32_t *u1 = reinterpret_cast<const uint32_t *>(&q1[q]);
                    const uint32_t *u2 = reinterpret_cast<const uint32_t *>(&q2[q]);
                    uint32_t *uo = reinterpret_cast<uint32_t *>(&o);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        // bf16 -> fp32 is a 16-bit shift; same rn sequence as three_interpolate
                        const float a0l = __uint_as_float(u0[e] << 16), a0h = __uint_as_float(u0[e] & 0xffff0000u);
                        const float a1l = __uint_as_float(u1[e] << 16), a1h = __uint_as_float(u1[e] & 0xffff0000u);
                        const float a2l = __uint_as_float(u2[e] << 16), a2h = __uint_as_float(u2[e] & 0xffff0000u);
                        const float lo = __fmaf_rn(x.w2, a2l, __fmaf_rn(x.w0, a0l, __fmul_rn(x.w1, a1l)));
                        const float hi = __fmaf_rn(x.w2, a2h, __fmaf_rn(x.w0, a0h, __fmul_rn(x.w1, a1h)));
                        uo[e] = pack_bf16(lo, hi);
                    }
                }
                *reinterpret_cast<uint4 *>(dst(c8 + q)) = o;
            }
        }
        // skip features stored as bf16 and chunk aligned: pure copies as well
        if ((kMode != MODE_SA) && p.skip_bf16 && (Dm & 7) == 0 && (p.d1 & 7) == 0) {
            const __nv_bfloat16 *b1 = reinterpret_cast<const __nv_bfloat16 *>(p.feat1);
            const int c8_skip_end = min(c8_end, (Dm + p.d1) / 8);
            for (; c8 < c8_skip_end; ++c8) {
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (ok) o = __ldg(reinterpret_cast<const uint4 *>(b1 + x.out_row * p.d1) + (c8 - Dm / 8));
                *reinterpret_cast<uint4 *>(dst(c8)) = o;
            }
        }
        // remaining chunks: centred xyz (SA) / fp32 skip channels (FP) / zero padding
        for (; c8 < c8_end; ++c8) {
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = c8 * 8 + j;
                float y = 0.f;
                if (ok) {
                    if ((kMode == MODE_SA)) {
                        if (c < Dm) y = __bfloat162float(b0[x.src0 + c]);
                        else if (c == Dm) y = x.dx;
                        else if (c == Dm + 1) y = x.dy;
                        else if (c == Dm + 2) y = x.dz;
                    } else if (c < Dm) {
                        y = fp3 ? __fmaf_rn(x.w2, __bfloat162float(b0[x.src2 + c]),
                                            __fmaf_rn(x.w0, __bfloat162float(b0[x.src0 + c]), __fmul_rn(x.w1, __bfloat162float(b0[x.src1 + c]))))
                                : __bfloat162float(b0[x.src0 + c]);
                    } else if (sk_valid && c8 == (Dm >> 3)) {
                        y = sk[j];  // narrow fp32 skip block, loaded at the start of the tile
                    } else if (c < Dm + p.d1) {
                        y = p.skip_bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(p.feat1)[x.out_row * p.d1 + (c - Dm)])
                                        : __ldg(p.feat1 + x.out_row * p.d1 + (c - Dm));
                    }
                }
                v[j] = y;
            }
            st_chunk(dst(c8), v);
        }
        return;
    } else if ((kMode == MODE_SA)) {
        const int D = p.d;
        const float *f = x.f;
        if (D <= 5) {
            // narrow input (xyz-only or xyz + colour levels): features and centred xyz fit the first 8-column chunk and
            // every other chunk is zero padding -- no per-element branches
            for (int c8 = c8_from; c8 < c8_end; ++c8) {
                float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                if (c8 == 0 && ok) {
#pragma unroll
                    for (int j = 0; j < 5; ++j)
                        if (j < D) v[j] = __ldg(f + j);
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = j == D ? x.dx : (j == D + 1 ? x.dy : (j == D + 2 ? x.dz : v[j]));
                }
                st_chunk(dst(c8), v);
            }
            return;
        }
        const bool vec = ok && (D % 4 == 0) && p.feat_aligned;
        int c8 = c8_from;
        if (vec) {
            // 4 chunks (32 channels, 8 x LDG.128) in flight per thread before the first use
            for (; c8 + 4 <= c8_end && (c8 + 4) * 8 <= D; c8 += 4) {
                float4 u[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) u[q] = __ldg(reinterpret_cast<const float4 *>(f + c8 * 8 + 4 * q));
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float v[8] = {u[2 * q].x, u[2 * q].y, u[2 * q].z, u[2 * q].w,
                                        u[2 * q + 1].x, u[2 * q + 1].y, u[2 * q + 1].z, u[2 * q + 1].w};
                    st_chunk(dst(c8 + q), v);
                }
            }
        }
        for (; c8 < c8_end; ++c8) {
            float v[8];
            const int c0 = c8 * 8;
            if (vec && c0 + 8 <= D) {
                const float4 u0 = __ldg(reinterpret_cast<const float4 *>(f + c0));
                const float4 u1 = __ldg(reinterpret_cast<const float4 *>(f + c0 + 4));
                v[0] = u0.x; v[1] = u0.y; v[2] = u0.z; v[3] = u0.w;
                v[4] = u1.x; v[5] = u1.y; v[6] = u1.z; v[7] = u1.w;
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int c = c0 + j;
                    float y = 0.f;
                    if (ok) {
                        if (c < D) y = __ldg(f + c);
                        else if (c == D) y = x.dx;
                        else if (c == D + 1) y = x.dy;
                        else if (c == D + 2) y = x.dz;
                    }
                    v[j] = y;
                }
            }
            st_chunk(dst(c8), v);
        }
    } else {
        const int D1 = p.d1, D2 = p.d2;
        const float *r0 = x.r0, *r1 = x.r1, *r2 = x.r2, *f1 = x.f1;
        const float w0 = x.w0, w1 = x.w1, w2 = x.w2;
        const bool single = p.fp_m == 1;
        const bool vec = ok && (D2 % 4 == 0) && p.feat_aligned;
        const float2 ww0 = make_float2(w0, w0), ww1 = make_float2(w1, w1), ww2 = make_float2(w2, w2);
        int c8 = c8_from;
        if (vec && !single) {
            // 2 chunks (16 channels) of the three neighbour rows: 12 x LDG.128 in flight per thread
            for (; c8 + 2 <= c8_end && (c8 + 2) * 8 <= D2; c8 += 2) {
                float4 a0[4], a1[4], a2[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    a0[q] = __ldg(reinterpret_cast<const float4 *>(r0 + c8 * 8 + 4 * q));
                    a1[q] = __ldg(reinterpret_cast<const float4 *>(r1 + c8 * 8 + 4 * q));
                    a2[q] = __ldg(reinterpret_cast<const float4 *>(r2 + c8 * 8 + 4 * q));
                }
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    float v[8];
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        // packed f32x2: per-lane IEEE results identical to the scalar rn sequence
                        const float4 x0 = a0[2 * h + q], x1 = a1[2 * h + q], x2 = a2[2 * h + q];
                        const float2 lo = __ffma2_rn(ww2, make_float2(x2.x, x2.y),
                                                     __ffma2_rn(ww0, make_float2(x0.x, x0.y), __fmul2_rn(ww1, make_float2(x1.x, x1.y))));
                        const float2 hi = __ffma2_rn(ww2, make_float2(x2.z, x2.w),
                                                     __ffma2_rn(ww0, make_float2(x0.z, x0.w), __fmul2_rn(ww1, make_float2(x1.z, x1.w))));
                        v[4 * q + 0] = lo.x; v[4 * q + 1] = lo.y; v[4 * q + 2] = hi.x; v[4 * q + 3] = hi.y;
                    }
                    st_chunk(dst(c8 + h), v);
                }
            }
        }
        for (; c8 < c8_end; ++c8) {
            float v[8];
            const int c0 = c8 * 8;
            if (vec && c0 + 8 <= D2) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const float4 a0 = __ldg(reinterpret_cast<const float4 *>(r0 + c0 + 4 * h));
                    if (single) {
                        v[4 * h] = a0.x; v[4 * h + 1] = a0.y; v[4 * h + 2] = a0.z; v[4 * h + 3] = a0.w;
                    } else {
                        const float4 a1 = __ldg(reinterpret_cast<const float4 *>(r1 + c0 + 4 * h));
                        const float4 a2 = __ldg(reinterpret_cast<const float4 *>(r2 + c0 + 4 * h));
                        v[4 * h + 0] = __fmaf_rn(w2, a2.x, __fmaf_rn(w0, a0.x, __fmul_rn(w1, a1.x)));
                        v[4 * h + 1] = __fmaf_rn(w2, a2.y, __fmaf_rn(w0, a0.y, __fmul_rn(w1, a1.y)));
                        v[4 * h + 2] = __fmaf_rn(w2, a2.z, __fmaf_rn(w0, a0.z, __fmul_rn(w1, a1.z)));
                        v[4 * h + 3] = __fmaf_rn(w2, a2.w, __fmaf_rn(w0, a0.w, __fmul_rn(w1, a1.w)));
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int c = c0 + j;
                    float y = 0.f;
                    if (ok) {
                        if (c < D2)
                            y = single ? __ldg(r0 + c)
                                       : __fmaf_rn(w2, __ldg(r2 + c), __fmaf_rn(w0, __ldg(r0 + c), __fmul_rn(w1, __ldg(r1 + c))));
                        else if (c < D2 + D1)
                            y = __ldg(f1 + (c - D2));
                    }
                    v[j] = y;
                }
            }
            st_chunk(dst(c8), v);
        }
    }
}

// Warp-cooperative gather of bf16 feature rows: the warp's 32 rows x nc 16-byte chunks are walked as one flat list,
// 32 items per step, so consecutive lanes read consecutive 16 bytes of the SAME source row (a 256-byte row is 2 L1
// wavefronts instead of 16 scattered ones -- the per-thread-row gather is L1-wavefront bound).  A lane gets the source
// row (and the interpolation weights) of the row it serves from that row's owner lane with shuffles.  U steps are
// batched so U (SA: copy) or 3U (FP: three neighbours) 128-bit loads are in flight per lane.
template <int U, int kMode>
__device__ __forceinline__ void coop_gather_bf16(const TcParams &p, const RowPre &pre, unsigned char *a, int warp, int lane,
                                                 int c8_begin, int c8_from, int c8_to) {
    const bool sa = (kMode == MODE_SA);
    // rows are addressed in 16-byte units with 32-bit row index x 32-bit pitch (one IMAD.WIDE.U32 per row pointer)
    const uint4 *base = reinterpret_cast<const uint4 *>(sa ? (const void *)p.feat : (const void *)p.feat2);
    const uint32_t pitch = (uint32_t)(sa ? p.d : p.d2) >> 3;
    const bool fp3 = !sa && p.fp_m != 1;
    const int nc = c8_to - c8_from;  // power of two, >= 4
    const int lg = 31 - __clz(nc);
    // rows past the end of the launch carry index 0 and weight 0 (row_prefetch): they read a valid row and produce finite
    // operand rows whose results are never stored, so the loads need no predicate and the registers no clearing
    const int my0 = pre.i0, my1 = pre.i1, my2 = pre.i2;
    for (int base_item = 0; base_item < 32 * nc; base_item += 32 * U) {
        // phase 1: every load of the batch is issued before the first use (3U x 128 bit in flight per lane for FP)
        uint4 q0[U], q1[U], q2[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int item = base_item + 32 * u + lane;
            const int rw = item >> lg;
            // 16-byte units, 32-bit unit index (launch_tc bounds rows x pitch): one IMAD + one wide IMAD per address
            const uint32_t col = (uint32_t)((item & (nc - 1)) + c8_from);
            const uint32_t s0 = (uint32_t)__shfl_sync(0xffffffffu, my0, rw);
            q0[u] = __ldg(base + (s0 * pitch + col));
            if (fp3) {
                const uint32_t s1 = (uint32_t)__shfl_sync(0xffffffffu, my1, rw);
                const uint32_t s2 = (uint32_t)__shfl_sync(0xffffffffu, my2, rw);
                q1[u] = __ldg(base + (s1 * pitch + col));
                q2[u] = __ldg(base + (s2 * pitch + col));
            }
        }
        // phase 2: the weights of the served row arrive by shuffle only now, so they are not live across the loads
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int item = base_item + 32 * u + lane;
            const int rw = item >> lg, ch = item & (nc - 1);
            uint4 o = q0[u];
            if (fp3) {
                const float w0 = __shfl_sync(0xffffffffu, pre.a, rw);
                const float w1 = __shfl_sync(0xffffffffu, pre.b, rw);
                const float w2 = __shfl_sync(0xffffffffu, pre.c, rw);
                const uint32_t *u0 = reinterpret_cast<const uint32_t *>(&q0[u]);
                const uint32_t *u1 = reinterpret_cast<const uint32_t *>(&q1[u]);
                const uint32_t *u2 = reinterpret_cast<const uint32_t *>(&q2[u]);
                uint32_t *uo = reinterpret_cast<uint32_t *>(&o);
                const float2 ww0 = make_float2(w0, w0), ww1 = make_float2(w1, w1), ww2 = make_float2(w2, w2);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    // bf16 -> fp32 is a 16-bit shift; packed f32x2 = the scalar rn sequence of three_interpolate per lane
                    const float2 a0 = make_float2(__uint_as_float(u0[e] << 16), __uint_as_float(u0[e] & 0xffff0000u));
                    const float2 a1 = make_float2(__uint_as_float(u1[e] << 16), __uint_as_float(u1[e] & 0xffff0000u));
                    const float2 a2 = make_float2(__uint_as_float(u2[e] << 16), __uint_as_float(u2[e] & 0xffff0000u));
                    const float2 y = __ffma2_rn(ww2, a2, __ffma2_rn(ww0, a0, __fmul2_rn(ww1, a1)));
                    uo[e] = pack_bf16(y.x, y.y);
                }
            }
            *reinterpret_cast<uint4 *>(a + swz_chunk(warp * 32 + rw, c8_from + ch - c8_begin, TC_ROWS)) = o;
        }
    }
}

// Two instantiations (kernels below): fp32 gathered features (lean: 80 registers, 4 CTAs/SM) and bf16 gathered features
// (96 registers, 3 CTAs/SM).
template <bool kInBf16, int NWW, int kMode>
__device__ __forceinline__ void row_mlp_tc_body(const TcParams &p) {
    // NWW worker warps: warp w serves TMEM lane quarter (w & 3), i.e. tile rows 32 (w & 3) .. +31; with NWW == 8 the warps
    // w and w + 4 share a quarter and split its work by columns (half = w >> 2): the gather of a tile has twice the loads
    // in flight and every epilogue is half as long -- the per-tile latency chain, not issue slots, is what bounds the kernel.
    constexpr int NHALF = NWW / 4;
    // 1024-byte alignment for the 128B-swizzled operand tiles.  The alignment is REQUESTED on the declaration (no manual
    // round-up through an integer: that hid the address space from the compiler, which then emitted generic LD.E / ST.E
    // for every shared-memory access of the gather and the epilogues) and verified once.
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = smem_raw;
    if ((smem_u32(smem_raw) & 1023u) != 0u) __trap();
    unsigned char *a_buf = smem;
    unsigned char *w_ring = smem + p.a_bytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(w_ring + (size_t)p.stages * p.stage_bytes);
    // bars: [0..4) full, [4..8) empty, [8] a_ready, [9] acc_ready, [10] a_free, [12..16) acc_ready of the transposed last
    // layer's 128-channel blocks (one barrier per block: each completes once per tile, so the issuer can never run two
    // phases ahead of a waiting warp); then the TMEM base slot, exchange, biases
    const int S = p.stages;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * MAX_STAGES + 8);
    long long *srow = reinterpret_cast<long long *>(tmem_slot + 4);       // FP: destination row of each tile row (-1 = past the end)
    float *sbias = reinterpret_cast<float *>(srow) + 4 * 32 * 2;          // all layers' biases, zero padded to npad

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + MAX_STAGES);
    const uint32_t bar_a = smem_u32(bars + 2 * MAX_STAGES), bar_acc = smem_u32(bars + 2 * MAX_STAGES + 1);
    const uint32_t bar_afree = smem_u32(bars + 2 * MAX_STAGES + 2);
    const uint32_t bar_blk = smem_u32(bars + 2 * MAX_STAGES + 4);  // [4]

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        // one arrival per worker warp (after __syncwarp): every arrival wakes the warps parked on ANY barrier of the CTA,
        // so 128 per-thread arrivals per layer kept the producer / issuer warps spinning (3 M wake-ups per sa1 launch)
        mbar_init(bar_a, NWW);
        mbar_init(bar_acc, 1);
        mbar_init(bar_afree, 1);
        for (int q = 0; q < 4; ++q) mbar_init(bar_blk + 8 * q, 1);
        fence_mbar_init();
    }
    for (int l = 0; l < p.num_layers; ++l) {
        const TcLayer &L = p.layer[l];
        for (int c = threadIdx.x; c < L.npad; c += (NWW + 2) * 32) sbias[L.bias_off + c] = c < L.cout ? __ldg(L.bias + c) : 0.f;
    }
    if (warp == NWW + 1) tmem_alloc(smem_u32(tmem_slot), (uint32_t)p.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // Persistent: each CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ...; barriers, TMEM and biases are set
    // up once.  Several CTAs share an SM, so one CTA's gather / epilogue overlaps another's MMAs.
    if (warp == NWW) {
        // ===== weight producer: every tile of every layer, in MMA order, through the ring =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (long long tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
                for (int l = 0; l < p.num_layers; ++l) {
                    const TcLayer &L = p.layer[l];
                    const int nkb = L.nkb;
                    const bool tr = (kMode == MODE_SA) && l == p.num_layers - 1;
                    // normal layers: one [nblk x 64] tile per stage.  Transposed last layer: a 128-row block of W (the
                    // M operand) per stage, assembled from the same packed tiles.
                    const int nnb = tr ? (L.npad + 127) / 128 : L.nnb;
                    const uint32_t tile_bytes = (uint32_t)L.nblk * 128u;
                    const unsigned char *src = p.packed + L.w_off;
                    const int kch = l == 0 ? p.kchunk : nkb;  // same (chunk, n-block, k-block) order as the MMA issuer
                    const int nfull = (l == 0) ? nkb - p.thin : nkb;
                    for (int k0 = 0; k0 < nfull; k0 += kch)
                        for (int nb = 0; nb < nnb; ++nb)
                            for (int kb = k0; kb < (k0 + kch >= nfull ? nkb : k0 + kch); ++kb) {
                                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                                const uint32_t dst = smem_u32(w_ring + (size_t)stage * p.stage_bytes);
                                if (!tr) {
                                    mbar_expect_tx(bar_full + 8 * stage, tile_bytes);
                                    bulk_g2s(dst, src + (size_t)(nb * nkb + kb) * tile_bytes, tile_bytes, bar_full + 8 * stage);
                                } else if (p.pool_dup > 1) {
                                    // the whole layer is one tile of npad <= 64 rows: pool_dup copies fill the 128 rows
                                    mbar_expect_tx(bar_full + 8 * stage, 128u * 128u);
                                    for (int q = 0; q < p.pool_dup; ++q)
                                        bulk_g2s(dst + (uint32_t)q * tile_bytes, src + (size_t)kb * tile_bytes, tile_bytes, bar_full + 8 * stage);
                                } else {
                                    const int row0 = nb * 128, rows = min(128, L.npad - row0);
                                    mbar_expect_tx(bar_full + 8 * stage, (uint32_t)rows * 128u);
                                    if (L.nblk >= 128) {
                                        const int t = row0 / L.nblk, off = row0 % L.nblk;
                                        bulk_g2s(dst, src + (size_t)(t * nkb + kb) * tile_bytes + (size_t)off * 128, (uint32_t)rows * 128u,
                                                 bar_full + 8 * stage);
                                    } else {
                                        for (int q = 0; q * L.nblk < rows; ++q)
                                            bulk_g2s(dst + (uint32_t)q * tile_bytes, src + (size_t)((row0 / L.nblk + q) * nkb + kb) * tile_bytes,
                                                     tile_bytes, bar_full + 8 * stage);
                                    }
                                }
                                if (++stage == S) {
                                    stage = 0;
                                    phase ^= 1;
                                }
                            }
                }
            }
        }
    } else if (warp == NWW + 1) {
        // ===== MMA issuer: all 32 lanes walk the schedule (uniform control flow), one elected lane issues =====
        {
            const uint32_t leader = elect_one();
            int stage = 0;
            uint32_t phase = 0, it = 0;
            const uint32_t a_lo0 = desc_lo(smem_u32(a_buf));
            const uint32_t w_lo0 = desc_lo(smem_u32(w_ring));
            // thin region: un-swizzled K-major, LBO (K step between core matrices) 128 B, SBO (8-row groups) 256 B
            const uint32_t thin_lo = (((smem_u32(a_buf) + (uint32_t)p.a_bytes - 4096u) & 0x3FFFFu) >> 4) | ((128u >> 4) << 16);
            const uint32_t stage_step = (uint32_t)p.stage_bytes >> 4;
            const uint32_t tmem_d = __shfl_sync(0xffffffffu, tmem_base, 0);
            long long *dbgm = (p.dbg && blockIdx.x == 0 && lane == 0) ? p.dbg + 256 : nullptr;  // operand seen / MMAs issued
            int dm = 0;
            for (long long tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
                for (int l = 0; l < p.num_layers; ++l) {
                    const bool tr = (kMode == MODE_SA) && l == p.num_layers - 1;  // D^T = W * A^T: W is the M operand, 128 samples are N
                    const int kpad = p.layer[l].kpad, nblk = tr ? 128 : p.layer[l].nblk;
                    const int nkb = p.layer[l].nkb;
                    const int nnb = tr ? (p.layer[l].npad + 127) / 128 : p.layer[l].nnb;
                    const uint32_t idesc = umma_idesc(nblk);
                    const int kch = l == 0 ? p.kchunk : nkb;
                    const int thin_kb = (l == 0 && p.thin) ? nkb - 1 : -1;  // the thin k-block rides with the last pass
                    const int nfull = nkb - (thin_kb >= 0);
                    for (int k0 = 0; k0 < nfull; k0 += kch, ++it) {
                        mbar_wait(bar_a, it & 1);  // this chunk of the operand is in shared memory
                        tc_fence_after();
                        if (dbgm && dm < 120) dbgm[dm++] = clock64();
                        long long wsum = 0;
                        const int k1 = (k0 + kch >= nfull) ? nkb : k0 + kch;
                        const bool per_block = tr && nfull <= kch;  // single pass: hand over each 128-channel block as it completes
                        for (int nb = 0; nb < nnb; ++nb) {
                            const uint32_t d = tmem_d + (uint32_t)(nb * nblk);
                            uint32_t a_lo = a_lo0;
                            for (int kb = k0; kb < k1; ++kb, a_lo += A_BLOCK_BYTES >> 4) {
                                const long long w0 = dbgm ? clock64() : 0;
                                mbar_wait(bar_full + 8 * stage, phase);
                                tc_fence_after();
                                if (dbgm) wsum += clock64() - w0;
                                const uint32_t w_lo = w_lo0 + (uint32_t)stage * stage_step;
                                const int k16n = min(KBLK, kpad - kb * KBLK) / 16;
                                if (tr) {
                                    // operands swapped: the weight block is the 128-row M operand
                                    if (kb == thin_kb)
                                        tc_mma_lo(d, w_lo, DESC_HI, thin_lo, DESC_HI_THIN, idesc, 1u, leader);
                                    else
                                        for (int k = 0; k < k16n; ++k)
                                            tc_mma_lo(d, w_lo + 2 * k, DESC_HI, a_lo + 2 * k, DESC_HI, idesc, (uint32_t)((kb | k) != 0), leader);
                                } else if (kb == thin_kb) {
                                    tc_mma_lo(d, thin_lo, DESC_HI_THIN, w_lo, DESC_HI, idesc, 1u, leader);  // never the first k-block
                                } else if (k16n == 4) {
                                    tc_mma_lo(d, a_lo, DESC_HI, w_lo, DESC_HI, idesc, (uint32_t)(kb != 0), leader);
                                    tc_mma_lo(d, a_lo + 2, DESC_HI, w_lo + 2, DESC_HI, idesc, 1u, leader);
                                    tc_mma_lo(d, a_lo + 4, DESC_HI, w_lo + 4, DESC_HI, idesc, 1u, leader);
                                    tc_mma_lo(d, a_lo + 6, DESC_HI, w_lo + 6, DESC_HI, idesc, 1u, leader);
                                } else {
                                    for (int k = 0; k < k16n; ++k)
                                        tc_mma_lo(d, a_lo + 2 * k, DESC_HI, w_lo + 2 * k, DESC_HI, idesc, (uint32_t)((kb | k) != 0), leader);
                                }
                                tc_commit_if(bar_empty + 8 * stage, leader);  // frees the ring slot when these MMAs retire
                                if (++stage == S) {
                                    stage = 0;
                                    phase ^= 1;
                                }
                            }
                            if (per_block) tc_commit_if(bar_blk + 8 * nb, leader);
                        }
                        // accumulators complete (last chunk) / operand buffer reusable (earlier chunks)
                        if (!per_block) tc_commit_if(k1 == nkb ? bar_acc : bar_afree, leader);
                        if (dbgm && dm < 120) {
                            dbgm[128 + dm / 2] = wsum + 1;  // cycles spent waiting for weight tiles in this chunk
                            dbgm[dm++] = clock64();
                        }
                    }
                }
            }
            __syncwarp();
        }
    } else {
        // ===== gather + epilogue warps: thread <-> row <-> TMEM lane =====
        const int r = threadIdx.x & (TC_ROWS - 1);  // tile row = TMEM lane
        const int wq = warp & 3;                     // lane quarter
        const int half = warp >> 2;                  // which share of the columns (NWW == 8)
        const uint32_t lane_base = tmem_base + ((uint32_t)(wq * 32) << 16);
        const uint32_t a_row = smem_u32(a_buf) + (uint32_t)r * 128u;  // this row of a k-block, shared-window address
        const uint32_t r7s = (uint32_t)(r & 7) << 4;                  // swizzle term of the row
        const uint32_t sbias_u32 = smem_u32(sbias);
        uint32_t it = 0;
        long long out_row = 0;
        bool srow_ok = false;
        long long *dbg = (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) ? p.dbg : nullptr;
        int di = 0;
        uint32_t afree_it = 0, tile_it = 0;
        RowPre pre = row_prefetch<kMode>(p, blockIdx.x, r);
        for (long long tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
            if (dbg && di < 240) dbg[di++] = clock64();
            {
                const RowCtx ctx = row_expand<kMode>(p, pre);
                out_row = ctx.out_row;
                srow_ok = ctx.ok;
                // FP: element offset of each tile row's destination (-1 = past the end); read after the layer barriers by
                // the same warp (odd-width store below)
                if ((kMode == MODE_FP)) srow[r] = ctx.ok ? ctx.out_row * p.layer[p.num_layers - 1].cout : -1;
                const int nkb0 = (p.layer[0].kpad + KBLK - 1) / KBLK;
                const int c8_total = p.layer[0].kpad / 8;
                // a narrow fp32 skip block (the xyz/colour rows of fp1) is fetched now, not after the first chunk's MMAs
                float sk[8];
                const bool sk_valid = kInBf16 && (kMode == MODE_FP) && !p.skip_bf16 && p.d1 <= 8 && (p.d2 & 7) == 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) sk[j] = (sk_valid && ctx.ok && j < p.d1) ? __ldg(ctx.f1 + j) : 0.f;
                const int nfull0 = nkb0 - p.thin;  // whole 64-column k-blocks; a thin last block rides with the last pass
                ADst dst;
                dst.a = a_buf;
                dst.r = r;
                dst.thin_c8 = p.thin ? nfull0 * 8 : (1 << 30);
                dst.thin_off = (uint32_t)p.a_bytes - 4096u;
                for (int k0 = 0; k0 < nfull0; k0 += p.kchunk) {
                    if (k0 > 0) {
                        mbar_wait(bar_afree, afree_it & 1);  // the MMAs of the previous chunk have consumed the buffer
                        ++afree_it;
                    }
                    const int cb = k0 * 8;
                    const int ce = (k0 + p.kchunk >= nfull0) ? c8_total : (k0 + p.kchunk) * 8;
                    dst.c8_begin = cb;
                    int from = cb;
                    if constexpr (kInBf16) {
                        // bf16 feature block: coalesced warp-cooperative gather when its chunk count in this pass is a
                        // power of two (>= 4) and the block ends on a k-block boundary; the tail stays one thread per row
                        const int Dm = (kMode == MODE_SA) ? p.d : p.d2;
                        const int blk0_end = min(ce, Dm >> 3);
                        const int nc = blk0_end - cb;
                        if ((Dm & 63) == 0 && nc >= 4 && (nc & (nc - 1)) == 0) {
                            // two warps per quarter: each takes half of the chunk columns of the same 32 rows
                            const bool split = NHALF == 2 && nc >= 8;
                            const int ncw = split ? nc >> 1 : nc;
                            const int c_lo = cb + (split ? half * ncw : 0);
                            if (split || half == 0) {
                                if ((kMode == MODE_SA)) coop_gather_bf16<4, kMode>(p, pre, a_buf, wq, lane, cb, c_lo, c_lo + ncw);
                                else coop_gather_bf16<FP_GATHER_U, kMode>(p, pre, a_buf, wq, lane, cb, c_lo, c_lo + ncw);
                            }
                            from = blk0_end;
                        }
                    }
                    if (from < ce) {
                        // thread-per-row part (fp32 features, tails): the two warps of a quarter take a chunk range each
                        int t_lo = from, t_hi = ce;
                        if (NHALF == 2) {
                            const int mid = from + (((ce - from + 1) >> 1) + 3 & ~3);  // multiples of 4 chunks keep the 128-bit paths
                            if (half == 0) t_hi = mid < ce ? mid : ce;
                            else t_lo = mid < ce ? mid : ce;
                        }
                        if (t_lo < t_hi) gather_tail_tc<kInBf16, kMode>(p, ctx, dst, t_lo, t_hi, sk, sk_valid);
                    }
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_a);
                }
            }
            pre = row_prefetch<kMode>(p, tile + gridDim.x, r);  // next tile's index-level loads fly while this tile's layers run
            if (dbg && di < 240) dbg[di++] = clock64();
            for (int l = 0; l < p.num_layers; ++l) {
                const TcLayer &L = p.layer[l];
                const bool last = (l == p.num_layers - 1);
                const int npad = L.npad, cout = L.cout, relu = L.relu;
                const float *bl = sbias + L.bias_off;
                // the transposed last layer hands its accumulators over per 128-channel block (when it is one pass)
                bool per_block = false;
                if (last && (kMode == MODE_SA)) {
                    const int nkb = (L.kpad + KBLK - 1) / KBLK;
                    per_block = (l == 0 ? nkb - p.thin : nkb) <= (l == 0 ? p.kchunk : nkb);
                }
                if (!per_block) {
                    mbar_wait(bar_acc, it & 1);
                    ++it;
                    tc_fence_after();
                }
                if (dbg && di < 240) dbg[di++] = clock64();
                if (last && (kMode == MODE_SA)) {
                    // Transposed last layer of an SA block: TMEM lane = output channel, column = sample, so the max over
                    // the nsample rows of a group is a register-local tree (no shuffles / CREDUX), bias and ReLU are
                    // applied once per group (max(x)+b == max(x+b) in fp32: rounding is monotone), and the 32 lanes of a
                    // warp store 32 consecutive channels.
                    const int K = p.k;
                    const int lgK = 31 - __clz(K);  // nsample is a power of two
                    const long long g_tile = tile << (7 - lgK);  // first group of this tile (128 / K groups per tile)
                    const int ncb = (npad + 127) / 128;
                    for (int cb = 0; cb < ncb; ++cb) {
                        if (per_block) {
                            mbar_wait(bar_blk + 8 * cb, tile_it & 1);
                            tc_fence_after();
                        }
                        int ch0 = cb * 128 + wq * 32;
                        int s_lo = 0, s_hi = TC_ROWS;
                        if (p.pool_dup > 1) {
                            // lanes 32 wq .. +31 hold channel quarter (wq mod nq) again: this warp pools sample part wq / nq
                            const int nq = npad >> 5;  // 1 or 2
                            ch0 = (wq & (nq - 1)) * 32;
                            s_lo = (wq >> (nq - 1)) * (32 * nq);
                            s_hi = s_lo + 32 * nq;
                        }
                        if (ch0 >= cout) continue;  // warp-uniform: e.g. 64 un-duplicated channels keep two warps busy
                        // two warps per quarter: samples [0, 64) and [64, 128) (whole groups while nsample <= 64)
                        const bool tsplit = NHALF == 2 && K <= 64;
                        if (!tsplit && half != 0) continue;
                        if (tsplit) {
                            s_lo = half * 64;
                            s_hi = s_lo + 64;
                        }
                        const int ch = ch0 + lane;
                        const float bias = bl[ch];
                        float run = 0.f;
                        for (int s0 = s_lo; s0 < s_hi; s0 += 32) {
                            uint32_t acc[32];
                            tmem_ld32(lane_base + (uint32_t)(cb * 128 + s0), acc);
                            float v[32];
#pragma unroll
                            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
#pragma unroll
                            for (int o = 1; o < 32; o <<= 1) {
                                if (o < K) {
#pragma unroll
                                    for (int j = 0; j < 32; j += 2 * o) v[j] = fmaxf(v[j], v[j + o]);
                                }
                            }
                            if (K >= 32) {
                                run = (s0 & (K - 1)) == 0 ? v[0] : fmaxf(run, v[0]);
                                if (((s0 + 32) & (K - 1)) == 0) {
                                    const long long g = g_tile + (((s0 + 32) >> lgK) - 1);
                                    if (g < p.groups && ch < cout) {
                                        const float y = relu ? fmaxf(run + bias, 0.f) : run + bias;
                                        const size_t o = (size_t)g * p.out_stride + p.out_offset + ch;
                                        if (p.out_bf16) reinterpret_cast<__nv_bfloat16 *>(p.out)[o] = __float2bfloat16_rn(y);
                                        else p.out[o] = y;
                                    }
                                }
                            } else {
#pragma unroll
                                for (int j = 0; j < 32; ++j) {
                                    if ((j & (K - 1)) == 0) {
                                        const long long g = g_tile + ((s0 + j) >> lgK);
                                        if (g < p.groups && ch < cout) {
                                            const float y = relu ? fmaxf(v[j] + bias, 0.f) : v[j] + bias;
                                            const size_t o = (size_t)g * p.out_stride + p.out_offset + ch;
                                            if (p.out_bf16) reinterpret_cast<__nv_bfloat16 *>(p.out)[o] = __float2bfloat16_rn(y);
                                            else p.out[o] = y;
                                        }
                                    }
                                }
                            }
                        }
                    }
                } else {
                float am_best = 0.f;  // running arg-max over the channels of this thread's row (PN2_FLAG_OUT_ARGMAX)
                int am_idx = -1;
                // two warps per quarter alternate 32-column chunks; outputs that need the whole row in one thread (arg-max)
                // or the warp-private staging (odd row pitch) stay with the first warp
                const bool csplit = NHALF == 2 && (!last || (!p.out_argmax && ((cout * (p.out_bf16 ? 2 : 4)) & 15) == 0));
                if (!last) {
                    // hidden layer: bias (packed f32x2), ReLU folded into the bf16x2 conversion, 128-bit stores of the next
                    // layer's operand, in 16-column pieces with the TMEM load of the next piece in flight.  Addresses are
                    // 32-bit shared-window values: row base + k-block + the swizzled 16-byte slot, where
                    // slot(c) = (c << 4) ^ ((r & 7) << 4) and c = (column / 8) mod 8.
                    if ((csplit || half == 0) && (kMode == MODE_SA || npad < 128)) {
                        // SA builds and narrow layers: one x32 load per chunk.  (The split loads below pay in the FP builds --
                        // fp1+head 107 -> 103 us, fp4 35 -> 33, fp2 27 -> 25 -- and cost in the SA builds: sa1 71.7 -> 74.6 us,
                        // sa2 35.3 -> 37.4, sa4 21 -> 23, also with this branch in place, so they are compiled out there.)
                        for (int c0 = csplit ? 32 * half : 0; c0 < npad; c0 += csplit ? 64 : 32) {
                            uint32_t acc[32];
                            tmem_ld32(lane_base + (uint32_t)c0, acc);
                            const uint32_t dst0 = a_row + (uint32_t)(c0 >> 6) * A_BLOCK_BYTES;
                            const uint32_t x0 = ((uint32_t)((c0 >> 3) & 4) << 4) ^ r7s;
                            const uint32_t bsrc = sbias_u32 + (uint32_t)(L.bias_off + c0) * 4u;
                            if (relu) epilogue_chunk<true>(acc, bsrc, dst0, x0);
                            else epilogue_chunk<false>(acc, bsrc, dst0, x0);
                        }
                    } else if (kMode != MODE_SA && (csplit || half == 0)) {
                        const int step = csplit ? 64 : 32;
                        int c0 = csplit ? 32 * half : 0;
                        uint32_t pa[16], pb[16];
                        if (c0 < npad) tmem_ld16_issue(lane_base + (uint32_t)c0, pa);
                        for (; c0 < npad; c0 += step) {
                            const uint32_t dst0 = a_row + (uint32_t)(c0 >> 6) * A_BLOCK_BYTES;
                            const uint32_t xa = ((uint32_t)((c0 >> 3) & 4) << 4) ^ r7s, xb = xa ^ 0x20u;
                            const uint32_t bsrc = sbias_u32 + (uint32_t)(L.bias_off + c0) * 4u;
                            tmem_ld16_wait(pa);
                            tmem_ld16_issue(lane_base + (uint32_t)(c0 + 16), pb);
                            if (relu) epilogue_piece<true>(pa, bsrc, dst0, xa);
                            else epilogue_piece<false>(pa, bsrc, dst0, xa);
                            tmem_ld16_wait(pb);
                            if (c0 + step < npad) tmem_ld16_issue(lane_base + (uint32_t)(c0 + step), pa);
                            if (relu) epilogue_piece<true>(pb, bsrc + 64u, dst0, xb);
                            else epilogue_piece<false>(pb, bsrc + 64u, dst0, xb);
                        }
                    }
                } else
                if (csplit || half == 0)
                for (int c0 = csplit ? 32 * half : 0; c0 < npad; c0 += csplit ? 64 : 32) {
                    uint32_t acc[32];
                    tmem_ld32(lane_base + (uint32_t)c0, acc);
                    float v[32];
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const float4 bv = *reinterpret_cast<const float4 *>(bl + c0 + 4 * q);
                        v[4 * q + 0] = __uint_as_float(acc[4 * q + 0]) + bv.x;
                        v[4 * q + 1] = __uint_as_float(acc[4 * q + 1]) + bv.y;
                        v[4 * q + 2] = __uint_as_float(acc[4 * q + 2]) + bv.z;
                        v[4 * q + 3] = __uint_as_float(acc[4 * q + 3]) + bv.w;
                    }
                    if (relu) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
                    }
                    {
                        // FP: rows are independent
                        const int esz = p.out_bf16 ? 2 : 4;
                        if (p.out_argmax) {
                            // class prediction: the thread holds every logit of its row, so the arg-max costs two
                            // instructions per channel and the row leaves as one byte (np.argmax order: first maximum)
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                if (c0 + j < cout && (am_idx < 0 || v[j] > am_best)) {
                                    am_best = v[j];
                                    am_idx = c0 + j;
                                }
                            }
                            if (c0 + 32 >= npad && srow_ok) reinterpret_cast<unsigned char *>(p.out)[out_row] = (unsigned char)am_idx;
                        } else if (((cout * esz) & 15) == 0) {
                            // rows start 16-byte aligned: the thread's 32 consecutive columns go out as 128-bit stores
                            if (srow_ok) {
                                if (p.out_bf16) {
                                    uint4 *dst = reinterpret_cast<uint4 *>(reinterpret_cast<__nv_bfloat16 *>(p.out) + (size_t)out_row * cout + c0);
#pragma unroll
                                    for (int q = 0; q < 4; ++q)
                                        if (c0 + 8 * q < cout) {
                                            uint4 o;
                                            o.x = pack_bf16(v[8 * q + 0], v[8 * q + 1]);
                                            o.y = pack_bf16(v[8 * q + 2], v[8 * q + 3]);
                                            o.z = pack_bf16(v[8 * q + 4], v[8 * q + 5]);
                                            o.w = pack_bf16(v[8 * q + 6], v[8 * q + 7]);
                                            dst[q] = o;
                                        }
                                } else {
                                    float4 *dst = reinterpret_cast<float4 *>(p.out + (size_t)out_row * cout + c0);
#pragma unroll
                                    for (int q = 0; q < 8; ++q)
                                        if (c0 + 4 * q < cout) dst[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                                }
                            }
                        } else {
                            // odd widths (the 21-class head): transpose through the (now idle) A buffer, one row per store
                            float *stg = reinterpret_cast<float *>(a_buf) + wq * (32 * 33);
#pragma unroll
                            for (int j = 0; j < 32; ++j) stg[lane * 33 + j] = v[j];
                            __syncwarp();
                            const int col = c0 + lane;
                            if (col < cout) {
                                // lane <-> column: a row leaves as one contiguous run of `cout` elements.  The per-row
                                // destination offsets were multiplied out when the tile started.
                                const long long *so = srow + wq * 32;
                                const float *sv = stg + lane;
                                if (p.out_bf16) {
                                    __nv_bfloat16 *oc = reinterpret_cast<__nv_bfloat16 *>(p.out) + col;
#pragma unroll 8
                                    for (int rr = 0; rr < 32; ++rr) {
                                        const long long off = so[rr];
                                        if (off >= 0) oc[off] = __float2bfloat16_rn(sv[rr * 33]);
                                    }
                                } else {
                                    float *oc = p.out + col;
#pragma unroll 8
                                    for (int rr = 0; rr < 32; ++rr) {
                                        const long long off = so[rr];
                                        if (off >= 0) oc[off] = sv[rr * 33];
                                    }
                                }
                            }
                            __syncwarp();
                        }
                    }
                }
                }
                if (!last) {
                    tc_fence_before();    // TMEM reads done before the next layer's MMAs overwrite the accumulators
                    fence_proxy_async();  // bf16 activations visible to the tensor core (async proxy)
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_a);
                }
                if (dbg && di < 240) dbg[di++] = clock64();
            }
            ++tile_it;
            // the FP store staging aliases other warps' rows of A: all four warps leave the tile together
            tc_fence_before();
            asm volatile("bar.sync 2, %0;" ::"n"(NWW * 32) : "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NWW + 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// Entry points.  fp32 features: 80 registers, 4 CTAs/SM.  bf16 features: 96 registers (a few spilled words) is what
// 3 CTAs x 6 warps allow -- the 18 warps spread 5/5/4/4 over the four 16 K-register partitions (__maxnreg__(112) removes
// the spills and drops to 2 CTAs/SM: fp1+head 120 -> 164 us); blocks that shared memory or TMEM limit to <= 2 CTAs/SM
// anyway use the un-spilled build.
#define PN2_TC_KERNEL(name, threads, ctas, bf16, nww)                                                                       \
    __global__ void __launch_bounds__(threads, ctas) name##_sa(const __grid_constant__ TcParams p) { row_mlp_tc_body<bf16, nww, MODE_SA>(p); } \
    __global__ void __launch_bounds__(threads, ctas) name##_fp(const __grid_constant__ TcParams p) { row_mlp_tc_body<bf16, nww, MODE_FP>(p); }
// One build per block kind (SA / FP): the mode is a compile-time constant in the gather and the epilogues.
PN2_TC_KERNEL(row_mlp_tc_kernel_f32, TC_THREADS, 4, false, 4)
PN2_TC_KERNEL(row_mlp_tc_kernel_bf16, TC_THREADS, 3, true, 4)
PN2_TC_KERNEL(row_mlp_tc_kernel_bf16_wide, TC_THREADS, 2, true, 4)
__global__ void __launch_bounds__(TC_THREADS, 4) row_mlp_tc_kernel_bf16_x4_sa(const __grid_constant__ TcParams p) { row_mlp_tc_body<true, 4, MODE_SA>(p); }
// Eight worker warps per 128-row tile, at most two CTAs per SM (102 registers): half the per-tile latency chain.
PN2_TC_KERNEL(row_mlp_tc_kernel_f32_w8, TC_THREADS_W8, 2, false, 8)
PN2_TC_KERNEL(row_mlp_tc_kernel_bf16_w8, TC_THREADS_W8, 2, true, 8)

// ---- weight packing -----------------------------------------------------------------------------------
// Packed image of one layer: for nb in n-blocks, for kb in k-blocks: a [nblk rows x 64 bf16] tile, row n at n*128 B,
// its 16-byte chunk c stored at position c ^ (n & 7) (128B swizzle), zero padded.  `perm_split` > 0 rotates the
// source columns of layer 0 so that operand column k reads W[:, (k + perm_split) mod cin] for k < cin
// (the gather writes [big block | small block]).
__global__ void pack_layer_kernel(const float *__restrict__ w, int cin, int cout, int kpad, int npad, int nblk,
                                  int perm_split, __nv_bfloat16 *__restrict__ dst) {
    const int nkb = (kpad + KBLK - 1) / KBLK;
    const long long total = (long long)npad * nkb * KBLK;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int k_in = (int)(e % KBLK);
        const long long t = e / KBLK;
        const int n_in = (int)(t % nblk);
        const long long tt = t / nblk;
        const int kb = (int)(tt % nkb), nb = (int)(tt / nkb);
        const int n = nb * nblk + n_in, k = kb * KBLK + k_in;
        float v = 0.f;
        if (n < cout && k < cin) {
            const int src = perm_split > 0 ? (k + perm_split) % cin : k;
            v = w[(size_t)n * cin + src];
        }
        const size_t tile_off = ((size_t)nb * nkb + kb) * (size_t)nblk * KBLK;
        const int c = k_in >> 3;
        const size_t off = tile_off + (size_t)n_in * KBLK + (size_t)((c ^ (n_in & 7)) << 3) + (k_in & 7);
        dst[off] = __float2bfloat16_rn(v);
    }
}

struct Plan {
    TcLayer layer[PN2_MAX_LAYERS];
    int num_layers;
    long long packed_bytes;
    int a_bytes, stage_bytes, stages, tmem_cols, bias_floats, kchunk, thin;
    size_t smem_bytes;
    bool fits;
};

constexpr size_t TC_SMEM_LIMIT = 227 * 1024;
constexpr int TC_TAIL_BYTES = (2 * MAX_STAGES + 8) * 8 + 16 + 4 * 32 * 8;  // barriers, TMEM slot, row table (+ biases)

Plan make_plan_capped(const pn2_mlp *mlp, int nblk_cap) {
    Plan P = {};
    P.num_layers = mlp->num_layers;
    long long off = 0;
    int amax = 0, smax = 0, nmax = 32, boff = 0;
    for (int l = 0; l < mlp->num_layers; ++l) {
        TcLayer &L = P.layer[l];
        L.cin = mlp->cin[l];
        L.cout = mlp->cout[l];
        L.kpad = (L.cin + 15) / 16 * 16;
        L.npad = (L.cout + 31) / 32 * 32;
        L.nblk = L.npad < nblk_cap ? L.npad : nblk_cap;
        if (L.npad % L.nblk) L.npad = (L.npad + L.nblk - 1) / L.nblk * L.nblk;
        L.relu = mlp->relu[l];
        L.bias = mlp->bias[l];
        L.w_off = off;
        L.bias_off = boff;
        boff += L.npad;
        const int nkb = (L.kpad + KBLK - 1) / KBLK;
        L.nkb = nkb;
        L.nnb = L.npad / L.nblk;
        off += (long long)L.npad * nkb * 128;
        if (l > 0) amax = amax > nkb ? amax : nkb;                        // operand of this layer (layer 0 is chunked)
        if (l + 1 < mlp->num_layers) {
            const int okb = (L.npad + KBLK - 1) / KBLK;                    // its epilogue writes npad columns
            amax = amax > okb ? amax : okb;
        }
        smax = smax > L.nblk * 128 ? smax : L.nblk * 128;
        nmax = nmax > L.npad ? nmax : L.npad;
    }
    P.packed_bytes = off;
    // first-layer operand: produced in passes of `kchunk` whole k-blocks; at least 2, at most what the hidden layers
    // need anyway.  A last k-block of only 16 columns (67, 131, 134, 259 ... input channels: features + xyz / colour)
    // gets its own 4 KB un-swizzled region and rides with the last pass instead of costing one.
    {
        const int nkb0 = (P.layer[0].kpad + KBLK - 1) / KBLK;
        P.thin = (nkb0 >= 2 && P.layer[0].kpad % KBLK == 16) ? 1 : 0;
        const int nfull0 = nkb0 - P.thin;
        int kc = amax > 2 ? amax : 2;
        if (kc > nfull0) kc = nfull0;
        P.kchunk = kc;
        amax = amax > kc ? amax : kc;
    }
    P.a_bytes = amax * A_BLOCK_BYTES;
    if (P.a_bytes < 4 * 32 * 33 * 4) P.a_bytes = ((4 * 32 * 33 * 4) + 1023) / 1024 * 1024;  // FP store staging
    if (P.thin) P.a_bytes += 4096;  // thin region = the last 4 KB of the operand buffer
    P.stage_bytes = smax;
    P.tmem_cols = 32;
    while (P.tmem_cols < nmax) P.tmem_cols *= 2;
    P.bias_floats = boff;
    P.fits = false;
    // Residency first (as many CTAs per SM as TMEM and the 4-CTA register budget allow), then the deepest ring that still
    // fits: a 2-stage ring of 128-row tiles holds one 128x128 layer just like 4 stages of 64-row tiles, with half the
    // MMAs and barrier hand-offs (fp1+head 133.5 -> 127.9 us).
    const size_t fixed = 1024 + (size_t)P.a_bytes + TC_TAIL_BYTES + (size_t)boff * 4;
    int best = 0;
    int cmax = 512 / P.tmem_cols;
    if (cmax > 4) cmax = 4;
    for (int c = cmax; c >= 1 && !best; --c)
        for (int s = MAX_STAGES; s >= 2 && !best; --s)
            if ((size_t)c * (fixed + (size_t)s * P.stage_bytes + 1024) <= TC_SMEM_LIMIT + 1024) best = s;
    if (best) {
        P.stages = best;
        P.smem_bytes = fixed + (size_t)best * P.stage_bytes;
        P.fits = nmax <= 512;
    }
    return P;
}

int g_tc_max_ctas = 8;  // developer knob (pn2_debug_set_tc_max_ctas)
int g_tc_workers = 0;   // worker warps per tile: 0 = by launch size, 4, or 8 (pn2_debug_set_tc_workers)

// CTAs of this plan that shared memory and TMEM let reside on one SM.  The developer cap (g_tc_max_ctas) is applied at
// launch only: make_plan compares these counts, and the packed weight image it describes must not depend on a knob.
int ctas_per_sm(const Plan &P) {
    int per_sm = (int)((TC_SMEM_LIMIT + 1024) / (P.smem_bytes + 1024));  // + 1 KB per CTA reserved by the system
    if (per_sm > 512 / P.tmem_cols) per_sm = 512 / P.tmem_cols;
    return per_sm < 1 ? 1 : per_sm;
}

// Weight tiles of 256, 128 or 64 rows: smaller tiles shrink the ring and let more CTAs share an SM (their
// gather / MMA / epilogue phases overlap); the packed image depends on the choice, so it is a pure function of the MLP.
Plan make_plan(const pn2_mlp *mlp) {
    Plan best = make_plan_capped(mlp, 256);
    const int caps[2] = {128, 64};
    for (int i = 0; i < 2; ++i) {
        const Plan q = make_plan_capped(mlp, caps[i]);
        if (q.fits && (!best.fits || ctas_per_sm(q) > ctas_per_sm(best))) best = q;
    }
    return best;
}

// SA launches compute the last layer transposed: its weight block is the 128-row M operand (a ring stage must hold
// 16 KB) and the accumulators take 128 columns per 128 output channels.  Same packed image, different residency:
// prefer as many CTAs per SM as TMEM / registers allow, then the deepest ring.
Plan sa_plan(const Plan &P0, bool in_bf16) {
    Plan P = P0;
    if (!P.fits) return P;
    const TcLayer &L = P.layer[P.num_layers - 1];
    const int need = (L.npad + 127) / 128 * 128;
    while (P.tmem_cols < need) P.tmem_cols *= 2;
    if (P.stage_bytes < 128 * 128) P.stage_bytes = 128 * 128;
    P.fits = false;
    if (P.tmem_cols > 512) return P;
    // (no alignment slack: the dynamic shared-memory base is 1024-byte aligned by declaration, and sa2-like blocks -- 20 KB
    // operand, two 16 KB stages -- fit four CTAs per SM only without it)
    const size_t fixed = (size_t)P.a_bytes + TC_TAIL_BYTES + (size_t)P.bias_floats * 4;
    int cmax = 512 / P.tmem_cols;
    const int reg_cap = 4;  // both SA builds (fp32 and bf16 features) fit 80 registers
    if (cmax > reg_cap) cmax = reg_cap;
    for (int c = cmax; c >= 1 && !P.fits; --c)
        for (int st = MAX_STAGES; st >= 2 && !P.fits; --st)
            if ((size_t)c * (fixed + (size_t)st * P.stage_bytes + 1024) <= TC_SMEM_LIMIT + 1024) {
                P.stages = st;
                P.smem_bytes = fixed + (size_t)st * P.stage_bytes;
                P.fits = true;
            }
    return P;
}

int check_mlp_tc(const char *op, const pn2_mlp *mlp, int c0) {
    PN2_REQUIRE(mlp, "%s: null mlp", op);
    PN2_REQUIRE(mlp->num_layers >= 1 && mlp->num_layers <= PN2_MAX_LAYERS, "%s: num_layers %d outside 1..%d", op,
                mlp->num_layers, PN2_MAX_LAYERS);
    int c = c0;
    for (int l = 0; l < mlp->num_layers; ++l) {
        PN2_REQUIRE(mlp->cin[l] == c, "%s: layer %d expects cin=%d but the previous stage produces %d", op, l, mlp->cin[l], c);
        PN2_REQUIRE(mlp->cout[l] >= 1 && mlp->bias[l], "%s: layer %d is malformed", op, l);
        c = mlp->cout[l];
    }
    return PN2_OK;
}

}  // namespace
long long *take_tc_dbg();
namespace {

// What the last pn2_*_bf16 call on this thread launched (developer hook pn2_debug_last_tc_launch); name "" = nothing.
struct TcLaunchRecord {
    const char *name;
    int grid, threads;
};
thread_local TcLaunchRecord g_tc_last = {"", 0, 0};

const char *tc_build_name(void (*kernel)(TcParams)) {
    static const struct {
        void (*fn)(TcParams);
        const char *name;
    } builds[] = {
        {row_mlp_tc_kernel_f32_sa, "f32_sa"},          {row_mlp_tc_kernel_f32_fp, "f32_fp"},
        {row_mlp_tc_kernel_bf16_sa, "bf16_sa"},        {row_mlp_tc_kernel_bf16_fp, "bf16_fp"},
        {row_mlp_tc_kernel_bf16_wide_sa, "bf16_wide_sa"}, {row_mlp_tc_kernel_bf16_wide_fp, "bf16_wide_fp"},
        {row_mlp_tc_kernel_bf16_x4_sa, "bf16_x4_sa"},  {row_mlp_tc_kernel_f32_w8_sa, "f32_w8_sa"},
        {row_mlp_tc_kernel_f32_w8_fp, "f32_w8_fp"},    {row_mlp_tc_kernel_bf16_w8_sa, "bf16_w8_sa"},
        {row_mlp_tc_kernel_bf16_w8_fp, "bf16_w8_fp"},
    };
    for (const auto &b : builds)
        if (b.fn == kernel) return b.name;
    return "?";
}

int launch_tc(TcParams &p, const Plan &P, const void *packed, long long tiles, cudaStream_t s) {
    p.dbg = take_tc_dbg();
    PN2_REQUIRE(tiles * TC_ROWS <= 2147483647ll, "row_mlp_tc: more than 2^31 rows in one launch");
    if (p.mode == MODE_SA)
        PN2_REQUIRE((p.groups / p.m) * (long long)p.n <= 2147483647ll, "row_mlp_tc: more than 2^31 source points in one launch");
    else
        PN2_REQUIRE((p.rows / p.n) * (long long)p.fp_m <= 2147483647ll, "row_mlp_tc: more than 2^31 coarse points in one launch");
    PN2_REQUIRE(((uintptr_t)packed & 15) == 0, "row_mlp_tc: packed weights must be 16-byte aligned");
    p.num_layers = P.num_layers;
    for (int l = 0; l < P.num_layers; ++l) p.layer[l] = P.layer[l];
    p.packed = (const unsigned char *)packed;
    p.stages = P.stages;
    p.stage_bytes = P.stage_bytes;
    p.a_bytes = P.a_bytes;
    p.tmem_cols = P.tmem_cols;
    p.bias_floats = P.bias_floats;
    p.kchunk = P.kchunk;
    p.thin = P.thin;
    p.tiles = tiles;
    const bool sa = p.mode == MODE_SA;
    // persistent grid: as many CTAs as can be resident (shared memory, 512 TMEM columns, registers), at most one per tile
    int per_sm = ctas_per_sm(P);
    if (per_sm > g_tc_max_ctas) per_sm = g_tc_max_ctas;
    // register budget of the bf16-input builds: the SA build fits 80 registers (4 CTAs/SM: sa2 39.3 -> 35.3 us), the FP
    // build (three-row interpolating gather) needs 96 (at 80 it spills 164 bytes: fp1+head 107 -> 115 us)
    if (p.in_bf16 && per_sm > (sa ? 4 : 3)) per_sm = sa ? 4 : 3;
#define PN2_TC_PICK(name) (sa ? name##_sa : name##_fp)
    void (*kernel)(TcParams) = !p.in_bf16 ? PN2_TC_PICK(row_mlp_tc_kernel_f32)
                                          : (per_sm <= 2 ? PN2_TC_PICK(row_mlp_tc_kernel_bf16_wide)
                                                         : (per_sm >= 4 ? row_mlp_tc_kernel_bf16_x4_sa : PN2_TC_PICK(row_mlp_tc_kernel_bf16)));
    int threads = TC_THREADS;
    // small launches (a few tiles per SM at most) cannot fill the SM with tiles in flight: split each tile over 8 worker
    // warps instead (measured, batch 32: sa3 31 -> 29, sa4 27 -> 25, fp4 40 -> 37, fp3 31 -> 28, fp2 31 -> 29 us; launches
    // with many tiles per SM are faster with 3-4 resident CTAs of 4 worker warps: sa1 93 vs 133 us)
    if (g_tc_workers == 8 || (g_tc_workers == 0 && tiles <= 4ll * sm_count())) {
        if (per_sm > 2) per_sm = 2;
        kernel = p.in_bf16 ? PN2_TC_PICK(row_mlp_tc_kernel_bf16_w8) : PN2_TC_PICK(row_mlp_tc_kernel_f32_w8);
        threads = TC_THREADS_W8;
    }
    p.pool_dup = 1;
    if (p.pool_t && threads == TC_THREADS) {
        const TcLayer &L = P.layer[P.num_layers - 1];
        if (L.npad <= 64 && L.nblk == L.npad && p.k <= L.npad) p.pool_dup = 128 / L.npad;
    }
    if (p.in_bf16) {
        const long long src_rows = p.mode == MODE_SA ? (p.groups / p.m) * (long long)p.n : (p.rows / p.n) * (long long)p.fp_m;
        PN2_REQUIRE(src_rows * ((p.mode == MODE_SA ? p.d : p.d2) / 8) <= 4294967295ll, "row_mlp_tc: bf16 feature tensor exceeds 2^32 16-byte units");
    }
    PN2_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.smem_bytes));
    long long grid = (long long)per_sm * sm_count();
    if (grid > tiles) grid = tiles;
    kernel<<<(unsigned)grid, threads, P.smem_bytes, s>>>(p);
    PN2_LAUNCH_OK("row_mlp_tc_kernel");
    g_tc_last = {tc_build_name(kernel), (int)grid, threads};
    return PN2_OK;
}

}  // namespace
}  // namespace pn2

extern "C" void pn2_debug_set_tc_max_ctas(int n) { pn2::g_tc_max_ctas = n < 1 ? 1 : n; }
extern "C" void pn2_debug_set_tc_workers(int n) { pn2::g_tc_workers = (n == 8 || n == 4) ? n : 0; }
extern "C" int pn2_debug_last_tc_launch(const char **name, int *grid, int *threads) {
    const pn2::TcLaunchRecord &r = pn2::g_tc_last;
    if (name) *name = r.name;
    if (grid) *grid = r.grid;
    if (threads) *threads = r.threads;
    return r.grid > 0;
}

extern "C" int pn2_mlp_bf16_supported(const pn2_mlp *mlp) {
    if (!mlp || mlp->num_layers < 1 || mlp->num_layers > PN2_MAX_LAYERS) return 0;
    const pn2::Plan P = pn2::make_plan(mlp);  // must fit as an FP block and as an SA block (transposed last layer)
    return (P.fits && pn2::sa_plan(P, true).fits) ? 1 : 0;
}

extern "C" long long pn2_mlp_pack_bf16_size(const pn2_mlp *mlp) {
    if (!mlp || mlp->num_layers < 1 || mlp->num_layers > PN2_MAX_LAYERS) return -1;
    return pn2::make_plan(mlp).packed_bytes;
}

extern "C" int pn2_mlp_pack_bf16(const pn2_mlp *mlp, int first_layer_rotate, void *packed, void *stream) {
    using namespace pn2;
    if (int st = check_mlp_tc("mlp_pack_bf16", mlp, mlp ? mlp->cin[0] : 0)) return st;
    PN2_REQUIRE(packed, "mlp_pack_bf16: null destination");
    PN2_REQUIRE(first_layer_rotate >= 0 && first_layer_rotate < mlp->cin[0], "mlp_pack_bf16: rotate %d outside [0, cin)", first_layer_rotate);
    const Plan P = make_plan(mlp);
    for (int l = 0; l < P.num_layers; ++l) {
        const TcLayer &L = P.layer[l];
        PN2_REQUIRE(mlp->weight[l], "mlp_pack_bf16: layer %d has a null weight", l);
        const long long total = (long long)L.npad * ((L.kpad + KBLK - 1) / KBLK) * KBLK;
        const int blocks = (int)((total + 255) / 256 < 1024 ? (total + 255) / 256 : 1024);
        pack_layer_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
            mlp->weight[l], L.cin, L.cout, L.kpad, L.npad, L.nblk, l == 0 ? first_layer_rotate : 0,
            reinterpret_cast<__nv_bfloat16 *>((unsigned char *)packed + L.w_off));
        PN2_LAUNCH_OK("pack_layer_kernel");
    }
    return PN2_OK;
}

extern "C" int pn2_sa_mlp_max_bf16(int b, int n, int m, int k, int d, const float *xyz, const float *feat,
                                   const float *new_xyz, const int32_t *idx, const pn2_mlp *mlp, const void *packed,
                                   float *out, int out_stride, int out_offset, int flags, void *stream) {
    using namespace pn2;
    g_tc_last = {"", 0, 0};
    PN2_REQUIRE(b >= 0 && n >= 1 && m >= 0 && k >= 1 && d >= 0, "sa_mlp_max_bf16: bad dims b=%d n=%d m=%d k=%d d=%d", b, n, m, k, d);
    if (int st = check_mlp_tc("sa_mlp_max_bf16", mlp, 3 + d)) return st;
    if (b == 0 || m == 0) return PN2_OK;
    PN2_REQUIRE(xyz && new_xyz && idx && out && packed && (feat || d == 0), "sa_mlp_max_bf16: null pointer");
    const int cl = mlp->cout[mlp->num_layers - 1];
    PN2_REQUIRE(out_offset >= 0 && out_stride >= out_offset + cl, "sa_mlp_max_bf16: out_stride/out_offset do not hold %d channels", cl);
    if (!(k == 1 || k == 2 || k == 4 || k == 8 || k == 16 || k == 32 || k == 64 || k == 128))
        return set_error(PN2_ERR_UNSUPPORTED, "sa_mlp_max_bf16: nsample must be a power of two <= 128 (got %d)", k);
    for (int l = 0; l < mlp->num_layers; ++l)
        if (!mlp->relu[l]) return set_error(PN2_ERR_UNSUPPORTED, "sa_mlp_max_bf16: every SA layer must end in ReLU");
    const Plan P = sa_plan(make_plan(mlp), (flags & PN2_FLAG_IN_BF16) != 0);
    if (!P.fits) return set_error(PN2_ERR_UNSUPPORTED, "sa_mlp_max_bf16: channel widths exceed shared memory / TMEM; use the fp32 path");
    TcParams p = {};
    p.mode = MODE_SA;
    p.pool_t = 1;
    p.n = n; p.m = m; p.k = k; p.d = d;
    p.groups = (long long)b * m;
    p.xyz = xyz; p.feat = feat; p.new_xyz = new_xyz; p.idx = idx;
    p.out = out; p.out_stride = out_stride; p.out_offset = out_offset;
    p.feat_aligned = (((uintptr_t)feat) & 15) == 0;
    p.in_bf16 = (flags & PN2_FLAG_IN_BF16) != 0;
    p.out_bf16 = (flags & PN2_FLAG_OUT_BF16) != 0;
    if (p.in_bf16) PN2_REQUIRE(d % 8 == 0 && p.feat_aligned, "sa_mlp_max_bf16: bf16 features need d %% 8 == 0 and 16-byte alignment");
    const long long tiles = (p.groups * k + TC_ROWS - 1) / TC_ROWS;
    return launch_tc(p, P, packed, tiles, (cudaStream_t)stream);
}

extern "C" int pn2_fp_mlp_bf16(int b, int n, int m, int d1, int d2, const float *feat1, const float *feat2,
                               const int32_t *idx, const float *weight, const pn2_mlp *mlp, const void *packed,
                               const int32_t *row_perm, float *out, int flags, void *stream) {
    using namespace pn2;
    g_tc_last = {"", 0, 0};
    PN2_REQUIRE(b >= 0 && n >= 0 && m >= 1 && d1 >= 0 && d2 >= 1, "fp_mlp_bf16: bad dims b=%d n=%d m=%d d1=%d d2=%d", b, n, m, d1, d2);
    if (int st = check_mlp_tc("fp_mlp_bf16", mlp, d1 + d2)) return st;
    if (b == 0 || n == 0) return PN2_OK;
    PN2_REQUIRE(feat2 && out && packed && (feat1 || d1 == 0) && (m == 1 || (idx && weight)), "fp_mlp_bf16: null pointer");
    const Plan P = make_plan(mlp);
    if (!P.fits) return set_error(PN2_ERR_UNSUPPORTED, "fp_mlp_bf16: channel widths exceed shared memory / TMEM; use the fp32 path");
    TcParams p = {};
    p.mode = MODE_FP;
    p.n = n; p.fp_m = m; p.d1 = d1; p.d2 = d2;
    p.rows = (long long)b * n;
    p.feat1 = feat1; p.feat2 = feat2; p.idx = idx; p.weight = weight;
    p.out = out;
    p.feat_aligned = (((uintptr_t)feat2) & 15) == 0;
    p.row_perm = row_perm;
    p.in_bf16 = (flags & PN2_FLAG_IN_BF16) != 0;
    p.skip_bf16 = (flags & PN2_FLAG_SKIP_BF16) != 0;
    p.out_bf16 = (flags & PN2_FLAG_OUT_BF16) != 0;
    p.out_argmax = (flags & PN2_FLAG_OUT_ARGMAX) != 0;
    if (p.out_argmax)
        PN2_REQUIRE(!p.out_bf16 && mlp->cout[mlp->num_layers - 1] <= 256, "fp_mlp_bf16: arg-max output needs at most 256 channels and excludes PN2_FLAG_OUT_BF16");
    if (p.in_bf16) PN2_REQUIRE(d2 % 8 == 0 && p.feat_aligned, "fp_mlp_bf16: bf16 features need d2 %% 8 == 0 and 16-byte alignment");
    if (p.skip_bf16)
        PN2_REQUIRE(p.in_bf16 && d1 % 8 == 0 && (((uintptr_t)feat1) & 15) == 0, "fp_mlp_bf16: bf16 skip features need bf16 coarse features, d1 %% 8 == 0 and 16-byte alignment");
    const long long tiles = (p.rows + TC_ROWS - 1) / TC_ROWS;
    return launch_tc(p, P, packed, tiles, (cudaStream_t)stream);
}

// Developer hook: the next pn2_*_bf16 launch on this thread records phase timestamps (clock64 of CTA 0, thread 0:
// tile start, gather done, then per layer accumulator-ready / epilogue-done; from [256]: the MMA issuer's operand-seen /
// MMAs-issued stamps per operand chunk) into `buf` (>= 512 int64, device).
static thread_local long long *g_tc_dbg = nullptr;
extern "C" void pn2_debug_set_tc_timestamps(long long *buf) { g_tc_dbg = buf; }
namespace pn2 { long long *take_tc_dbg() { long long *b = g_tc_dbg; g_tc_dbg = nullptr; return b; } }
