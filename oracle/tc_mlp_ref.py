"""bf16-exact reference of one launch of the tensor-core MLP kernel (csrc/row_mlp_tc.cu) (TEST INFRASTRUCTURE ONLY).

The kernel rounds its operands to bf16 and accumulates in fp32.  Compared with the fp32 modules, that rounding alone
costs a few 1e-3 of the output scale, which hides bugs of the same size (a dropped xyz column, a wrong rounding mode).
This reference rounds to bf16 at exactly the points where the kernel does -- weights, the layer-0 operand, every hidden
activation, and the output under PN2_FLAG_OUT_BF16 -- and does everything else in float64, so a correct kernel differs
from it only by fp32-versus-fp64 accumulation: on almost every element by less than 1e-4 of the output scale.

Every bf16 conversion is round-to-nearest-even from fp32, as pack_layer_kernel (__float2bfloat16_rn), the gather
(__floats2bfloat162_rn) and the epilogue (cvt.rn.bf16x2.f32) do.  Inputs are the tensors the launch received (any
device; float64 math throughout): the folded fp32 layers [(W, b, relu), ...] of the FoldedMlp, and the geometry the
kernels produced (ball-query idx, 3-NN idx / weights).

The pieces are separate (operand, layers, output) so that tests can plant an error at one place of the reference.
"""
import torch

F64 = torch.float64


def _f32_bits(x):
    return x.to(torch.float32).contiguous().view(torch.int32)


def bf16_rn(x):
    """Round to fp32, then to bf16 (nearest, ties to even) -> float64.  Finite inputs (NaN payloads are not kept)."""
    bits = _f32_bits(x)
    lsb = torch.bitwise_and(torch.bitwise_right_shift(bits, 16), 1)
    r = torch.bitwise_and(bits + 0x7FFF + lsb, -65536)  # -65536 == 0xFFFF0000 as int32
    return r.view(torch.float32).to(F64)


def bf16_rz(x):
    """Round to fp32, then to bf16 toward zero (drop the low 16 bits) -> float64.  A deliberately wrong rounding."""
    return torch.bitwise_and(_f32_bits(x), -65536).view(torch.float32).to(F64)


def f32(x):
    """float64 value rounded to fp32, kept as float64."""
    return x.to(torch.float32).to(F64)


def fma_f32(a, b, c):
    """fp32 fused multiply-add a * b + c: the product is exact in float64, the sum is rounded once to fp32 (a double
    rounding through float64 that can differ from a true fma only on exact float64 ties)."""
    return f32(a * b + c)


def sa_operand(xyz, feat, new_xyz, idx, order, rnd=bf16_rn):
    """Layer-0 operand of an SA launch: (B, M, K, cin) float64, each entry rounded by `rnd`.

    xyz (B,N,3) fp32; feat (B,N,D) fp32 / bf16 or None; new_xyz (B,M,3) fp32; idx (B,M,K) int;
    order 0 = PN2_ORDER_XYZ_FIRST ([centred xyz | features]), 1 = PN2_ORDER_FEAT_FIRST ([features | centred xyz])."""
    B, M, K = idx.shape
    bi = torch.arange(B, device=idx.device).view(B, 1, 1)
    ii = idx.long()
    # the centring is an fp32 subtraction in the kernel (row_prefetch): exact in fp32 arithmetic here too
    c = (xyz.to(torch.float32)[bi, ii] - new_xyz.to(torch.float32)[:, :, None, :]).to(F64)
    parts = [c]
    if feat is not None and feat.shape[2] > 0:
        f = feat[bi, ii].to(F64)
        parts = [c, f] if order == 0 else [f, c]
    return rnd(torch.cat(parts, dim=-1))


def interpolate_f32(feat2, idx, weight):
    """Interpolated coarse rows of an FP launch, (B, n, D2) float64 holding fp32 values:
    f32(fma(w2, a2, f32(fma(w0, a0, f32(w1 * a1))))) with a_k the coarse rows as stored (fp32 or bf16); m >= 2."""
    B = feat2.shape[0]
    a = feat2.to(F64)
    bi = torch.arange(B, device=feat2.device).view(B, 1)
    ii = idx.long()
    w = weight.to(torch.float32).to(F64)
    a0, a1, a2 = a[bi, ii[:, :, 0]], a[bi, ii[:, :, 1]], a[bi, ii[:, :, 2]]
    w0, w1, w2 = w[:, :, 0:1], w[:, :, 1:2], w[:, :, 2:3]
    return fma_f32(w2, a2, fma_f32(w0, a0, f32(w1 * a1)))


def fp_operand(feat1, feat2, idx, weight, n, rnd=bf16_rn):
    """Layer-0 operand of an FP launch: (B, n, D1 + D2) float64 = [rnd(feat1) | rnd(interp)].
    feat1 (B,n,D1) or None; feat2 (B,m,D2); idx / weight (B,n,3) (unused when m == 1)."""
    B, m, _ = feat2.shape
    if m == 1:
        interp = feat2.to(F64).expand(B, n, feat2.shape[2])
    else:
        interp = interpolate_f32(feat2, idx, weight)
    parts = [interp] if feat1 is None or feat1.shape[2] == 0 else [feat1.to(F64), interp]
    return rnd(torch.cat(parts, dim=-1))


def weights_bf16(layers):
    """[(bf16(W), b, relu)] in float64: the weights as pn2_mlp_pack_bf16 packs them, biases fp32."""
    return [(bf16_rn(w), b.to(F64), bool(r)) for (w, b, r) in layers]


def mlp_rows(a, layers):
    """a (..., cin) float64 layer-0 operand (already rounded); layers from weights_bf16.  Every layer: z = a W^T + b in
    float64, ReLU where the layer has it; a hidden layer hands bf16(z) to the next.  -> the last layer's output."""
    x = a
    for i, (w, b, r) in enumerate(layers):
        z = torch.matmul(x, w.t()) + b
        if r:
            z = torch.clamp_min(z, 0.0)
        x = bf16_rn(z) if i + 1 < len(layers) else z
    return x


def finish(out, out_bf16=False):
    """The stored result: fp32 or, under PN2_FLAG_OUT_BF16, bf16 (both as float64)."""
    return bf16_rn(out) if out_bf16 else f32(out)


def sa_ref(xyz, feat, new_xyz, idx, order, layers, out_bf16=False):
    """pn2_sa_mlp_max_bf16: (B, M, cout) float64."""
    z = mlp_rows(sa_operand(xyz, feat, new_xyz, idx, order), weights_bf16(layers))
    return finish(z.amax(dim=2), out_bf16)


def fp_ref(feat1, feat2, idx, weight, n, layers, out_bf16=False):
    """pn2_fp_mlp_bf16: (B, n, cout) float64."""
    return finish(mlp_rows(fp_operand(feat1, feat2, idx, weight, n), weights_bf16(layers)), out_bf16)


def first_argmax(x):
    """PN2_FLAG_OUT_ARGMAX: index of the first largest channel of each row (numpy.argmax)."""
    return torch.argmax(x, dim=-1)


# Acceptance.  An element "differs" when |got - ref| > FRAC_REL * max|ref|; (a) at most FRAC_MAX of the elements may
# differ, (b) max|got - ref| <= MAX_REL * max|ref|.  What separates a correct kernel from this reference is its fp32
# accumulation: where it lands a hidden activation on the other side of a bf16 rounding boundary, the flip (one bf16 ulp)
# propagates through the later layers.  Measured on a B200 (1000 W), correct kernel (every build bit-identical): at most
# 6.2e-4 on every launch of the semseg and MSG forwards, but 3.9e-3 for a 259 -> 256, 256, 512 SA block, 3.4e-3 for a
# 1536-channel FP input and 1.9e-3 for a 5-layer head with random weights (an fp32 round-to-nearest emulation of the same
# head on the CPU already gives 1.6e-3).  Hence 1e-2 for (a); the planted errors of tests/test_tc_mlp_gpu.py (a dropped
# or swapped xyz / skip column, a dropped bias slice, round-toward-zero operands, an unwritten last tile) make 0.1 to
# 0.9 of the elements differ, 10x and more above it.
FRAC_REL = 1e-4
FRAC_MAX = 1e-2
MAX_REL = 1e-2


def stats(got, ref):
    """(fraction of elements with |got - ref| > FRAC_REL * max|ref|, max|got - ref| / max|ref|), in float64."""
    ref = ref.to(F64)
    got = got.to(device=ref.device, dtype=F64)
    scale = ref.abs().max().item()
    if scale == 0.0:
        scale = 1.0
    d = (got - ref).abs()
    return (d > FRAC_REL * scale).double().mean().item(), d.max().item() / scale


def agrees(got, ref):
    """The acceptance rule of the tensor-core kernel against this reference: (a) and (b) above."""
    frac, mx = stats(got, ref)
    return frac <= FRAC_MAX and mx <= MAX_REL
