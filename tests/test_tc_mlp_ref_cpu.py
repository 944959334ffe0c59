"""CPU checks of oracle/tc_mlp_ref.py, the bf16-exact reference the tensor-core MLP kernel is tested against
(tests/test_tc_mlp_gpu.py): its bf16 rounding is torch's, with bf16-exact operands it is plain float64 arithmetic, and on
small SA / FP blocks it stays within the fp32 path's 2e-2 of the reference's modules (oracle/modules_ref.py)."""
import numpy as np
import torch

from oracle import modules_ref
from oracle import oracle as orc
from oracle import tc_mlp_ref as ref
from pn2_b200 import scenes
from pn2_b200.pointnet_util import PointNetFeaturePropagation, PointNetSetAbstraction, fold_conv_bn


def _randomize_bn(mod, seed):
    g = torch.Generator().manual_seed(seed)
    for m in mod.modules():
        if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)


def _ties():
    """fp32 values exactly halfway between two bf16 neighbours, with even and with odd bf16 mantissa below."""
    g = torch.Generator().manual_seed(3)
    hi = torch.randint(0, 1 << 15, (4096,), generator=g, dtype=torch.int32) << 16  # positive finite bf16 patterns
    hi = hi[(hi >> 23) < 254]  # keep the exponent below the one that rounds to inf
    ties = (hi | 0x8000).view(torch.float32)
    return torch.cat([ties, -ties])


def test_bf16_rounding_equals_torch_including_ties():
    g = torch.Generator().manual_seed(0)
    x = torch.cat([torch.randn(200000, generator=g) * 10.0 ** torch.randint(-30, 30, (200000,), generator=g).float(),
                   _ties(),
                   torch.tensor([0.0, -0.0, 1.0, -1.0, 1e-45, -1e-45, 1e-40, 3.0e38, -3.0e38, 3.3895e38, float("inf"),
                                 -float("inf")]),
                   torch.randint(-(1 << 31), (1 << 31) - 1, (100000,), generator=g, dtype=torch.int64).to(torch.int32).view(torch.float32)])
    x = x[~torch.isnan(x)]  # NaN payloads are outside the reference's domain
    want = x.to(torch.bfloat16).to(torch.float64)
    got = ref.bf16_rn(x)
    assert torch.equal(got.view(torch.int64), want.view(torch.int64))
    # ties really are ties, and half of them round up (odd mantissa below), half down
    t = _ties()
    up = ref.bf16_rn(t).abs() > t.abs().double()
    assert 0.3 < up.double().mean().item() < 0.7
    # a float64 input is rounded to fp32 first, as the kernel's fp32 accumulators are
    d = torch.tensor([1.0 + 2.0 ** -8 + 2.0 ** -40], dtype=torch.float64)  # a tie in fp32, above it in float64
    assert ref.bf16_rn(d).item() == torch.tensor([1.0 + 2.0 ** -8]).to(torch.bfloat16).double().item()


def test_bf16_round_toward_zero_is_truncation():
    x = torch.tensor([1.0 + 2.0 ** -8 + 2.0 ** -20, -(1.0 + 2.0 ** -7 + 2.0 ** -9), 3.0])
    assert ref.bf16_rz(x).tolist() == [1.0, -(1.0 + 2.0 ** -7), 3.0]


def _bf16_exact(*shape, gen, scale=1.0):
    return (torch.randn(*shape, generator=gen) * scale).to(torch.bfloat16).to(torch.float32)


def test_exact_operands_give_plain_float64_arithmetic():
    """With bf16-exact inputs, weights and coordinates whose centring is bf16-exact, the reference is A W^T + b (one
    layer: no hidden rounding), ReLU, max over the samples, rounded once to fp32."""
    g = torch.Generator().manual_seed(1)
    B, N, M, K, D, C = 2, 50, 7, 8, 13, 24
    xyz = torch.randint(-64, 64, (B, N, 3), generator=g).float() / 32  # multiples of 1/32: differences exact in bf16
    new_xyz = torch.randint(-64, 64, (B, M, 3), generator=g).float() / 32
    feat = _bf16_exact(B, N, D, gen=g)
    idx = torch.randint(0, N, (B, M, K), generator=g, dtype=torch.int32)
    w = _bf16_exact(C, D + 3, gen=g, scale=0.3)
    b = torch.randn(C, generator=g)
    for order in (0, 1):
        got = ref.sa_ref(xyz, feat, new_xyz, idx, order, [(w, b, True)])
        xn, fn, nn, wn, bn = (t.double().numpy() for t in (xyz, feat, new_xyz, w, b))
        want = np.zeros((B, M, C))
        for bb in range(B):
            for j in range(M):
                rows = []
                for s in range(K):
                    p = int(idx[bb, j, s])
                    c = xn[bb, p] - nn[bb, j]
                    rows.append(np.concatenate([c, fn[bb, p]] if order == 0 else [fn[bb, p], c]))
                want[bb, j] = np.maximum(np.asarray(rows) @ wn.T + bn, 0.0).max(axis=0)
        np.testing.assert_allclose(got.numpy(), want.astype(np.float32).astype(np.float64), rtol=1e-7, atol=1e-7)

    # FP, m == 1 (the interpolation is a copy, so exact too) with a bf16-exact skip block
    f1 = _bf16_exact(B, 9, 5, gen=g)
    f2 = _bf16_exact(B, 1, 16, gen=g)
    w2 = _bf16_exact(C, 21, gen=g, scale=0.3)
    got = ref.fp_ref(f1, f2, None, None, 9, [(w2, b, False)])
    a = torch.cat([f1, f2.expand(B, 9, 16)], dim=-1).double()
    want = (a @ w2.double().t() + b.double()).float().double()
    assert torch.allclose(got, want, rtol=1e-7, atol=1e-7)


def test_interpolation_follows_the_kernels_fma_order():
    """interp = f32(fma(w2, a2, f32(fma(w0, a0, f32(w1 a1))))) -- not the plain weighted sum."""
    g = torch.Generator().manual_seed(2)
    f2 = torch.randn(1, 6, 4000, generator=g)
    idx = torch.randint(0, 6, (1, 50, 3), generator=g, dtype=torch.int32)
    wt = torch.rand(1, 50, 3, generator=g)
    got = ref.interpolate_f32(f2, idx, wt)
    a = f2[0].double()
    w = wt[0].double()
    for i in range(50):
        i0, i1, i2 = (int(v) for v in idx[0, i])
        t = (w[i, 1] * a[i1]).float().double()
        t = (w[i, 0] * a[i0] + t).float().double()
        t = (w[i, 2] * a[i2] + t).float().double()
        assert torch.equal(got[0, i], t)


def _close(got, want, rel):
    scale = want.abs().max().item()
    err = (got.double() - want.double()).abs().max().item()
    assert err <= rel * scale, "max abs err %.3e vs %.1e * %.3e" % (err, rel, scale)


def _scene(B, N, D, seed):
    pts = scenes.scannet_batch(seed, B, N)
    xyz = torch.from_numpy(pts[:, :, :3]).permute(0, 2, 1).contiguous()
    feat = torch.randn(B, D, N, generator=torch.Generator().manual_seed(seed))
    return xyz, feat


def test_sa_reference_within_bf16_tolerance_of_the_modules():
    torch.manual_seed(4)
    D = 13
    mod = PointNetSetAbstraction(64, 0.4, 32, D + 3, [32, 32, 64], False).eval()
    _randomize_bn(mod, 4)
    xyz, feat = _scene(2, 800, D, 40)
    with torch.no_grad():
        new_xyz, want = modules_ref.sa_forward_ref(mod, xyz, feat)
        nx, _, _, idx = modules_ref.sample_and_group_ref(mod.npoint, mod.radius, mod.nsample, xyz.permute(0, 2, 1),
                                                         feat.permute(0, 2, 1))
        layers = [fold_conv_bn(c, b) + (True,) for c, b in zip(mod.mlp_convs, mod.mlp_bns)]
        got = ref.sa_ref(xyz.permute(0, 2, 1).contiguous(), feat.permute(0, 2, 1).contiguous(), nx,
                         torch.from_numpy(idx), 0, layers)
    _close(got.permute(0, 2, 1), want, 2e-2)


def test_fp_reference_within_bf16_tolerance_of_the_modules():
    torch.manual_seed(5)
    D1, D2, S, N = 6, 64, 100, 700
    mod = PointNetFeaturePropagation(D1 + D2, [64, 32]).eval()
    _randomize_bn(mod, 5)
    xyz1, p1 = _scene(2, N, D1, 50)
    xyz2 = xyz1[:, :, :S].contiguous()
    p2 = torch.randn(2, D2, S, generator=torch.Generator().manual_seed(6))
    with torch.no_grad():
        want = modules_ref.fp_forward_ref(mod, xyz1, xyz2, p1, p2)
        dist, idx = orc.three_nn(np.ascontiguousarray(xyz1.permute(0, 2, 1).numpy()),
                                 np.ascontiguousarray(xyz2.permute(0, 2, 1).numpy()))
        dist = torch.from_numpy(dist)
        dist[dist < 1e-10] = 1e-10
        w = 1.0 / dist
        w = w / torch.sum(w, dim=-1, keepdim=True)
        layers = [fold_conv_bn(c, b) + (True,) for c, b in zip(mod.mlp_convs, mod.mlp_bns)]
        got = ref.fp_ref(p1.permute(0, 2, 1).contiguous(), p2.permute(0, 2, 1).contiguous(), torch.from_numpy(idx), w, N,
                         layers)
    _close(got.permute(0, 2, 1), want, 2e-2)


def test_acceptance_statistics():
    want = torch.linspace(-1.0, 1.0, 10000, dtype=torch.float64)
    assert ref.stats(want, want) == (0.0, 0.0)
    got = want.clone()
    got[:5] += 2e-4  # 5 of 10000 elements off by 2e-4 of the scale: (a) 5e-4 passes
    frac, mx = ref.stats(got, want)
    assert frac == 5e-4 and abs(mx - 2e-4) < 1e-12 and ref.agrees(got, want)
    got[:200] += 2e-4  # 2e-2 of the elements: (a) fails
    assert not ref.agrees(got, want)
    got = want.clone()
    got[0] += 0.02  # one element 2e-2 off: (b) fails
    assert not ref.agrees(got, want)
