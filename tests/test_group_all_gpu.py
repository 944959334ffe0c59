"""The group_all SA layer (one group of all N points per cloud, model/pointnet_util.py:50-67) on the project's kernels:
the fp32 inference kernel (pn2_sa_all_mlp_max) against the reference vectors and a float64 CPU copy of the module, its
output slice and repeatability, the training Function (train_mlp.sa_all_train) against the composition it replaces and
against float64, ties, which path runs when, and a graphed training step of a small classifier."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from module_cases import MODS, mgm, unit_seed
from oracle.seeded import fill_seeded
from pn2_b200 import pointnet2_utils, pointnet_util as pu, train_mlp
from pn2_b200.pointnet_util import PointNetSetAbstraction, sample_and_group_all, set_fused_training
from test_train_blocks_gpu import _compare, _grad_errs, _kernel_names, rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["fp32", "bf16"])
def precision(request):
    prev = pu.set_mlp_precision(request.param)
    yield request.param
    pu.set_mlp_precision(prev)


def _randomize_bn(mod, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for bn in mod.mlp_bns:
            c = bn.num_features
            bn.weight.copy_(torch.rand(c, generator=g) + 0.5)
            bn.bias.copy_(torch.randn(c, generator=g) * 0.1)
            bn.running_mean.copy_(torch.randn(c, generator=g) * 0.1)
            bn.running_var.copy_(torch.rand(c, generator=g) + 0.5)
    return mod


# ---- 1. the reference's own vectors --------------------------------------------------------------------------------------
def test_golden_group_all_meets_the_fp32_bound(cuda, precision):
    gold = np.load(MODS)
    name = "sa_group_all"
    _, args, B, N, D, _ = mgm.UNIT_CASES[name]
    mod = fill_seeded(PointNetSetAbstraction(*args), unit_seed(name)).eval().to(cuda)
    xyz, feat = [torch.from_numpy(a).to(cuda) for a in mgm.unit_inputs(name)]
    with torch.no_grad():
        new_xyz, out = mod(xyz, feat)
    assert new_xyz.shape == (B, 3, 1) and bool((new_xyz == 0).all())
    want = gold[name + "/out"]
    err = float(np.abs(out.cpu().numpy() - want).max() / np.abs(want).max())
    print("sa_group_all %s: max error %.3e of max|ref|" % (precision, err))
    assert err <= 1e-5, err


# ---- 2. eval against a float64 CPU copy (on the CPU the module is the reference composition) --------------------------------
SMALL, WIDE, SIX = [32, 64], [256, 512, 1024], [64, 64, 128, 128, 64, 32]


@pytest.mark.parametrize("N,B,D,stack", [
    (1, 1, 5, SMALL), (7, 3, 0, SMALL), (16, 3, 5, SMALL), (128, 1, 256, SMALL), (129, 3, 5, SMALL), (1000, 3, 256, SMALL),
    (8192, 3, 5, SMALL), (1, 3, 256, WIDE), (7, 1, 5, WIDE), (128, 3, 256, WIDE), (129, 3, 0, WIDE), (1000, 3, 256, WIDE),
    (7, 3, 5, SIX), (129, 1, 256, SIX), (8192, 1, 0, SIX),
])
def test_eval_matches_float64(cuda, N, B, D, stack):
    torch.manual_seed(N * 7 + B + D)
    mod = _randomize_bn(PointNetSetAbstraction(None, None, None, 3 + D, stack, True), N + D).eval()
    xyz, feat = torch.randn(B, 3, N), (torch.randn(B, D, N) if D else None)
    with torch.no_grad():
        _, ref = copy.deepcopy(mod).double()(xyz.double(), None if feat is None else feat.double())
        g = mod.to(cuda)
        for prec in ("fp32", "bf16"):   # the group_all kernel is fp32 under both settings
            prev = pu.set_mlp_precision(prec)
            try:
                new_xyz, out = g(xyz.to(cuda), None if feat is None else feat.to(cuda))
            finally:
                pu.set_mlp_precision(prev)
            assert out.shape == ref.shape and bool((new_xyz == 0).all())
            err = float((out.cpu().double() - ref).abs().max() / ref.abs().max())
            assert err <= 1e-5, (prec, err)


# ---- 3. output slice, repeatability, graph replay -------------------------------------------------------------------------
def test_out_slice_is_exact_and_repeatable(cuda):
    torch.manual_seed(3)
    B, N, D, C, W, off = 3, 8192, 64, 128, 141, 5   # many tiles per cloud: the cross-CTA combine is exercised
    mod = _randomize_bn(PointNetSetAbstraction(None, None, None, 3 + D, [64, C], True), 3).eval().to(cuda)
    mlp = mod.folded()
    xyz, feat = torch.randn(B, N, 3, device=cuda), torch.randn(B, N, D, device=cuda)
    sentinel = -12345.5
    ref = pu.sa_all_mlp_max_cl(xyz, feat, mlp)
    outs = []
    for _ in range(2):
        out = torch.full((B, 1, W), sentinel, device=cuda)
        pu.sa_all_mlp_max_cl(xyz, feat, mlp, out=out, out_offset=off)
        outs.append(out)
    graph_out = torch.full((B, 1, W), sentinel, device=cuda)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pu.sa_all_mlp_max_cl(xyz, feat, mlp, out=graph_out, out_offset=off)   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        pu.sa_all_mlp_max_cl(xyz, feat, mlp, out=graph_out, out_offset=off)
    graph_out.fill_(sentinel)
    graph.replay()
    torch.cuda.synchronize()
    for out in outs + [graph_out]:
        assert torch.equal(out[:, :, off:off + C], ref)
        assert bool((out[:, :, :off] == sentinel).all()) and bool((out[:, :, off + C:] == sentinel).all())
    assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))
    assert torch.equal(outs[0].view(torch.int32), graph_out.view(torch.int32))


# ---- 4. training against the composition it replaces and against float64 -------------------------------------------------
def _old_all(mod, xyz, points):
    _, grouped = sample_and_group_all(xyz.permute(0, 2, 1), points.permute(0, 2, 1) if points is not None else None)
    B, S, K, C0 = grouped.shape
    a = train_mlp.fused_mlp_train(grouped.reshape(B * S * K, C0), mod.mlp_convs, mod.mlp_bns)
    return a.view(B, S, K, -1).max(dim=2)[0].permute(0, 2, 1)


@pytest.mark.parametrize("B,N,D,stack", [(2, 1000, 0, [32, 64]), (3, 129, 9, [32, 64, 48]), (9, 8192, 16, [32, 64]),
                                         (2, 128, 256, [256, 512, 1024])])
def test_training_matches_the_composition_it_replaces(cuda, B, N, D, stack):
    torch.manual_seed(B + N + D)
    sa = PointNetSetAbstraction(None, None, None, 3 + D, stack, True).to(cuda).train()
    xyz = torch.randn(B, 3, N, device=cuda)
    feat = torch.randn(B, N, D, device=cuda, requires_grad=True).permute(0, 2, 1) if D else None  # channel-last view
    _compare(lambda ms, xs: ms[0](xs[0], xs[1])[1], lambda ms, xs: _old_all(ms[0], xs[0], xs[1]), [sa], [xyz, feat],
             lambda m: m.mlp_bns)


@pytest.mark.parametrize("B,N,D", [(3, 129, 5), (2, 1000, 0)])
def test_training_matches_float64(cuda, B, N, D):
    torch.manual_seed(20 + D)
    sa = PointNetSetAbstraction(None, None, None, 3 + D, [32, 64], True).train()
    xyz, feat, target = torch.randn(B, 3, N), (torch.randn(B, D, N) if D else None), torch.randn(B, 64, 1)
    res = []
    for dev, dt in (("cpu", torch.float64), (cuda, torch.float32)):
        m = copy.deepcopy(sa).to(dev, dt)
        f = feat.to(dev, dt).requires_grad_(True) if D else None
        _, out = m(xyz.to(dev, dt), f)
        loss = ((out - target.to(dev, dt)) ** 2).mean()
        loss.backward()
        res.append((float(loss.detach()), f.grad if D else None, [p.grad for p in m.parameters()], m))
    (l0, f0, p0, m0), (l1, f1, p1, m1) = res
    assert abs(l1 - l0) <= 1e-5 * abs(l0)
    if D:
        assert rel_err(f1, f0) <= 2e-4
    bias_ids = {id(c.bias) for c in m1.mlp_convs}   # exactly-zero true gradient (a batch-statistics BatchNorm follows)
    keep = [i for i, q in enumerate(m1.parameters()) if id(q) not in bias_ids]
    assert max(_grad_errs([p1[i] for i in keep], [p0[i].float() for i in keep])) <= 2e-4
    for bg, br in zip(m1.mlp_bns, m0.mlp_bns):
        np.testing.assert_allclose(bg.running_mean.cpu().numpy(), br.running_mean.numpy(), rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(bg.running_var.cpu().numpy(), br.running_var.numpy(), rtol=1e-4, atol=1e-6)
        assert int(bg.num_batches_tracked) == 1


# ---- 5. ties -----------------------------------------------------------------------------------------------------------------
def test_ties_route_to_the_first_maximum(cuda):
    """Every point is one of 16 base points (coordinates AND features), so each cloud holds many identical rows: exact
    ties at non-zero activations between different points.  A quarter of the last layer's channels get a BatchNorm shift
    that makes them 0 on every row.  The feature gradient must be the composition's: torch.max sends it to the first
    maximum."""
    torch.manual_seed(9)
    B, N, D, base_n = 2, 1000, 6, 16
    pick = torch.randint(0, base_n, (B, N))
    base_xyz, base_feat = torch.randn(B, base_n, 3), torch.randn(B, base_n, D)
    xyz = torch.gather(base_xyz, 1, pick[:, :, None].expand(B, N, 3)).permute(0, 2, 1).contiguous().to(cuda)
    feat_cl = torch.gather(base_feat, 1, pick[:, :, None].expand(B, N, D)).contiguous().to(cuda).requires_grad_(True)
    sa = PointNetSetAbstraction(None, None, None, 3 + D, [16, 32], True).to(cuda).train()
    with torch.no_grad():
        sa.mlp_bns[-1].bias[:8] = -100.0   # |zhat| <= sqrt(rows) < 50: these columns are 0 after the ReLU everywhere
    out = copy.deepcopy(sa)(xyz, feat_cl.detach().permute(0, 2, 1))[1]
    assert bool((out[:, :8] == 0).all()) and bool((out[:, 8:] > 0).any())
    _compare(lambda ms, xs: ms[0](xs[0], xs[1])[1], lambda ms, xs: _old_all(ms[0], xs[0], xs[1]), [sa],
             [xyz, feat_cl.permute(0, 2, 1)], lambda m: m.mlp_bns)


# ---- 6. which path runs when -------------------------------------------------------------------------------------------------
def _ours_or_fill(names):
    """Kernels that are neither the project's (namespace pn2) nor a zero fill / a num_batches_tracked increment."""
    return [k for k in names if "pn2::" not in k and "FillFunctor" not in k and not ("long" in k and "add" in k.lower())
            and not k.startswith("Memset")]


def _nodes(t):
    seen, todo = [], [t.grad_fn]
    while todo and len(seen) < 50:
        node = todo.pop()
        if node is None:
            continue
        seen.append(type(node).__name__)
        todo += [n for n, _ in node.next_functions]
    return seen


def test_eval_issues_the_kernel_and_no_torch_compute(cuda):
    torch.manual_seed(10)
    B, N, D = 2, 1000, 32
    mod = PointNetSetAbstraction(None, None, None, 3 + D, [64, 128], True).to(cuda).eval()
    xyz, feat = torch.randn(B, 3, N, device=cuda), torch.randn(B, D, N, device=cuda)

    def run():
        with torch.no_grad():
            mod(xyz, feat)

    run()
    names = _kernel_names(run)
    assert any("row_mlp_kernel" in k for k in names), names
    assert not _ours_or_fill(names), sorted(set(_ours_or_fill(names)))


def test_training_issues_the_function_and_no_cat_or_max_kernels(cuda):
    torch.manual_seed(11)
    B, N, D = 2, 1000, 32
    sa = PointNetSetAbstraction(None, None, None, 3 + D, [64, 128], True).to(cuda).train()
    xyz = torch.randn(B, N, 3, device=cuda).permute(0, 2, 1)   # channel-last, as new_xyz travels between blocks
    feat_cl = torch.randn(B, N, D, device=cuda, requires_grad=True)
    g = torch.randn(B, 1, 128, device=cuda).permute(0, 2, 1)

    def step():
        for t in [feat_cl] + list(sa.parameters()):
            t.grad = None
        _, out = sa(xyz, feat_cl.permute(0, 2, 1))
        out.backward(g)

    step()
    names = _kernel_names(step)
    assert not _ours_or_fill(names), sorted(set(_ours_or_fill(names)))
    assert any("train_bn_relu_max_all_kernel" in k for k in names) and any("train_max_bwd_kernel" in k for k in names)
    _, out = sa(xyz, feat_cl.permute(0, 2, 1))
    assert any("SaAllTrain" in c for c in _nodes(out))


@pytest.mark.parametrize("mode", ["xyz_grad", "deterministic", "unfused"])
def test_other_modes_keep_the_composed_path(cuda, mode):
    torch.manual_seed(12)
    B, N, D = 2, 300, 6
    sa = PointNetSetAbstraction(None, None, None, 3 + D, [16, 32], True).to(cuda).train()
    xyz = torch.randn(B, 3, N, device=cuda).requires_grad_(mode == "xyz_grad")
    feat = torch.randn(B, D, N, device=cuda, requires_grad=True)
    prev_det = pointnet2_utils.set_deterministic(mode == "deterministic")
    prev_fused = set_fused_training(mode != "unfused")
    try:
        _, out = sa(xyz, feat)
        chain = _nodes(out)
        out.square().mean().backward()
    finally:
        pointnet2_utils.set_deterministic(prev_det)
        set_fused_training(prev_fused)
    assert not any("SaAllTrain" in c for c in chain), chain
    assert feat.grad is not None and bool(torch.isfinite(feat.grad).all())
    if mode == "xyz_grad":
        assert xyz.grad is not None and float(xyz.grad.abs().max()) > 0


# ---- 7. a small classifier, eager and graphed ----------------------------------------------------------------------------------
class _TinyCls(torch.nn.Module):
    def __init__(self, D, classes):
        super().__init__()
        self.sa1 = PointNetSetAbstraction(128, 0.4, 16, 3 + D, [32, 64], False)
        self.sa2 = PointNetSetAbstraction(None, None, None, 3 + 64, [64, 128], True)
        self.fc = torch.nn.Linear(128, classes)

    def forward(self, xyz, feat):
        l1_xyz, l1 = self.sa1(xyz, feat)
        _, l2 = self.sa2(l1_xyz, l1)
        return self.fc(l2.reshape(l2.shape[0], -1))


def test_graphed_classifier_step_reproduces_the_eager_loop(cuda):
    from pn2_b200.models import GraphedTrainStep
    B, N, D, classes = 8, 1024, 4, 10
    g = torch.Generator(device=cuda).manual_seed(13)
    xyz = torch.rand(B, 3, N, device=cuda, generator=g)
    feat = torch.randn(B, D, N, device=cuda, generator=g)
    target = torch.randint(0, classes, (B,), device=cuda, generator=g)

    def make():
        torch.manual_seed(14)
        net = _TinyCls(D, classes).to(cuda).train()
        return net, torch.optim.Adam(net.parameters(), lr=1e-3, capturable=True)

    net_e, opt_e = make()
    eager, eager_grads = [], None
    for _ in range(3):
        opt_e.zero_grad(set_to_none=True)
        loss = F.cross_entropy(net_e(xyz, feat), target)
        loss.backward()
        if eager_grads is None:
            eager_grads = [p.grad.detach().clone() for p in net_e.parameters()]
        opt_e.step()
        eager.append(float(loss.detach()))
    assert any("SaAllTrain" in c for c in _nodes(loss))
    net_g, opt_g = make()
    stepper = GraphedTrainStep(net_g, opt_g, F.cross_entropy, xyz, feat, target)
    graphed = [float(stepper.step(xyz, feat, target))]
    graphed_grads = [p.grad.detach().clone() for p in net_g.parameters()]
    graphed += [float(stepper.step(xyz, feat, target)) for _ in range(2)]
    torch.cuda.synchronize()
    for a, b in zip(graphed, eager):
        assert abs(a - b) <= 2e-4 * abs(b), (graphed, eager)
    assert max(_grad_errs(graphed_grads, eager_grads)) <= 2e-4
