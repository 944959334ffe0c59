"""BatchNorm layers that normalise with their RUNNING statistics on the fused training kernels: eval() networks under
autograd and frozen-BatchNorm fine-tuning (`net.train()`, then `m.eval()` on every BatchNorm), and stacks that mix the two
modes.  Every block against a float64 CPU run of the reference's composition (torch modules in float64, each BatchNorm in
the same mode, neighbour indices from the GPU geometry kernels), the running statistics, the no-grad inference output,
which kernels run, and graph replay."""
import copy
import re

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from pn2_b200 import models, pointnet2_utils, pointnet_util, scenes, train_mlp
from pn2_b200.pointnet_util import (PointNetFeaturePropagation, PointNetSetAbstraction, PointNetSetAbstractionMsg,
                                    set_mlp_precision)

pytestmark = pytest.mark.gpu

MODES = ["eval", "frozen", "mixed"]


def rel_err(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _grad_errs(pgrads, pgrads_ref):
    # as in test_train_blocks_gpu.py: errors against the largest parameter gradient, with a floor of 5 % of it (the conv
    # biases of batch-statistics layers have an exactly-zero true gradient)
    scale = max(float(r.abs().max()) for r in pgrads_ref)
    return [float((g.detach().cpu().double() - r.cpu()).abs().max()) / max(float(r.abs().max()), 0.05 * scale)
            for g, r in zip(pgrads, pgrads_ref)]


def _bns(mod):
    return [m for m in mod.modules() if isinstance(m, nn.modules.batchnorm._BatchNorm)]


def _prepare(mod, seed, mode):
    """Non-trivial affine and running statistics, then the BatchNorm modes: "eval" = mod.eval(); "frozen" = mod.train()
    with every BatchNorm in eval; "mixed" = mod.train() with every other BatchNorm (the first of each stack) in eval."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for bn in _bns(mod):
            c = bn.num_features
            bn.weight.copy_(torch.rand(c, generator=g) + 0.5)
            bn.bias.copy_(torch.randn(c, generator=g) * 0.1)
            if bn.running_mean is not None:
                bn.running_mean.copy_(torch.randn(c, generator=g) * 0.1)
                bn.running_var.copy_(torch.rand(c, generator=g) + 0.5)
    for m in mod.modules():
        if isinstance(m, nn.Dropout):
            m.p = 0.0
    if mode == "eval":
        mod.eval()
    else:
        mod.train()
        for i, bn in enumerate(_bns(mod)):
            if mode == "frozen" or i % 2 == 0:
                bn.eval()
    return mod


def _cloud(seed, B, N):
    return torch.from_numpy(scenes.scannet_batch(seed, B, N)[:, :, :3]).permute(0, 2, 1).contiguous()


# ---- float64 restatement of the reference's composition (model/pointnet_util.py) on the GPU's neighbour indices --------------
def _sa_geometry(xyz_gpu, npoint, radii, nsamples):
    """new_xyz (B, S, 3) and ball indices per radius, exactly as the modules compute them."""
    xyz_cl = xyz_gpu.permute(0, 2, 1).contiguous()
    _, new_xyz = pointnet_util.fps_gather_cl(xyz_cl, npoint)
    idxs = [pointnet2_utils.ball_query(r, k, xyz_cl, new_xyz).long().cpu() for r, k in zip(radii, nsamples)]
    return new_xyz.cpu().double(), idxs


def _group(xyz, feat, new_xyz, idx, feat_first):
    """-> (B, C, K, S): [centred xyz | feat] (SSG) or [feat | centred xyz] (MSG) of every ball."""
    B = xyz.shape[0]
    S, K = idx.shape[1], idx.shape[2]
    flat = idx.reshape(B, 1, S * K)
    gx = torch.gather(xyz, 2, flat.expand(B, 3, S * K)).reshape(B, 3, S, K) - new_xyz.permute(0, 2, 1)[..., None]
    parts = [gx]
    if feat is not None:
        gf = torch.gather(feat, 2, flat.expand(B, feat.shape[1], S * K)).reshape(B, feat.shape[1], S, K)
        parts = [gf, gx] if feat_first else [gx, gf]
    return torch.cat(parts, 1).permute(0, 1, 3, 2)


def _stack(x, convs, bns):
    for conv, bn in zip(convs, bns):
        x = F.relu(bn(conv(x)))
    return x


def _interp(feat2, idx, w, n):
    B, D2, m = feat2.shape
    if m == 1:
        return feat2.expand(B, D2, n)
    out = 0
    for j in range(3):
        out = out + torch.gather(feat2, 2, idx[:, None, :, j].expand(B, D2, n)) * w[:, None, :, j]
    return out


# ---- the cases: (modules, inputs needing grad, GPU forward, float64 reference forward) ---------------------------------------
def _case(name, cuda):
    torch.manual_seed(3)
    B = 2
    if name == "ssg":
        D, N = 6, 1024
        sa = PointNetSetAbstraction(128, 0.3, 32, D + 3, [16, 32, 24], False)
        xyz = _cloud(21, B, N)
        new_xyz, (idx,) = _sa_geometry(xyz.to(cuda), 128, [0.3], [32])

        def ref(ms, xs):
            return _stack(_group(xyz.double(), xs[0], new_xyz, idx, False), ms[0].mlp_convs, ms[0].mlp_bns).max(dim=2)[0]
        return [sa], [torch.randn(B, D, N)], lambda ms, xs: ms[0](xyz.to(cuda), xs[0])[1], ref
    if name == "msg":
        D, N = 9, 1024
        msg = PointNetSetAbstractionMsg(128, [0.15, 0.3], [16, 32], D, [[16, 32], [24, 16, 32]])
        xyz = _cloud(22, B, N)
        new_xyz, idxs = _sa_geometry(xyz.to(cuda), 128, msg.radius_list, msg.nsample_list)

        def ref(ms, xs):
            outs = [_stack(_group(xyz.double(), xs[0], new_xyz, idx, True), ms[0].conv_blocks[i], ms[0].bn_blocks[i]).max(dim=2)[0]
                    for i, idx in enumerate(idxs)]
            return torch.cat(outs, 1)
        return [msg], [torch.randn(B, D, N)], lambda ms, xs: ms[0](xyz.to(cuda), xs[0])[1], ref
    if name in ("fp_skip", "fp_noskip", "fp_one"):
        n, m, D1, D2 = 1024, (1 if name == "fp_one" else 256), (0 if name == "fp_noskip" else 7), 33
        fp = PointNetFeaturePropagation(D1 + D2, [32, 24, 16])
        xyz1 = _cloud(23, B, n)
        xyz2 = xyz1[:, :, :m].contiguous()
        if m > 1:
            idx, w = pointnet_util._three_nn_weights_torch(xyz1.to(cuda).permute(0, 2, 1).contiguous(),
                                                          xyz2.to(cuda).permute(0, 2, 1).contiguous())
            idx, w = idx.long().cpu(), w.cpu().double()
        else:
            idx = w = None
        inputs = ([torch.randn(B, D1, n)] if D1 else []) + [torch.randn(B, D2, m)]

        def gpu(ms, xs):
            p1, p2 = (xs[0], xs[1]) if D1 else (None, xs[0])
            return ms[0](xyz1.to(cuda), xyz2.to(cuda), p1, p2)

        def ref(ms, xs):
            p1, p2 = (xs[0], xs[1]) if D1 else (None, xs[0])
            rows = _interp(p2, idx, w, n)
            if p1 is not None:
                rows = torch.cat([p1, rows], 1)
            return _stack(rows, ms[0].mlp_convs, ms[0].mlp_bns)
        return [fp], inputs, gpu, ref
    if name == "group_all":
        D, N = 5, 1024
        sa = PointNetSetAbstraction(None, None, None, 3 + D, [16, 32], True)
        xyz = torch.randn(B, 3, N)

        def ref(ms, xs):
            rows = torch.cat([xyz.double(), xs[0]], 1)[..., None]  # (B, 3 + D, N, 1): not centred
            return _stack(rows, ms[0].mlp_convs, ms[0].mlp_bns).max(dim=2)[0]
        return [sa], [torch.randn(B, D, N)], lambda ms, xs: ms[0](xyz.to(cuda), xs[0])[1], ref
    if name == "mlp":
        R, widths = 3000, [10, 32, 24, 16]
        stack = nn.ModuleList([nn.Conv1d(widths[i], widths[i + 1], 1) for i in range(3)] +
                              [nn.BatchNorm1d(widths[i + 1]) for i in range(3)])

        def gpu(ms, xs):
            return train_mlp.fused_mlp_train(xs[0], list(ms[0])[:3], list(ms[0])[3:])

        def ref(ms, xs):
            return _stack(xs[0].t()[None], list(ms[0])[:3], list(ms[0])[3:])[0].t()
        return [stack], [torch.randn(R, widths[0])], gpu, ref
    if name == "head":
        N = 2048
        net = models.PointNet2SemSeg(13)

        def ref(ms, xs):
            m = ms[0]
            return m.conv2(F.relu(m.bn1(m.conv1(xs[0])))).permute(0, 2, 1)
        return [net], [torch.randn(B, 128, N)], lambda ms, xs: models._semseg_head(ms[0], xs[0]), ref
    raise KeyError(name)


CASES = ["ssg", "msg", "fp_skip", "fp_noskip", "fp_one", "group_all", "mlp", "head"]
BLOCK_FN = {"ssg": "_SaScaleTrain", "msg": "_SaScaleTrain", "fp_skip": "_FpBlockTrain", "fp_noskip": "_FpBlockTrain",
            "fp_one": "_FpBlockTrain", "group_all": "_SaAllTrain", "mlp": "_FusedMlpTrain", "head": "_FusedMlpTrain"}


def _graph_nodes(t):
    seen, todo, names = set(), [t.grad_fn], []
    while todo:
        node = todo.pop()
        if node is None or node in seen:
            continue
        seen.add(node)
        names.append(type(node).__name__)
        todo += [f for f, _ in node.next_functions]
    return names


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", CASES)
def test_block_matches_float64_composition(cuda, case, mode):
    mods, inputs, gpu_fn, ref_fn = _case(case, cuda)
    mods = [_prepare(m, 17, mode) for m in mods]
    g_mods = [copy.deepcopy(m).to(cuda) for m in mods]
    r_mods = [copy.deepcopy(m).double() for m in mods]
    before = [(bn.training, bn.running_mean.clone(), bn.running_var.clone(), int(bn.num_batches_tracked))
              for m in g_mods for bn in _bns(m)]
    gx = [t.to(cuda).requires_grad_(True) for t in inputs]
    rx = [t.double().requires_grad_(True) for t in inputs]
    out, ref = gpu_fn(g_mods, gx), ref_fn(r_mods, rx)
    assert out.shape == ref.shape
    assert BLOCK_FN[case] + "Backward" in _graph_nodes(out)
    target = torch.randn(ref.shape, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    loss = ((out - target.to(cuda).float()) ** 2).mean()
    loss_ref = ((ref - target) ** 2).mean()
    loss.backward()
    loss_ref.backward()

    assert rel_err(out, ref) <= 1e-5
    assert abs(float(loss.detach()) - float(loss_ref.detach())) <= 1e-5 * abs(float(loss_ref.detach()))
    for a, b in zip(gx, rx):
        assert rel_err(a.grad, b.grad) <= 2e-4, (rel_err(a.grad, b.grad))
    pg = [p.grad for m in g_mods for p in m.parameters()]
    pr = [p.grad for m in r_mods for p in m.parameters()]
    used = [i for i, r in enumerate(pr) if r is not None]  # the head case holds a whole network; only its head is used
    assert all(pg[i] is not None for i in used)
    errs = _grad_errs([pg[i] for i in used], [pr[i] for i in used])
    assert max(errs) <= 2e-4, errs
    # the conv bias in front of a running-statistics BatchNorm has a real gradient (sum dz)
    for mg, mr in zip(g_mods, r_mods):
        convs = [c for c in mg.modules() if isinstance(c, (nn.Conv1d, nn.Conv2d))]
        convs_r = [c for c in mr.modules() if isinstance(c, (nn.Conv1d, nn.Conv2d))]
        bns_g = _bns(mg)
        for c, cr, bn in zip(convs, convs_r, bns_g):
            if not bn.training and c.bias.grad is not None:
                assert float(cr.bias.grad.abs().max()) > 0 and float(c.bias.grad.abs().max()) > 0
    # running-statistics layers leave their state bit-unchanged; batch-statistics layers update it as the composition does
    for (was_training, rm, rv, nbt), bn, bn_r in zip(before, [b for m in g_mods for b in _bns(m)], [b for m in r_mods for b in _bns(m)]):
        if not was_training:
            assert torch.equal(bn.running_mean, rm) and torch.equal(bn.running_var, rv)
            assert int(bn.num_batches_tracked) == nbt
        else:
            np.testing.assert_allclose(bn.running_mean.cpu().numpy(), bn_r.running_mean.numpy(), rtol=1e-4, atol=1e-6)
            np.testing.assert_allclose(bn.running_var.cpu().numpy(), bn_r.running_var.numpy(), rtol=1e-4, atol=1e-6)
            assert int(bn.num_batches_tracked) == int(bn_r.num_batches_tracked)  # nbt + 1 where the layer ran


def test_frozen_recipe_leaves_running_statistics_untouched(cuda):
    """net.train(), then m.eval() on every BatchNorm: a fine-tuning step must not move the running statistics (it did when
    the fused training path normalised every layer with the batch statistics)."""
    torch.manual_seed(9)
    net = _prepare(models.PointNet2SemSeg(13), 4, "frozen").to(cuda)
    pts = torch.from_numpy(scenes.scannet_batch(6, 2, 2048)).permute(0, 2, 1).contiguous().to(cuda)
    state = {k: v.clone() for k, v in net.state_dict().items() if "running" in k or "num_batches" in k}
    out = net(pts[:, :3].contiguous(), pts[:, 3:].contiguous())
    out.square().mean().backward()
    for k, v in state.items():
        assert torch.equal(net.state_dict()[k], v), k


def test_track_running_stats_false_uses_batch_statistics_in_eval(cuda):
    torch.manual_seed(10)
    D, B, N = 6, 2, 1024
    sa = PointNetSetAbstraction(128, 0.3, 32, D + 3, [16, 32], False)
    sa.mlp_bns = nn.ModuleList([nn.BatchNorm2d(16, track_running_stats=False), nn.BatchNorm2d(32, track_running_stats=False)])
    sa = _prepare(sa, 2, "eval")
    xyz = _cloud(24, B, N)
    new_xyz, (idx,) = _sa_geometry(xyz.to(cuda), 128, [0.3], [32])
    feat = torch.randn(B, D, N)
    sg, sr = copy.deepcopy(sa).to(cuda), copy.deepcopy(sa).double()
    fg, fr = feat.to(cuda).requires_grad_(True), feat.double().requires_grad_(True)
    out = sg(xyz.to(cuda), fg)[1]
    ref = _stack(_group(xyz.double(), fr, new_xyz, idx, False), sr.mlp_convs, sr.mlp_bns).max(dim=2)[0]
    assert "_SaScaleTrainBackward" in _graph_nodes(out)
    assert rel_err(out, ref) <= 1e-5
    out.sum().backward()
    ref.sum().backward()
    assert rel_err(fg.grad, fr.grad) <= 2e-4


def test_eval_with_coordinate_gradient_matches_float64_composition(cuda):
    """eval() with coordinates that need a gradient: the grouping stays the composition (differentiable gathers of xyz
    and new_xyz), its MLP runs on the fused training chain with the running statistics."""
    torch.manual_seed(14)
    D, B, N, S, K = 6, 2, 1024, 128, 32
    sa = _prepare(PointNetSetAbstraction(S, 0.3, K, D + 3, [16, 32], False), 12, "eval")
    xyz, feat = _cloud(26, B, N), torch.randn(B, D, N)
    xyz_g = xyz.to(cuda)
    fps = pointnet2_utils.furthest_point_sample(xyz_g.permute(0, 2, 1).contiguous(), S)
    new_xyz_g = pointnet2_utils.gather_operation(xyz_g.contiguous(), fps).permute(0, 2, 1).contiguous()
    idx = pointnet2_utils.ball_query(0.3, K, xyz_g.permute(0, 2, 1).contiguous(), new_xyz_g).long().cpu()
    fps = fps.long().cpu()
    sg, sr = copy.deepcopy(sa).to(cuda), copy.deepcopy(sa).double()
    before = [(bn.running_mean.clone(), bn.running_var.clone(), int(bn.num_batches_tracked)) for bn in sg.mlp_bns]
    xg, fg = xyz.to(cuda).requires_grad_(True), feat.to(cuda).requires_grad_(True)
    xr, fr = xyz.double().requires_grad_(True), feat.double().requires_grad_(True)
    out = sg(xg, fg)[1]
    new_xyz_r = torch.gather(xr, 2, fps[:, None, :].expand(B, 3, S)).permute(0, 2, 1)
    ref = _stack(_group(xr, fr, new_xyz_r, idx, False), sr.mlp_convs, sr.mlp_bns).max(dim=2)[0]
    nodes = _graph_nodes(out)
    assert "_FusedMlpTrainBackward" in nodes and "_SaScaleTrainBackward" not in nodes, nodes
    assert rel_err(out, ref) <= 1e-5
    target = torch.randn(ref.shape, generator=torch.Generator().manual_seed(6), dtype=torch.float64)
    ((out - target.to(cuda).float()) ** 2).mean().backward()
    ((ref - target) ** 2).mean().backward()
    assert rel_err(xg.grad, xr.grad) <= 2e-4 and rel_err(fg.grad, fr.grad) <= 2e-4
    assert max(_grad_errs([p.grad for p in sg.parameters()], [p.grad for p in sr.parameters()])) <= 2e-4
    for bn, (rm, rv, nbt) in zip(sg.mlp_bns, before):
        assert torch.equal(bn.running_mean, rm) and torch.equal(bn.running_var, rv) and int(bn.num_batches_tracked) == nbt


def _blocks_and_inputs(cuda):
    torch.manual_seed(11)
    B, N, D = 2, 2048, 6
    xyz = _cloud(25, B, N).to(cuda)
    feat = torch.randn(B, D, N, device=cuda)
    sa = PointNetSetAbstraction(256, 0.2, 32, D + 3, [32, 64], False)
    msg = PointNetSetAbstractionMsg(256, [0.1, 0.2], [16, 32], D, [[16, 32], [32, 32]])
    fp = PointNetFeaturePropagation(D + 64, [64, 32])
    ga = PointNetSetAbstraction(None, None, None, 3 + D, [32, 64], True)
    return [_prepare(m, 3, "eval").to(cuda) for m in (sa, msg, fp, ga)], xyz, feat


def test_forward_under_grad_matches_the_inference_kernels(cuda):
    """eval(): the output with autograd (running-statistics training kernels) and without (the fused inference kernels,
    fp32) agree within 1e-5 relative, block by block; the whole semseg network within 2e-5, as its own inference test
    allows for 13 layers of fp32 rounding."""
    prev = set_mlp_precision("fp32")
    try:
        (sa, msg, fp, ga), xyz, feat = _blocks_and_inputs(cuda)
        fg = feat.clone().requires_grad_(True)
        l1_xyz = sa(xyz, feat)[0]
        l1 = torch.randn(2, 64, l1_xyz.shape[2], device=cuda)
        calls = [lambda f: sa(xyz, f)[1], lambda f: msg(xyz, f)[1], lambda f: fp(xyz, l1_xyz, f, l1), lambda f: ga(xyz, f)[1]]
        for call in calls:
            with torch.no_grad():
                want = call(feat)
            got = call(fg)
            assert got.grad_fn is not None
            assert rel_err(got, want) <= 1e-5
        net = _prepare(models.PointNet2SemSeg(13), 5, "eval").to(cuda)
        pts = torch.from_numpy(scenes.scannet_batch(7, 2, 4096)).permute(0, 2, 1).contiguous().to(cuda)
        x, c = pts[:, :3].contiguous(), pts[:, 3:].contiguous()
        with torch.no_grad():
            want = net(x, c)
        got = net(x, c.clone().requires_grad_(True))
        assert got.grad_fn is not None
        assert rel_err(got, want) <= 2e-5
    finally:
        set_mlp_precision(prev)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


_NO_STATS = re.compile(r"train_linear_fwd_kernel.*(false|\(bool\)0|Lb0E)")
_STATS = re.compile(r"train_linear_fwd_kernel.*(true|\(bool\)1|Lb1E)")
_TORCH_CONV_BN = ("cudnn", "batch_norm", "batchnorm", "bn_fw_", "bn_bw_", "convolve", "conv2d", "conv1d", "fprop", "dgrad", "wgrad")


def test_eval_under_grad_runs_the_running_statistics_kernels(cuda):
    net = _prepare(models.PointNet2SemSeg(13), 6, "eval").to(cuda)
    pts = torch.from_numpy(scenes.scannet_batch(8, 2, 2048)).permute(0, 2, 1).contiguous().to(cuda)
    x, c = pts[:, :3].contiguous(), pts[:, 3:].contiguous()

    def step():
        net.zero_grad(set_to_none=True)
        out = net(x, c)
        out.square().mean().backward()
        return out

    out = step()  # warm-up
    nodes = _graph_nodes(out)
    for fn in ("_SaScaleTrainBackward", "_FpBlockTrainBackward", "_FusedMlpTrainBackward"):
        assert fn in nodes, nodes
    names = _kernel_names(step)
    assert not [k for k in names if any(s in k.lower() for s in _TORCH_CONV_BN)], sorted(set(names))
    assert any(_NO_STATS.search(k) for k in names) and not any(_STATS.search(k) for k in names)
    assert any("train_bn_running_kernel" in k for k in names) and any("train_bn_running_bwd_coeffs_kernel" in k for k in names)
    assert not any("train_bn_finalize_kernel" in k for k in names)
    # training mode: batch statistics everywhere, the statistics-reducing builds only
    net.train()
    step()
    names = _kernel_names(step)
    assert any(_STATS.search(k) for k in names) and not any(_NO_STATS.search(k) for k in names)
    assert not any("train_bn_running" in k for k in names)


def test_graphed_frozen_step_reproduces_the_eager_loop(cuda):
    B, N = 2, 2048
    pts = torch.from_numpy(scenes.scannet_batch(44, B, N)).to(cuda)
    xyz = pts[:, :, :3].permute(0, 2, 1).contiguous()
    rgb = pts[:, :, 3:].permute(0, 2, 1).contiguous()
    target = (pts[:, :, 2].clamp(0, 2.69) / 2.7 * 12).long() + 1

    def loss_fn(logits, tgt):
        return F.cross_entropy(logits.reshape(-1, 13), tgt.reshape(-1), ignore_index=0)

    def make():
        torch.manual_seed(8)
        net = _prepare(models.PointNet2SemSeg(13), 7, "frozen").to(cuda)
        return net, torch.optim.Adam(net.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)

    # gradients are compared at the first step (later steps amplify the atomics' rounding noise through Adam, see
    # test_graphed_msg_step_reproduces_the_eager_loop)
    net_e, opt_e = make()
    stats0 = {k: v.clone() for k, v in net_e.state_dict().items() if "running" in k or "num_batches" in k}
    eager, eager_grads = [], None
    for _ in range(3):
        opt_e.zero_grad(set_to_none=True)
        loss = loss_fn(net_e(xyz, rgb), target)
        loss.backward()
        if eager_grads is None:
            eager_grads = [p.grad.detach().clone() for p in net_e.parameters()]
        opt_e.step()
        eager.append(float(loss.detach()))
    net_g, opt_g = make()
    stepper = models.GraphedTrainStep(net_g, opt_g, loss_fn, xyz, rgb, target)
    graphed = [float(stepper.step(xyz, rgb, target))]
    graphed_grads = [p.grad.detach().clone() for p in net_g.parameters()]
    graphed += [float(stepper.step(xyz, rgb, target)) for _ in range(2)]
    torch.cuda.synchronize()
    for a, b in zip(graphed, eager):
        assert abs(a - b) <= 2e-4 * abs(b), (graphed, eager)
    assert max(_grad_errs(graphed_grads, [g.double() for g in eager_grads])) <= 2e-4
    for net in (net_e, net_g):
        for k, v in stats0.items():
            assert torch.equal(net.state_dict()[k], v), k
