"""GPU: the backward of the multi-view lifting with respect to the 2-D feature maps (pn2_lift_views_grad, lift_views under
autograd).  Anchors: the float64 restatement oracle/lift_grad_ref.lift_grad_ref, itself pinned to torch autograd through the
reference's composition (Projection.apply per view + view reduction) by tests/test_lift_grad_ref_cpu.py; and that
composition on the GPU for the end-to-end training step."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import lift_grad_ref as lgr
from pn2_b200 import _lib, projection, scenes

pytestmark = pytest.mark.gpu

INTR = torch.from_numpy(scenes.SCANNET_INTRINSIC)
DMIN, DMAX = scenes.SCANNET_DEPTH_RANGE
ACC = scenes.SCANNET_ACCURACY
DIMS = scenes.SCANNET_IMAGE_DIMS


def make_batch(B, N, V, C, seed):
    xyz, feats, depth, poses = [], [], [], []
    for b in range(B):
        x, _ = scenes.scannet_scene(seed + b, N)
        f, d, p = scenes.multiview_inputs(seed + b, x, V, C)
        xyz.append(x); feats.append(f); depth.append(d); poses.append(p)
    return np.stack(xyz), np.stack(feats), np.stack(depth), np.stack(poses)


def dyadic(shape, seed, device):
    """integers in [-4, 4] x 2^-3: every fp32 sum of a few thousand of them is exact, whatever the order"""
    g = np.random.default_rng(seed).integers(-4, 5, size=shape) * 0.125
    return torch.from_numpy(g.astype(np.float32)).to(device)


def check_against_ref(cuda, xyz, feats, depth, poses, reduce, intr=INTR, dims=DIMS, acc=ACC, form="poses", seed=0):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    B, N = xyz.shape[:2]
    C = feats.shape[2]
    if form == "poses":
        kw = dict(camera_to_world=t(poses), view_parameters=None)
    else:
        kw = dict(camera_to_world=None, view_parameters=projection.view_params(t(poses), intr, DMIN, DMAX, dims))
    f = t(feats).requires_grad_(True)
    out, pix, count = projection.lift_views(t(xyz), f, t(depth), kw["camera_to_world"], intr, DMIN, DMAX, dims, acc,
                                            reduce=reduce, return_pixels=True, view_parameters=kw["view_parameters"])
    assert out.grad_fn is not None and not pix.requires_grad and not count.requires_grad
    g = dyadic((B, C, N), seed, cuda)
    out.backward(g)
    want = lgr.lift_grad_ref(feats, pix.cpu(), g.cpu(), reduce)
    got = f.grad.cpu().to(torch.float64)
    bad = (got != want).sum().item()
    assert bad == 0, "%d of %d elements differ (max |d| %g)" % (bad, got.numel(), (got - want).abs().max().item())
    assert (pix >= 0).float().mean() > 0.05, "the synthetic views must actually see the scene"
    assert want.abs().sum() > 0
    # the forward is the one without autograd, bit for bit
    with torch.no_grad():
        out0, pix0, count0 = projection.lift_views(t(xyz), t(feats), t(depth), kw["camera_to_world"], intr, DMIN, DMAX, dims,
                                                   acc, reduce=reduce, return_pixels=True, view_parameters=kw["view_parameters"])
    assert torch.equal(out.detach(), out0) and torch.equal(pix, pix0) and torch.equal(count, count0)


@pytest.mark.parametrize("form", ["poses", "view_parameters"])
@pytest.mark.parametrize("reduce", ["max", "first"])
@pytest.mark.parametrize("B,N,V,C", [(2, 8192, 3, 128), (1, 3001, 5, 6), (1, 8192, 5, 12), (2, 4096, 1, 16), (1, 2048, 8, 8)])
def test_backward_bit_exact_vs_restatement(cuda, form, reduce, B, N, V, C):
    """Synthetic scenes at the ENet map size: n % 4 != 0, C % 4 != 0, one view, eight views, grad_out rows staged in shared
    memory or read from global memory (8192 points x 5 views do not fit beside the slab)."""
    xyz, feats, depth, poses = make_batch(B, N, V, C, 40)
    if reduce == "first":
        feats[:, 0, :, 5, :] = 0.0    # seen all-zero columns in view 0: later views fill them
        feats[:, :, :, 9, :] = 0.0    # all-zero in every view: the gradient goes to view V-1 if it sees the point
    check_against_ref(cuda, xyz, feats, depth, poses, reduce, form=form, seed=B * N + V)


@pytest.mark.parametrize("form", ["poses", "view_parameters"])
@pytest.mark.parametrize("reduce", ["max", "first"])
@pytest.mark.parametrize("N", [2048, 13001])
def test_backward_with_maps_too_large_for_the_staged_forward(cuda, form, reduce, N):
    """3 views of 128 x 160 (V*H*W > 51 200): the forward runs lift_views_kernel, the backward reads the maps from global
    memory; with 13 001 points the grad_out rows do not fit shared memory either."""
    H, W, V, C = 128, 160, 3, 8
    x, _ = scenes.scannet_scene(90, N)
    _, _, poses = scenes.multiview_inputs(90, x, V, 4)
    intr = INTR.clone()
    intr[0, 0] *= W / DIMS[0]; intr[1, 1] *= H / DIMS[1]; intr[0, 2] = W / 2; intr[1, 2] = H / 2
    feats = np.random.default_rng(3).standard_normal((1, V, C, H, W)).astype(np.float32)
    if reduce == "first":
        feats[:, 1, :, ::3, :] = 0.0
    depth = np.full((1, V, H, W), 2.0, np.float32)  # with accuracy 100 every projected point passes the depth test
    check_against_ref(cuda, x[None], feats, depth, poses[None], reduce, intr=intr, dims=[W, H], acc=100.0, form=form, seed=N)


@pytest.mark.parametrize("reduce", ["max", "first"])
@pytest.mark.parametrize("seed,V", [(1, 3), (2, 4), (3, 2), (4, 5), (6, 8)])
def test_tie_inputs_on_the_gpu(cuda, reduce, seed, V):
    """The tie-heavy inputs of the CPU test (values in {-1, 0, 1}, all-zero columns, partly visible views) through the
    kernel, pixel indices given directly."""
    feats, pix, g = lgr.tie_inputs(seed, V=V)
    assert min(lgr.tie_cases(feats, pix).values()) > 0
    t = lambda a: torch.from_numpy(a).to(cuda)
    got = projection.lift_views_grad(t(feats), t(pix), t(g), reduce)
    want = lgr.lift_grad_ref(feats, pix, g, reduce)
    assert torch.equal(got.cpu().to(torch.float64), want)


def test_edge_shapes_write_the_whole_output(cuda):
    """N = 0 (zeros everywhere), C = 0, B = 0 and every element written over a NaN-filled buffer; more than 8 views is
    refused like the forward."""
    for B, N, V, C in ((2, 0, 3, 5), (2, 17, 3, 0), (0, 17, 3, 5), (2, 17, 3, 5), (1, 1, 1, 1)):
        feats, pix, g = lgr.tie_inputs(7, B=B, V=V, C=C, N=N) if B and N else (
            np.zeros((B, V, C, 4, 5), np.float32), np.zeros((B, V, N), np.int32), np.zeros((B, C, N), np.float32))
        for reduce, code in (("max", _lib.REDUCE_MAX), ("first", _lib.REDUCE_FIRST)):
            f, p, go = (torch.from_numpy(a).to(cuda) for a in (feats, pix, g))
            grad = torch.full((B, V, C, 4, 5), float("nan"), device=cuda)
            _lib.call("pn2_lift_views_grad", B, N, V, C, 4, 5, _lib.ptr(f), _lib.ptr(p), code, _lib.ptr(go), _lib.ptr(grad),
                      _lib.stream_ptr(cuda))
            assert torch.equal(grad.cpu().to(torch.float64), lgr.lift_grad_ref(feats, pix, g, reduce)), (B, N, V, C, reduce)
    f = torch.zeros((1, 9, 4, 4, 5), device=cuda)
    with pytest.raises(_lib.Pn2Error, match="at most 8 views"):
        projection.lift_views_grad(f, torch.zeros((1, 9, 6), dtype=torch.int32, device=cuda), torch.zeros((1, 4, 6), device=cuda))


@pytest.mark.parametrize("reduce", ["max", "first"])
def test_backward_is_deterministic_and_graph_replay_matches(cuda, reduce):
    """N(0,1) grad_out (sums that do depend on the order): two eager backwards give the same bits, and a CUDA-graph replay
    of forward + backward gives the eager bits."""
    B, N, V, C = 2, 8192, 3, 128
    xyz, feats, depth, poses = make_batch(B, N, V, C, 50)
    if reduce == "first":
        feats[:, 0, :, 5, :] = 0.0
    t = lambda a: torch.from_numpy(a).to(cuda)
    pts, dep, pos = t(xyz), t(depth), t(poses)
    f = t(feats).requires_grad_(True)
    g = torch.randn(B, C, N, device=cuda, generator=torch.Generator(device=cuda).manual_seed(4))

    def step():
        out = projection.lift_views(pts, f, dep, pos, INTR, DMIN, DMAX, DIMS, ACC, reduce=reduce)
        return out.detach(), torch.autograd.grad(out, f, g)[0]

    out1, g1 = step()
    out2, g2 = step()
    assert torch.equal(g1, g2) and torch.equal(out1, out2)
    side = torch.cuda.Stream(cuda)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out_s, g_s = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out_s, out1) and torch.equal(g_s, g1)
    assert g1.abs().sum() > 0


@pytest.mark.parametrize("reduce,launches", [("max", 2), ("first", 3)])
def test_forward_without_gradient_is_unchanged(cuda, reduce, launches):
    """No gradient needed (feats without requires_grad, or under no_grad): no grad_fn and the launches of the plain forward
    (projection + gather, plus the non-zero flags for "first"); with a gradient the output bits are the same."""
    xyz, feats, depth, poses = make_batch(2, 4096, 3, 128, 60)
    t = lambda a: torch.from_numpy(a).to(cuda)
    args = (t(xyz), t(feats), t(depth), t(poses), INTR, DMIN, DMAX, DIMS, ACC)
    projection.lift_views(*args, reduce=reduce)
    n0 = _lib.launch_count()
    out = projection.lift_views(*args, reduce=reduce)
    assert _lib.launch_count() - n0 == launches and out.grad_fn is None
    f = args[1].clone().requires_grad_(True)
    with torch.no_grad():
        n0 = _lib.launch_count()
        out_ng = projection.lift_views(args[0], f, *args[2:], reduce=reduce)
        assert _lib.launch_count() - n0 == launches and out_ng.grad_fn is None
    out_g = projection.lift_views(args[0], f, *args[2:], reduce=reduce)
    assert out_g.grad_fn is not None
    assert torch.equal(out, out_ng) and torch.equal(out, out_g.detach())


def _multiview_setup(cuda, B=2, N=2048, V=3, seed=61):
    pts = scenes.scannet_batch(seed, B, N)
    mv = [scenes.multiview_inputs(seed + b, pts[b, :, :3], V, 128) for b in range(B)]
    xyz = torch.from_numpy(pts[:, :, :3]).to(cuda).permute(0, 2, 1).contiguous()
    depth = torch.from_numpy(np.stack([m[1] for m in mv])).to(cuda)
    poses = torch.from_numpy(np.stack([m[2] for m in mv]).astype(np.float32)).to(cuda)
    H, W = depth.shape[-2:]
    maps = torch.randn(B, V, 128, H, W, device=cuda, generator=torch.Generator(device=cuda).manual_seed(seed))
    target = (torch.from_numpy(pts[:, :, 2]).to(cuda).clamp(0, 2.69) / 2.7 * 20).long() + 1
    return xyz, depth, poses, maps, target


def _point_branch(cls, cuda):
    torch.manual_seed(5)
    net = cls(21).to(cuda).train()
    for m in net.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
    return net


def _loss(logits, tgt):
    return F.cross_entropy(logits.reshape(-1, 21), tgt.reshape(-1), ignore_index=0)


@pytest.mark.parametrize("model", ["PointNet2Multiview2", "PointNet2Multiview2Msg"])
def test_end_to_end_gradient_of_a_trainable_2d_layer(cuda, model):
    """A trainable 1x1 Conv2d (stand-in for the reference's enet_trainable) -> lift_views -> point branch in train mode ->
    cross-entropy: the conv's gradients equal those of the same step built from Projection.apply per scene and view plus
    the reference's reduction (same pixel indices), within 1e-5 of the largest."""
    from pn2_b200 import models
    from pn2_b200 import pointnet2_utils as pu
    xyz, depth, poses, maps, target = _multiview_setup(cuda)
    B, V = maps.shape[:2]
    net = _point_branch(getattr(models, model), cuda)
    conv = torch.nn.Conv2d(128, 128, 1).to(cuda)
    points = xyz.permute(0, 2, 1).contiguous()
    prev = pu.set_deterministic(True)
    try:
        f = conv(maps.reshape(B * V, *maps.shape[2:])).reshape(maps.shape)
        img, pix, _ = projection.lift_views(points, f, depth, poses, INTR, DMIN, DMAX, DIMS, ACC, reduce=net.reduce,
                                            return_pixels=True)
        gw, gb = torch.autograd.grad(_loss(net(xyz, img), target), [conv.weight, conv.bias])
        f = conv(maps.reshape(B * V, *maps.shape[2:])).reshape(maps.shape)
        img_ref = lgr.composition_forward(f, pix, net.reduce)
        rw, rb = torch.autograd.grad(_loss(net(xyz, img_ref), target), [conv.weight, conv.bias])
    finally:
        pu.set_deterministic(prev)
    assert torch.equal(img.detach(), img_ref.detach())
    assert (pix >= 0).float().mean() > 0.05
    for got, ref in ((gw, rw), (gb, rb)):
        assert ref.abs().max() > 0
        assert (got - ref).abs().max() <= 1e-5 * ref.abs().max(), ((got - ref).abs().max().item(), ref.abs().max().item())


class _LiftAndPoints(torch.nn.Module):
    """2-D layer -> lift_views (depth and poses held as buffers) -> point branch: a multi-view training net whose inputs
    are (xyz, feature maps), the form GraphedTrainStep replays."""

    def __init__(self, point, depth, poses):
        super().__init__()
        self.conv = torch.nn.Conv2d(128, 128, 1)
        self.point = point
        self.register_buffer("depth", depth.clone())
        self.register_buffer("poses", poses.clone())

    def forward(self, xyz, maps):
        B, V = maps.shape[:2]
        f = self.conv(maps.reshape(B * V, *maps.shape[2:])).reshape(maps.shape)
        img = projection.lift_views(xyz.permute(0, 2, 1).contiguous(), f, self.depth, self.poses, INTR, DMIN, DMAX, DIMS, ACC,
                                    reduce=self.point.reduce)
        return self.point(xyz, img)


@pytest.mark.parametrize("model", ["PointNet2Multiview2", "PointNet2Multiview2Msg"])
def test_graphed_train_step_through_the_lifting_reproduces_the_eager_loop(cuda, model):
    """GraphedTrainStep over conv -> lift_views -> point branch against the eager loop from the same initial weights,
    deterministic mode: identical losses and weights over 3 steps (the conv does get trained)."""
    from pn2_b200 import models
    from pn2_b200 import pointnet2_utils as pu
    from pn2_b200.models import GraphedTrainStep
    xyz, depth, poses, maps, target = _multiview_setup(cuda, seed=71)

    def make():
        net = _LiftAndPoints(_point_branch(getattr(models, model), cuda), depth, poses).to(cuda).train()
        return net, torch.optim.Adam(net.parameters(), lr=1e-3, capturable=True)

    prev = pu.set_deterministic(True)
    try:
        net_e, opt_e = make()
        w0 = net_e.conv.weight.detach().clone()
        eager = []
        for _ in range(3):
            opt_e.zero_grad(set_to_none=True)
            loss = _loss(net_e(xyz, maps), target)
            loss.backward()
            opt_e.step()
            eager.append(float(loss.detach()))
        net_g, opt_g = make()
        stepper = GraphedTrainStep(net_g, opt_g, _loss, xyz, maps, target)
        graphed = [float(stepper.step(xyz, maps, target)) for _ in range(3)]
    finally:
        pu.set_deterministic(prev)
    assert graphed == eager, (graphed, eager)
    assert not torch.equal(net_e.conv.weight.detach(), w0)
    for (k, a), (_, b) in zip(net_e.state_dict().items(), net_g.state_dict().items()):
        assert torch.equal(a, b), k
