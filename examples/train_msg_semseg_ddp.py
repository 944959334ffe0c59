"""BASELINE config 2: MSG semseg TRAIN step, 8192 points, scenes sharded across GPUs (one process per GPU, DDP).

    torchrun --nproc-per-node N examples/train_msg_semseg_ddp.py --steps 20 --batch-per-gpu 4
    python examples/train_msg_semseg_ddp.py --rooms 16 --model ssg [--graph]

The point branch of PointNet2Multiview2Msg (the reference's only MSG semseg stack, model/pointnet2multiview.py:179-233)
is trained on synthetic ScanNet-shaped scenes with synthetic lifted image features, with the loss / optimiser of
train_scannet_semseg.py:89-95,135-140 (weighted cross-entropy with ignore_index 0, Adam lr 1e-3, weight decay 1e-4).
Geometry (FPS, ball query, grouping, 3-NN, interpolation and their backward scatter-adds) runs on the B200 kernels;
conv / BatchNorm(train) / autograd are torch, as in the reference.  The ONLY collective is DDP's gradient all-reduce
(NCCL); the forward path has none.  BatchNorm statistics stay per rank, as with the reference's DataParallel replicas.

With --rooms K the batches are the training loader's crops instead (data_utils/ScanNetDataLoader.py:394-418): K synthetic
whole rooms, split round-robin over the ranks, are held on the GPU in a pn2_b200.whole_scene.SceneBank; each step takes
the next B room ids of a per-epoch host shuffle and draws their random 1.5 m columns on the device (bank.crops), with
the loader's class weights in the loss.
"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "multi-modal-learning-on-3d-point-clouds_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from pn2_b200 import scenes, sharding, whole_scene  # noqa: E402
from pn2_b200.models import PointNet2Multiview2Msg, PointNet2SemSeg  # noqa: E402


def room_bank(k, rank, world, device):
    """The rooms rank, rank + world, ... < k in a SceneBank, and the loader's class weights of that split."""
    rooms = [scenes.scannet_room(r, 60000 + 10000 * (r % 10), 4.0 + 0.3 * (r % 10)) for r in sharding.scene_ids_for_rank(k, rank, world)]
    if not rooms:
        raise SystemExit("--rooms %d leaves rank %d without a room" % (k, rank))
    cat = [torch.from_numpy(np.concatenate([r[i] for r in rooms])).to(device) for i in range(3)]
    offsets = torch.tensor(np.concatenate([[0], np.cumsum([len(r[0]) for r in rooms])]), dtype=torch.int64, device=device)
    bank = whole_scene.SceneBank(cat[0], cat[1], cat[2], offsets)
    return bank, bank.label_weights(21)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--batch-per-gpu", type=int, default=4)
    ap.add_argument("--npoints", type=int, default=8192)
    ap.add_argument("--model", default="msg", choices=["msg", "ssg"])
    ap.add_argument("--deterministic", action="store_true",
                    help="bit-reproducible training: fixed-order backwards of gather / grouping / interpolation "
                         "(pn2_scatter_rows_det) and torch's deterministic algorithms")
    ap.add_argument("--graph", action="store_true",
                    help="replay the step as CUDA graphs (pn2_b200.models.GraphedTrainStep): zero-grad + forward + backward in one "
                         "graph, one all-reduce of the flat gradient buffer, the Adam update in a second graph")
    ap.add_argument("--rooms", type=int, default=0,
                    help="train on device-drawn crops of K synthetic whole rooms (pn2_b200.whole_scene.SceneBank), the rooms "
                         "split round-robin over the ranks; 0 (default) keeps the fixed synthetic batches")
    args = ap.parse_args()
    if args.deterministic:
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
        torch.use_deterministic_algorithms(True, warn_only=True)  # pn2_b200.pointnet2_utils follows this switch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    torch.manual_seed(0)
    net = (PointNet2Multiview2Msg(21) if args.model == "msg" else PointNet2SemSeg(21)).to(device).train()
    model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[local]) if world > 1 and not args.graph else net
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4, capturable=args.graph)
    stepper = None
    B, N = args.batch_per_gpu, args.npoints
    g = torch.Generator(device="cpu").manual_seed(1234 + rank)
    if args.rooms:
        bank, labelweights = room_bank(args.rooms, rank, world, device)
        ids_dev = torch.empty(B, dtype=torch.int32, device=device)
        order = []  # room ids still to visit in this epoch
        wbuf = torch.empty(B, N, device=device)  # the graphed loss reads the weights from here
    losses, t_steps = [], []
    for step in range(args.steps):
        if args.rooms:
            while len(order) < B:
                order += torch.randperm(bank.num_scenes, generator=g).tolist()
            ids_dev.copy_(torch.tensor(order[:B], dtype=torch.int32))
            order = order[B:]
            crops = bank.crops(ids_dev, labelweights, N, seed=rank)
            pts, target, weights = crops.points, crops.target, crops.weights
        else:
            ids = sharding.weak_scene_ids(rank, B, step % 4)  # a few fixed batches so the loss can go down
            pts = torch.from_numpy(scenes.scannet_batch(ids[0], B, N)).to(device)
            # labels derived from the geometry so that they are learnable: height band (1..20); 0 = unannotated
            target = (pts[:, :, 2].clamp(0, 2.69) / 2.7 * 20).long() + 1
            target[torch.rand(target.shape, generator=g).to(device) < 0.05] = 0
            weights = torch.ones_like(target, dtype=torch.float32)
        xyz = pts[:, :, :3].permute(0, 2, 1).contiguous()
        second = (torch.randn(B, 128, N, generator=g).to(device) if args.model == "msg"
                  else pts[:, :, 3:].permute(0, 2, 1).contiguous())
        if args.graph and stepper is None:
            from pn2_b200.models import GraphedTrainStep

            if args.rooms:
                def loss_fn(pred, tgt):
                    loss = F.cross_entropy(pred.reshape(-1, 21), tgt.reshape(-1), ignore_index=0, reduction="none")
                    return (loss * wbuf.reshape(-1)).mean()
                wbuf.copy_(weights)
            else:
                def loss_fn(pred, tgt):
                    return F.cross_entropy(pred.reshape(-1, 21), tgt.reshape(-1), ignore_index=0)
            stepper = GraphedTrainStep(net, opt, loss_fn, xyz, second, target)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if stepper is not None:
            if args.rooms:
                wbuf.copy_(weights)
            loss = stepper.step(xyz, second, target)                     # graphs + one flat all-reduce
        else:
            opt.zero_grad(set_to_none=True)
            pred = model(xyz, second)                                    # (B, N, 21)
            loss = F.cross_entropy(pred.reshape(-1, 21), target.reshape(-1), ignore_index=0, reduction="none")
            loss = (loss * weights.reshape(-1)).mean()
            loss.backward()                                              # DDP all-reduces the gradients here
            opt.step()
        torch.cuda.synchronize()
        t_steps.append(time.perf_counter() - t0)
        losses.append(float(loss.detach()))
    t = torch.tensor([sum(t_steps[2:]) / max(len(t_steps) - 2, 1)], dtype=torch.float64, device=device)
    sharding.max_over_ranks(t)
    if rank == 0:
        print("model=%s world=%d batch/gpu=%d npoints=%d  step %.1f ms  -> %.1f scenes/s   loss %.4f -> %.9f%s" % (
            args.model, world, B, N, float(t) * 1e3, world * B / float(t), losses[0], losses[-1],
            "  (deterministic)" if args.deterministic else ""))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
