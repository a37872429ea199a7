"""CPU, world_size 2 over gloo: the data-parallel gradient sync (bucketed all-reduce of the flat gradient buffer)
produces the MEAN of the per-shard gradients, which is what DistributedDataParallel gives the reference
(train.py:346; SURVEY.md Appendix B)."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import unet_pytorch_b200 as b2u
        from unet_pytorch_b200.trainer import FlatBuckets, GradientSync, _backward_order
        shapes = {k: v for k, v in b2u.vgg_unet_param_shapes(2).items()}
        order = _backward_order(list(shapes))
        lay = FlatBuckets(shapes, order, torch.device("cpu"), bucket_bytes=4 << 20)
        flat = lay.new_buffer()
        g = torch.Generator().manual_seed(100 + rank)
        flat.copy_(torch.randn(lay.total, generator=g))
        mine = flat.clone()
        sync = GradientSync(lay, flat)
        assert sync.enabled and sync.world == world
        sync.reset()
        # gradients become ready in backward order, two names (weight, bias) at a time like the engine reports them
        for i in range(0, len(order), 2):
            sync.ready(order[i:i + 2])
        scale = sync.finish()
        assert all(p == 0 for p in sync._pending)
        flat.mul_(scale)
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        expect = sum(gathered) / world
        torch.testing.assert_close(flat, expect, rtol=0, atol=1e-6)
        # frozen backbone: only decoder + head names are reported; encoder buckets must not fire or hang
        flat.copy_(mine)
        active = [n for n in order if not n.startswith("vgg.")]
        sync.reset(active)
        for i in range(0, len(active), 2):
            sync.ready(active[i:i + 2])
        sync.finish()
        if rank == 0:
            out.put("ok")
    finally:
        dist.destroy_process_group()


def test_gradient_sync_is_mean_of_shards():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    assert q.get(timeout=5) == "ok"


def _ddp_reference_worker(rank, world, port, out):
    """The reference model under DistributedDataParallel (gloo, CPU) exactly as train.py:346 wraps it, next to this package's
    GradientSync fed with the same per-shard gradients: both must produce the mean of the shard gradients.  The reference
    model and losses are the oracle's restatement (nets/unet.py::Unet, CE_Loss, Dice_loss), which tests/test_oracle.py pins
    to the reference's own outputs stored under tests/golden/."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import sys
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        if root not in sys.path:
            sys.path.insert(0, root)
        from oracle import unet_oracle as O
        from unet_pytorch_b200.trainer import FlatBuckets, GradientSync, _backward_order

        class RefUnet(torch.nn.Module):
            def __init__(self, params):
                super().__init__()
                self.names = list(params)
                self.weights = torch.nn.ParameterList(torch.nn.Parameter(v.clone()) for v in params.values())

            def forward(self, x):
                return O.unet_forward(dict(zip(self.names, self.weights)), x)

        C = 3
        params = O.make_params(C, seed=11)
        model = RefUnet(params)
        ddp = torch.nn.parallel.DistributedDataParallel(model, find_unused_parameters=True)      # train.py:346
        imgs, pngs = O.make_inputs(4, C, 32, 32, seed=21)
        n = imgs.shape[0] // world
        xs, ys = imgs[rank * n:(rank + 1) * n], pngs[rank * n:(rank + 1) * n]      # DistributedSampler shard (train.py:425-427)
        w = torch.ones(C)
        out_logits = ddp(xs)
        loss = O.ce_loss(out_logits, ys, w, C) + O.dice_loss(out_logits, O.one_hot(ys, C))
        loss.backward()
        ddp_grads = {k: p.grad.detach().clone() for k, p in zip(model.names, model.weights)}
        # oracle gradient of THIS shard alone (each rank normalises CE / Dice over its own shard, utils_fit.py:70-81)
        _, _, shard = O.train_step(params, xs, ys, w, C, dice=True)
        shapes = {k: tuple(v.shape) for k, v in params.items()}
        order = _backward_order(list(shapes))
        lay = FlatBuckets(shapes, order, torch.device("cpu"), bucket_bytes=1 << 20)
        flat = lay.new_buffer()
        views = lay.views(flat)
        for k in shapes:
            views[k].copy_(shard[k])
        sync = GradientSync(lay, flat)
        sync.reset()
        for i in range(0, len(order), 2):
            sync.ready(order[i:i + 2])
        flat.mul_(sync.finish())
        worst = max((views[k] - ddp_grads[k]).abs().max().item() / (ddp_grads[k].abs().max().item() + 1e-12) for k in shapes)
        out.put((rank, worst))
    finally:
        dist.destroy_process_group()


def test_reference_under_ddp_equals_bucketed_mean_of_shards():
    """Runs the oracle's restatement of the reference Unet-VGG16 (not the reference module itself) under gloo-DDP: its
    averaged gradients must equal GradientSync's bucketed mean of the per-shard oracle gradients."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_ddp_reference_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    got = dict(q.get(timeout=5) for _ in range(2))
    assert max(got.values()) <= 1e-4, got          # the reference's DDP gradients == bucketed mean of the per-shard oracle gradients
