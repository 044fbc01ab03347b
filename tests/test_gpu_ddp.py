"""Multi-rank GPU parity of the data-parallel training step (BASELINE.json configs[4]; SURVEY.md 8d "config 5"):
N ranks through NCCL, each on its shard of the batch, end with the gradients of the single-rank run on the concatenated
batch (per-sample InstanceNorm; every loss is a mean over equal-sized shards, so averaging the shard gradients commutes).
Needs >= 2 GPUs in the machine; skipped on a single-GPU machine."""
import os
import socket
import tempfile

import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _make(precision, impl, seeds=(111, 112)):
    import nirgan_oracle as O
    from nirgan_b200.config import px2px_config
    from nirgan_b200.model.pix2pix import Px2Px
    model = Px2Px(px2px_config())
    model.netG.load_state_dict(O.random_state_dict(O.generator_param_shapes(), seed=seeds[0]))
    model.netD.load_state_dict(O.random_state_dict(O.discriminator_param_shapes(), seed=seeds[1]))
    model = model.cuda().train()
    model.netG.configure_b200(precision=precision, impl=impl)
    model.netD.configure_b200(precision=precision, impl=impl)
    return model


def _batches(total, size):
    g = torch.Generator().manual_seed(21)
    return torch.rand(total, 3, size, size, generator=g), torch.rand(total, 1, size, size, generator=g)


def _worker(rank, world, port, precision, impl, size, out_dir):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "oracle"), os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    import nirgan_b200  # noqa: F401
    from nirgan_b200.trainer import Trainer
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    model = _make(precision, impl)
    tr = Trainer(model)
    rgb, nir = _batches(2 * world, size)
    sl = slice(2 * rank, 2 * rank + 2)
    batch = {"rgb": rgb[sl].cuda(), "nir": nir[sl].cuda()}
    # the gradients that entered the optimizers: arena contents (sums over ranks) times 1/world
    grads = {}
    ld = tr._pass(batch, 0, model.netD, tr.opt_d, "d")
    grads["d"] = {k: (p.grad / world).cpu() for k, p in model.netD.named_parameters()}
    lg = tr._pass(batch, 1, model.netG, tr.opt_g, "g")
    grads["g"] = {k: (p.grad / world).cpu() for k, p in model.netG.named_parameters()}
    # configs[4] mixes resolutions from step to step: two more steps at other tile sizes (each shape has its own plans,
    # all of them carved from the shared buffer pool) through the public step()
    for s2 in (96, size):
        rgb2, nir2 = _batches(2 * world, s2)
        tr.step({"rgb": rgb2[sl].cuda(), "nir": nir2[sl].cuda()})
    torch.cuda.synchronize()
    weights = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    torch.save({"grads": grads, "weights": weights, "loss": (float(ld), float(lg)),
                "buckets": {k: r.last_buckets for k, r in tr.reducers.items()}},
               os.path.join(out_dir, f"rank{rank}.pt"))
    dist.destroy_process_group()


@pytest.mark.parametrize("precision,impl,tol", [("fp32", "simt", 2e-3), ("fp16", "tc", 3e-2)], ids=["fp32-verify", "fp16-tc"])
def test_two_rank_nccl_step_equals_single_rank_on_concatenated_batch(precision, impl, tol):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    world, size = 2, 64
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_worker, args=(world, _free_port(), precision, impl, size, d), nprocs=world, join=True)
        ranks = [torch.load(os.path.join(d, f"rank{r}.pt")) for r in range(world)]
    # single rank, concatenated batch
    torch.cuda.set_device(0)
    from nirgan_b200.trainer import Trainer
    model = _make(precision, impl)
    tr = Trainer(model)
    rgb, nir = _batches(2 * world, size)
    batch = {"rgb": rgb.cuda(), "nir": nir.cuda()}
    tr._pass(batch, 0, model.netD, tr.opt_d, "d")
    full = {"d": {k: p.grad.cpu() for k, p in model.netD.named_parameters()}}
    tr._pass(batch, 1, model.netG, tr.opt_g, "g")
    full["g"] = {k: p.grad.cpu() for k, p in model.netG.named_parameters()}

    def rel(a, b):
        return float((a - b).norm() / (b.norm() + 1e-20))

    # every rank holds the same averaged gradients and the same updated weights (DDP invariant)
    for net in ("d", "g"):
        for k in ranks[0]["grads"][net]:
            assert torch.equal(ranks[0]["grads"][net][k], ranks[1]["grads"][net][k]), (net, k)
    for k in ranks[0]["weights"]:       # after three steps at mixed resolutions (64, 96, 64 px)
        assert torch.equal(ranks[0]["weights"][k], ranks[1]["weights"][k]), k
    # ... and they are the single-rank gradients of the concatenated batch.  (D pass exactly so; in the G pass each rank's D
    # has already taken its -- identical -- optimizer step, as in the single-rank run.)
    worst = 0.0
    for net in ("d", "g"):
        for k, g in full[net].items():
            if k.endswith("weight"):
                r = rel(ranks[0]["grads"][net][k], g)
                worst = max(worst, r)
                assert r <= tol, (net, k, r)
    print(f"2-rank NCCL vs 1-rank concatenated batch ({precision}/{impl}): worst rel-L2 {worst:.3e}, "
          f"buckets per pass {ranks[0]['buckets']}")
    assert ranks[0]["buckets"]["g"] >= 1 and ranks[0]["buckets"]["d"] >= 1
