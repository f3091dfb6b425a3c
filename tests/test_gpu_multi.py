"""Data-parallel CORRECTNESS on real GPUs (SURVEY.md section 8(e)): needs >= 2 devices (`gpurun --gpus 2`); skipped on a
one-GPU box.  One process per GPU over NCCL, like bench.py under torchrun.

  * the all-reduced gradient of N ranks on their shards == the one-GPU gradient on the concatenated batch
    (DDP's mean, base_model.py:725-737) up to fp32 summation order;
  * after 3 optimizer steps the replicas hold bit-identical parameters, Adam moments and EMA;
  * CUDA-graph replay with the overlapped bucketed all-reduce gives the same parameters as the eager path.
"""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


CFG = dict(image_size=32, inner_channel=32, channel_mults=(1, 2), res_blocks=(1, 1), attn_res=(2,), num_head_channels=16)
BATCH = 4


def _draws(O, cfg, seed):
    data = O.synthetic_batch(BATCH, cfg.image_size, seed)
    torch.manual_seed(seed + 7)
    t, u = O.sample_t_gamma(cfg, BATCH)
    noise = torch.randn_like(data["gt"])
    return data, noise, t, u


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    solo_groups = [dist.new_group([r]) for r in range(world)]
    from joligen_b200 import nets
    from joligen_b200.trainer import PaletteTrainer
    from oracle import palette_oracle as O
    cfg = O.UNetCfg(**CFG)

    def trainer(seed, pg=None, graph=False):
        net = nets.build_palette_generator(**CFG)
        net.load_state_dict(O.init_params(cfg, seed), strict=False)
        return PaletteTrainer(net, lr=1e-3, optim="adamw", ema=True, ema_beta=0.9, device="cuda:%d" % rank,
                              process_group=pg, cuda_graph=graph, graph_warmup=1, comm_min_bucket=1 << 16)

    def feed(tr, parts):
        cat = lambda xs: torch.cat(xs, dim=0)  # noqa: E731
        tr.set_input({"A": cat([p[0]["cond"] for p in parts]), "B": cat([p[0]["gt"] for p in parts]),
                      "B_label_mask": cat([p[0]["mask"] for p in parts])})
        return dict(noise=cat([p[1] for p in parts]).cuda(), t=cat([p[2] for p in parts]).cuda(),
                    u=cat([p[3] for p in parts]).cuda())

    res = {}
    # different initial weights per rank: broadcast_parameters must make them rank 0's
    tr = trainer(50 + rank)
    tr.broadcast_parameters()
    # ---- gradient of the global batch
    shards = [_draws(O, cfg, 1000 + r) for r in range(world)]
    g_dp = tr.reduced_gradient(**feed(tr, [shards[rank]])).clone() / world
    if rank == 0:
        solo = trainer(50, pg=solo_groups[0])
        g_one = solo.reduced_gradient(**feed(solo, shards)).clone()
        g_two = solo.reduced_gradient(**feed(solo, shards)).clone()   # the same evaluation again: run-to-run floor
        res["grad_rel"] = _rel_l2(g_dp.cpu(), g_one.cpu())
        res["grad_floor"] = _rel_l2(g_two.cpu(), g_one.cpu())
        res["grad_norm"] = float(g_one.norm())
    # ---- the exchange itself, exactly: known per-rank values through the bucket machinery (unpack / fold / one
    # all-reduce per bucket on the communication stream / wait) must come back as their sum over the ranks, bit for bit
    known = torch.arange(tr.flat.total, device="cuda", dtype=torch.float32).remainder_(1013.0) * (rank + 1)
    tr.flat.rebind_grads()
    tr.flat.grad.copy_(known)
    tr.buckets.begin()
    for i in reversed(range(len(tr.flat.params))):
        tr.buckets.ready(i)
    tr.buckets.finish()
    tr.comm.wait()
    torch.cuda.synchronize()
    want = torch.arange(tr.flat.total, device="cuda", dtype=torch.float32).remainder_(1013.0) * sum(
        r + 1 for r in range(world))
    res["exchange_exact"] = bool(torch.equal(tr.flat.grad, want))
    res["buckets"] = len(tr.buckets.buckets)
    tr.flat.grad.zero_()
    # ---- three optimizer steps, eager
    for step in range(3):
        tr.optimize_parameters(**feed(tr, [_draws(O, cfg, 2000 + 10 * step + rank)]))
    torch.cuda.synchronize()
    res["params"] = tr.flat.data.cpu()
    res["exp_avg"] = tr.exp_avg.cpu()
    res["ema"] = tr.ema.cpu()
    # ---- the same three steps through CUDA-graph replay (implicit draws: only the plumbing is compared)
    trg = trainer(50, graph=True)
    tre = trainer(50, graph=False)
    for t_ in (trg, tre):
        t_.broadcast_parameters()
    data = _draws(O, cfg, 3000 + rank)[0]
    batch = {"A": data["cond"], "B": data["gt"], "B_label_mask": data["mask"]}
    for step in range(4):
        for t_ in (trg, tre):
            torch.manual_seed(4000 + step)
            torch.cuda.manual_seed(4000 + step)
            t_.set_input(batch)
            t_.optimize_parameters()
    torch.cuda.synchronize()
    res["graph_params"] = trg.flat.data.cpu()
    res["graph_used"] = trg._graph_fb is not None
    res["finite"] = bool(torch.isfinite(trg.flat.data).all()) and bool(torch.isfinite(tre.flat.data).all())
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_gradient_and_replicas():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    a, b = out[0], out[1]
    assert a["grad_norm"] > 0
    assert a["exchange_exact"] and b["exchange_exact"] and a["buckets"] > 1
    # N-rank mean gradient == 1-rank gradient on the concatenated batch.  Not bit for bit: split-K / statistics atomics
    # reorder fp32 sums, a flipped bf16 ulp is then amplified by the (chaotic, random-init) net — the bound is the
    # run-to-run difference of the SAME one-GPU evaluation, measured here
    assert a["grad_rel"] < max(2e-3, 3.0 * a["grad_floor"]), (a["grad_rel"], a["grad_floor"])
    for k in ("params", "exp_avg", "ema", "graph_params"):
        assert torch.equal(a[k], b[k]), "replicas differ in %s" % k
    assert a["graph_used"] and b["graph_used"] and a["finite"] and b["finite"]


# ---------------------------------------------------------------------------------------------------------------------
# The drop-in path of INTEGRATION.md section 2: the B200 modules inside torch's DistributedDataParallel (what
# BaseModel.parallelize builds, base_model.py:725-737) with gradient accumulation (train_iter_size = 2: the first
# micro-step under no_sync, base_model.py:1313-1315).  Two ranks share ONE GPU over gloo, so it runs on the one-GPU box.
# What it pins (ADVICE r1): every parameter's gradient reaches autograd's AccumulateGrad — so DDP's reducer hooks fire for
# the convolution weights too, on the first AND the second micro-step (when .grad already exists).
# ---------------------------------------------------------------------------------------------------------------------
def _ddp_worker(rank, world, port, out):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from joligen_b200 import nets
    from oracle import palette_oracle as O
    cfg = O.UNetCfg(**CFG)

    def make():
        net = nets.build_palette_generator(**CFG)
        net.load_state_dict(O.init_params(cfg, 50), strict=False)
        return net.cuda()

    def loss_of(model, draw):
        data, noise, t, u = draw
        _, noise_hat, _ = model(data["gt"].cuda(), data["cond"].cuda(), data["mask"].cuda(), noise.cuda(),
                                t=t.cuda(), u=u.cuda())
        return torch.nn.functional.mse_loss(noise_hat, noise.cuda())

    draws = {(r, m): _draws(O, cfg, 5000 + 10 * r + m) for r in range(world) for m in range(2)}
    ddp = DDP(make(), device_ids=[0])
    with ddp.no_sync():
        (loss_of(ddp, draws[(rank, 0)]) / 2).backward()
    (loss_of(ddp, draws[(rank, 1)]) / 2).backward()   # .grad exists now: must still go through AccumulateGrad
    torch.cuda.synchronize()
    got = {k: p.grad.detach().float().cpu() for k, p in ddp.module.named_parameters() if p.grad is not None}
    res = {"n_grads": len(got), "n_params": sum(1 for _ in ddp.module.parameters())}
    if rank == 0:
        solo = make()
        for r in range(world):
            for m in range(2):
                (loss_of(solo, draws[(r, m)]) / (2 * world)).backward()
        torch.cuda.synchronize()
        worst, worst_k = 0.0, None
        for k, p in solo.named_parameters():
            ref = p.grad.detach().float().cpu()
            e = float((got[k].double() - ref.double()).norm() / (ref.double().norm() + 1e-12))
            if e > worst and float(ref.norm()) > 1e-6:
                worst, worst_k = e, k
        res["worst"], res["worst_k"] = worst, worst_k
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_ddp_wrapped_modules_with_gradient_accumulation():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_ddp_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    a, b = out[0], out[1]
    assert a["n_grads"] == a["n_params"] == b["n_grads"]
    # DDP's mean over ranks of the accumulated micro-step gradients == the plain sum / (2 * world) on one model; a
    # parameter whose gradient skipped the reducer would hold its rank-local value (different data: error ~ 1)
    assert a["worst"] < 5e-2, (a["worst_k"], a["worst"])
