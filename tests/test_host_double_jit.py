"""The b2b video backbone (BASELINE.json config 5 as written: b2b_model + vit_vid) on the CPU through the kernel TEST
DOUBLE: nets_jit.B2BGenerator / JiTViD and trainer_b2b.B2BTrainer vs the golden vectors of the unmodified reference —
the comparisons of tests/test_gpu_jit.py.  See tests/test_host_double.py for what a pass proves."""
import os
import socket
from unittest import mock

import pytest
import torch

import kernel_double as KD

from oracle import ref_stubs  # noqa: E402

REF_MISSING = "needs the reference's own code: build() stages it under oracle/_ref where the checkout is readable"


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _small_net(golden_dir):
    from joligen_b200 import nets_jit
    from oracle import jit_oracle as J
    from oracle.vid_oracle import init_params_from_shapes
    gold = torch.load(os.path.join(golden_dir, "jit_b200.pt"))
    cfg = J.JitCfg(**gold["cfg"])
    net = nets_jit.B2BGenerator(nets_jit.JiTViD(
        input_size=cfg.input_size, patch_size=cfg.patch_size, in_channels=cfg.in_channels, out_channels=cfg.out_channels,
        hidden_size=cfg.hidden_size, depth=cfg.depth, num_heads=cfg.num_heads, num_classes=cfg.num_classes,
        in_context_len=cfg.in_context_len, in_context_start=cfg.in_context_start, max_frames=cfg.max_frames,
        motion_num_heads=cfg.motion_num_heads, motion_num_layers=cfg.motion_num_layers), t_eps=cfg.t_eps,
        noise_scale=cfg.noise_scale)
    mine = {k: tuple(v.shape) for k, v in net.named_parameters() if v.requires_grad}
    assert mine == dict(gold["shapes"]), set(mine) ^ set(dict(gold["shapes"]))
    missing, unexpected = net.load_state_dict({**init_params_from_shapes(gold["shapes"], gold["wseed"]),
                                               **gold["frozen"]}, strict=False)
    assert not unexpected and all(m.endswith("pos_encoder.pe") for m in missing), (missing, unexpected)
    return gold, cfg, net


def test_b2b_generator_and_sampler_on_the_double(golden_dir):
    from oracle.gen_golden_jit import inputs
    gold, cfg, net = _small_net(golden_dir)
    gt, cond, mask, label = inputs(cfg, gold["batch"], gold["frames"], gold["dseed"])
    torch.manual_seed(gold["rseed"])
    t_base = torch.sigmoid(torch.randn(gold["batch"]) * 0.8 - 0.8)
    e = torch.randn_like(gt)
    m = mask.bool().expand_as(gt)
    with KD.installed():
        v_pred, v, x_pred = net(gt, mask, cond, label, return_x_pred=True, t_base=t_base, e=e)
        assert rel(x_pred, gold["x_pred"]) < 3e-2
        assert torch.equal(x_pred[~m], gt[~m])
        loss = net.masked_region_loss(v_pred, v, torch.clamp(mask, 0, 1))
        assert abs(float(loss.detach()) - gold["loss"]) < 3e-2 * gold["loss"]
        loss.backward()
        torch.manual_seed(gold["rseed"] + 1)
        init_noise = torch.randn_like(gt)
        with torch.no_grad():
            out = net.restoration(gt, cond, gold["denoise_timesteps"], mask=mask, labels=label, init_noise=init_noise)
    scale = max(g["l2"] for g in gold["grads"].values())
    named = dict(net.named_parameters())
    bad = {}
    for k, g in gold["grads"].items():
        got = named[k].grad
        assert got is not None, k
        tol = 6e-2 * max(g["l2"], 2e-2 * scale)
        if abs(float(got.double().norm()) - g["l2"]) > tol or float((got.flatten()[:16] - g["head"]).abs().max()) > tol:
            bad[k] = (float(got.double().norm()), g["l2"])
    assert not bad, bad
    assert torch.equal(out[~m], gt[~m].clamp(-1, 1))
    assert rel(out, gold["restored"]) < 3e-2


def _b2b_trainer(net, **kw):
    from joligen_b200.trainer_b2b import B2BTrainer
    with mock.patch("torch.cuda.is_available", return_value=True):
        return B2BTrainer(net, device="cpu", **kw)


def _dp_worker(rank, world, port, golden_dir, out):
    import torch.distributed as dist
    from oracle.gen_golden_jit import inputs
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(2)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    solo_groups = [dist.new_group([r]) for r in range(world)]
    gold, cfg, net = _small_net(golden_dir)

    def draw(seed):
        gt, cond, mask, label = inputs(cfg, gold["batch"], gold["frames"], seed)
        torch.manual_seed(seed)
        return ({"A": cond, "B": gt, "B_label_mask": mask}, torch.sigmoid(torch.randn(gold["batch"]) * 0.8 - 0.8),
                torch.randn_like(gt))

    with KD.installed():
        tr = _b2b_trainer(net, lr=1e-3, ema_beta=0.9, use_cond=True, process_group=dist.group.WORLD)
        if rank == 1:
            tr.flat.data.mul_(1.01)       # a replica that starts elsewhere ...
        tr.broadcast_parameters()         # ... is overwritten by rank 0's weights
        p0 = tr.flat.data.clone()
        losses = []
        step_grads = []
        orig = tr.comm.allreduce_async

        def spy(t):
            orig(t)
            tr.comm.wait()
            step_grads.append(t.clone())
        tr.comm.allreduce_async = spy
        for s in range(2):
            data, t_base, e = draw(900 + 10 * s + rank)
            tr.set_input(data)
            losses.append(float(tr.optimize_parameters(t_base=t_base, e=e)))
        res = {"params": tr.flat.data.clone(), "ema": tr.ema.clone(), "losses": losses, "p0": p0,
               "sum_grad0": step_grads[0]}
        if rank == 0:
            # one process on the concatenated batch of step 0 must take the same first step
            _, _, net1 = _small_net(golden_dir)
            solo = _b2b_trainer(net1, lr=1e-3, ema_beta=0.9, use_cond=True, process_group=solo_groups[0])
            parts = [draw(900 + r) for r in range(world)]
            solo.set_input({k: torch.cat([p[0][k] for p in parts]) for k in parts[0][0]})
            solo.net.zero_grad()
            solo.flat.rebind_grads()
            loss = solo.net.forward_loss(solo.gt, solo.mask, solo.cond, solo.label, t_base=torch.cat([p[1] for p in parts]),
                                         e=torch.cat([p[2] for p in parts]), lambda_G=1.0)
            loss.backward()
            res["solo_grad"] = solo.flat.grad.clone()
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_b2b_trainer_two_ranks_over_gloo(golden_dir):
    """B2BTrainer(process_group=...): the flat gradient is summed over the ranks before the fused AdamW, 1/world folded
    into the optimizer — replicas stay bit-identical."""
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_dp_worker, args=(2, port, golden_dir, out), nprocs=2, join=True)
    a, b = out[0], out[1]
    assert torch.equal(a["p0"], b["p0"])
    assert torch.equal(a["params"], b["params"]) and torch.equal(a["ema"], b["ema"])
    assert a["losses"] != b["losses"]  # different shards
    # DDP's mean gradient of the two ranks == one process on the concatenated batch (the loss is a mean over the batch)
    assert rel(a["sum_grad0"] / 2, a["solo_grad"]) < 1e-5, rel(a["sum_grad0"] / 2, a["solo_grad"])


def test_b2b_trainer_two_steps_vs_reference_plumbing_on_the_double(golden_dir):
    """BASELINE.json config 5 as written (JiTVid-B/16, 156 M parameters): two optimize_parameters() of the unmodified
    reference's b2b_model (AdamW(0.9, 0.95) + EMA, its trainable-pos_embed quirk) with the random draws replayed."""
    from joligen_b200 import nets_jit
    from oracle.gen_golden_b2b_plumbing import batch, draws
    from oracle.vid_oracle import init_params_from_shapes
    gold = torch.load(os.path.join(golden_dir, "b2b_plumbing.pt"))
    gen = gold["gen"]
    net = nets_jit.B2BGenerator(nets_jit.JiTViD(**gold["cfg"]), t_eps=gen["t_eps"], noise_scale=gen["noise_scale"])
    missing, unexpected = net.load_state_dict({**init_params_from_shapes(gold["shapes"], gold["wseed"]),
                                               **gold["frozen"]}, strict=False)
    assert not unexpected and all(m.endswith("pos_encoder.pe") for m in missing), (missing, unexpected)
    o = gold["optim"]
    with KD.installed():
        tr = _b2b_trainer(net, lr=o["lr"], beta1=o["beta1"], beta2=o["beta2"], eps=o["eps"],
                          weight_decay=o["weight_decay"], optim=o["kind"], ema=True, ema_beta=o["ema_beta"],
                          lambda_G=gold["lambda_G"])
        for step in range(2):
            tr.set_input(batch(gold["data_seeds"][step]))
            t_base, e = draws(gold["rng_seeds"][step], gen["P_mean"], gen["P_std"], gen["mix"])
            loss = tr.optimize_parameters(t_base=t_base, e=e)
            assert abs(float(loss) - gold["losses"][step]) < 3e-2 * gold["losses"][step], (step, float(loss))
        got, ema = tr.params(), tr.ema_state_dict()
    for k, (_, nrm) in gold["param_stats"].items():
        assert abs(float(got[k].double().norm()) - nrm) <= 2e-3 * nrm + 1e-6, k
    for k, (_, nrm) in gold["ema_stats"].items():
        assert abs(float(ema[k].double().norm()) - nrm) <= 2e-3 * nrm + 1e-6, k


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
def test_reference_b2b_model_trains_with_accelerated_generator(golden_dir):
    """BASELINE.json config 5 as written, as a DROP-IN: the unmodified reference's b2b_model control path
    (example_b2b_vid_mario.json: create_model -> set_input -> optimize_parameters(): compute_b2b_loss with its keyword
    call of netG_A, backward, AdamW(0.9, 0.95), ema_step) with `accelerate(netG_A)` — B2BGenerator(JiTVid-B/16), 156 M
    parameters — vs the reference's own two steps (b2b_plumbing.pt), seeded identically."""
    from oracle import gen_golden_b2b_plumbing as P
    import joligen_b200
    from joligen_b200 import nets_jit
    gold = torch.load(os.path.join(golden_dir, "b2b_plumbing.pt"))
    model, _, _, _, _ = P.create_reference_model()
    ref_params = dict(model.netG_A.named_parameters())
    keys = [k for k in model.netG_A.state_dict()]
    model.netG_A = joligen_b200.accelerate(model.netG_A)
    assert isinstance(model.netG_A, nets_jit.B2BGenerator)
    assert all(p is ref_params[k] for k, p in model.netG_A.named_parameters()) and len(ref_params) == len(list(model.netG_A.parameters()))
    assert set(keys) <= set(model.netG_A.state_dict())
    losses = []
    with KD.installed():
        for step in range(2):
            data = P.batch(gold["data_seeds"][step])
            model.set_input(dict(data, A_img_paths=["a"] * P.BATCH, B_label_cls=torch.zeros(P.BATCH, dtype=torch.long)))
            torch.manual_seed(gold["rng_seeds"][step])
            model.optimize_parameters()
            losses.append(float(model.loss_G_tot.detach()))
    for got, want in zip(losses, gold["losses"]):
        assert abs(got - want) < 3e-2 * abs(want), (losses, gold["losses"])
    sd = dict(model.netG_A.named_parameters())
    for k, (_, nrm) in gold["param_stats"].items():
        assert abs(float(sd[k].double().norm()) - nrm) <= 2e-3 * nrm + 1e-6, k
    ema = dict(model.netG_A_ema.named_parameters())
    for k, (_, nrm) in gold["ema_stats"].items():
        assert abs(float(ema[k].double().norm()) - nrm) <= 2e-3 * nrm + 1e-6, k


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
def test_reference_b2b_inference_with_accelerated_generator():
    """B2BModel.inference (b2b_model.py:1230-1360: netG.restoration(y_t, y_cond, steps, mask, labels, use_gt=, ref_idx=,
    init_noise=, ...)) on the accelerated generator == the reference's own sampling with the same seed."""
    import contextlib
    from oracle import gen_golden_b2b_plumbing as P
    import joligen_b200
    outs = []
    for fast in (False, True):
        model, _, _, _, _ = P.create_reference_model()
        if fast:
            model.netG_A = joligen_b200.accelerate(model.netG_A)
        model.set_input(dict(P.batch(300), A_img_paths=["a"] * P.BATCH, B_label_cls=torch.zeros(P.BATCH, dtype=torch.long)))
        with (KD.installed() if fast else contextlib.nullcontext()), torch.no_grad():
            torch.manual_seed(8)
            model.inference(2)
        outs.append(model.fake_B.clone())
    assert outs[0].shape == outs[1].shape and rel(outs[1], outs[0]) < 3e-2, rel(outs[1], outs[0])


def test_b2b_trainer_checkpoint_resume_is_exact(golden_dir):
    from oracle.gen_golden_jit import inputs

    def step(tr, cfg, gold, seed):
        gt, cond, mask, _ = inputs(cfg, gold["batch"], gold["frames"], seed)
        torch.manual_seed(seed)
        t_base, e = torch.sigmoid(torch.randn(gold["batch"]) * 0.8 - 0.8), torch.randn_like(gt)
        tr.set_input({"A": cond, "B": gt, "B_label_mask": mask})
        return float(tr.optimize_parameters(t_base=t_base, e=e))

    with KD.installed():
        gold, cfg, net = _small_net(golden_dir)
        tr = _b2b_trainer(net, lr=1e-3, ema_beta=0.9, use_cond=True)
        for s in (40, 41):
            step(tr, cfg, gold, s)
        net_sd, tr_sd = {k: v.clone() for k, v in net.state_dict().items()}, tr.state_dict()
        want = step(tr, cfg, gold, 42)
        _, _, net2 = _small_net(golden_dir)
        tr2 = _b2b_trainer(net2, lr=1e-3, ema_beta=0.9, use_cond=True)
        with torch.no_grad():
            tr2.flat.data.mul_(1.01)
        net2.load_state_dict(net_sd)
        tr2.load_state_dict(tr_sd)
        assert step(tr2, cfg, gold, 42) == want
        assert torch.equal(tr.flat.data, tr2.flat.data) and torch.equal(tr.ema, tr2.ema) and tr.step == tr2.step == 3
