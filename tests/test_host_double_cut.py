"""CUT (BASELINE.json config 3) on the CPU through the kernel TEST DOUBLE: trainer_cut.CutTrainer (G on
cat(real_A, real_B), GAN + NCE + identity NCE for the (G, F) group, then D; flat Adam per group) and trainer_gan vs the
reference's own two optimize_parameters() (tests/golden/cut_plumbing*.pt) — the comparison of
tests/test_gpu_widen_cut.py — and the gradient exchange of its three parameter groups over two gloo ranks."""
import os
import socket
from unittest import mock

import pytest
import torch

import kernel_double as KD

from oracle import ref_stubs  # noqa: E402

REF_MISSING = "needs the reference's own code: build() stages it under oracle/_ref where the checkout is readable"


def _build(golden_dir, golden_name, **kw):
    from joligen_b200 import nets_cut, nets_gan
    from joligen_b200.trainer_cut import CutTrainer
    from oracle.gen_golden_cut_plumbing import batch
    from oracle.vid_oracle import init_params_from_shapes
    gold = torch.load(os.path.join(golden_dir, golden_name))
    opt, cut = gold["optim"], gold["cut"]
    pG, pF, pD = (init_params_from_shapes(gold[k], seed)
                  for k, seed in zip(("shapes_G", "shapes_F", "shapes_D"), gold["seeds"]))
    netG = nets_gan.ResnetGenerator(3, 3, gold["ngf"], n_blocks=gold["n_blocks"])
    netD = nets_gan.NLayerDiscriminator(3, gold["ndf"], n_layers=3)
    netG.load_state_dict(pG)
    netD.load_state_dict(pD)
    netF = nets_cut.PatchSampleF(use_mlp=True, nc=256)
    a0, _ = batch(40)
    netF.data_dependent_initialize(netG.get_feats(a0, cut["nce_layers"]))
    assert [(k, tuple(v.shape)) for k, v in netF.named_parameters()] == [(k, tuple(s)) for k, s in gold["shapes_F"]]
    netF.load_state_dict(pF)
    with mock.patch("torch.cuda.is_available", return_value=True):
        tr = CutTrainer(netG, netF, netD, nce_layers=cut["nce_layers"], num_patches=cut["num_patches"], nce_T=cut["T"],
                        lambda_NCE=cut["lambda_NCE"], nce_idt=cut["nce_idt"], nce_loss=cut["nce_loss"],
                        gan_mode=cut["gan_mode"], lambda_gan=cut["lambda_GAN"], G_lr=opt["G_lr"], D_lr=opt["D_lr"],
                        beta1=opt["beta1"], beta2=opt["beta2"], eps=opt["eps"], weight_decay=opt["weight_decay"],
                        optim=opt["kind"], device="cpu", **kw)
    return gold, tr, (netG, netF, netD)


@pytest.mark.parametrize("golden_name", ["cut_plumbing_patchnce.pt", "cut_plumbing.pt"])
def test_cut_trainer_vs_reference_plumbing_on_the_double(golden_dir, golden_name):
    from oracle import cut_oracle as C
    from oracle import palette_oracle as O
    from oracle.gen_golden_cut_plumbing import batch, patch_ids
    from oracle.vid_oracle import init_params_from_shapes
    with KD.installed():
        gold, tr, (netG, netF, netD) = _build(golden_dir, golden_name)
        opt, cut = gold["optim"], gold["cut"]
        mk = lambda lr: O.OptimCfg(lr=lr, beta1=opt["beta1"], beta2=opt["beta2"], eps=opt["eps"],  # noqa: E731
                                   weight_decay=opt["weight_decay"], kind=opt["kind"], ema_beta=0.0)
        sG, sF, sD = (O.TrainState(params=init_params_from_shapes(gold[k], seed))
                      for k, seed in zip(("shapes_G", "shapes_F", "shapes_D"), gold["seeds"]))
        for step in range(2):
            a, b = batch(gold["data_seeds"][step])
            ids_a, ids_b = patch_ids(gold["rng_seeds"][step], cut["hw"])
            tr.set_input({"A": a, "B": b})
            tr.optimize_parameters(patch_ids_A=ids_a, patch_ids_B=ids_b)
            # the bf16-storage floor of this step: the oracle with the CUDA path's rounding points vs the fp32 golden
            O.EMULATE_BF16[0] = True
            try:
                lo = C.cut_train_step(sG, sF, sD, mk(opt["G_lr"]), mk(opt["G_lr"]), mk(opt["D_lr"]), a, b, ids_a, ids_b,
                                      cut["nce_layers"], n_blocks=gold["n_blocks"], n_layers=3,
                                      lambda_gan=cut["lambda_GAN"], lambda_nce=cut["lambda_NCE"], T=cut["T"],
                                      num_patches=cut["num_patches"], mode=cut["gan_mode"], nce_idt=cut["nce_idt"],
                                      nce_kind=cut["nce_loss"])
            finally:
                O.EMULATE_BF16[0] = False
            ref = gold["losses"][step]
            for mine, key, emu in ((tr.loss_G_tot, "G_tot", lo["G_tot"]), (tr.loss_G_GAN, "G_GAN_D_B_basic", lo["G_GAN"]),
                                   (tr.loss_G_NCE, "G_NCE", lo["G_NCE"]), (tr.loss_G_NCE_Y, "G_NCE_Y", lo["G_NCE_Y"]),
                                   (tr.loss_D_tot, "D_tot", lo["D_tot"])):
                floor = abs(float(emu) - ref[key]) / abs(ref[key])
                # step 0: a pure forward comparison; step 1 sits behind one Adam update of a GAN (sign-like steps from
                # near-zero gradients): the bounds of tests/test_gpu_widen_cut.py
                bound = max(3e-2, 3 * floor) if step == 0 else max(7e-2, 5 * floor)
                assert abs(float(mine.detach()) - ref[key]) < bound * abs(ref[key]), (step, key, float(mine.detach()), floor)
    for net, stats in ((netG, gold["stats_G"]), (netF, gold["stats_F"]), (netD, gold["stats_D"])):
        sd = net.state_dict()
        for k, (_, n) in stats.items():
            assert abs(float(sd[k].double().norm()) - n) <= (5e-2 if k.endswith(".bias") else 1e-2) * n + 1e-6, k


def _dp_worker(rank, world, port, golden_dir, out):
    import torch.distributed as dist
    from oracle.gen_golden_cut_plumbing import batch, patch_ids
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(2)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    with KD.installed():
        gold, tr, nets_ = _build(golden_dir, "cut_plumbing.pt", process_group=dist.group.WORLD)
        losses = []
        for step in range(2):
            a, b = batch(700 + 10 * step + rank)
            ids_a, ids_b = patch_ids(800 + step, gold["cut"]["hw"])
            tr.set_input({"A": a, "B": b})
            tr.optimize_parameters(patch_ids_A=ids_a, patch_ids_B=ids_b)
            losses.append(float(tr.loss_G_tot))
        out[rank] = {"losses": losses, "flat": [torch.cat([p.detach().reshape(-1) for p in n.parameters()]) for n in nets_]}
    dist.barrier()
    dist.destroy_process_group()


def test_cut_trainer_two_ranks_over_gloo(golden_dir):
    """CutTrainer(process_group=...): the G, F and D gradients are averaged over the ranks before their Adam steps —
    replicas that see different images stay bit-identical."""
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_dp_worker, args=(2, port, golden_dir, out), nprocs=2, join=True)
    a, b = out[0], out[1]
    assert a["losses"] != b["losses"]
    for x, y in zip(a["flat"], b["flat"]):
        assert torch.equal(x, y)


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def test_patch_sample_and_nce_on_the_double(golden_dir):
    """PatchSampleF (gather -> MLP as 1x1 convolutions -> L2 norm) + PatchNCELoss vs the reference's golden vectors:
    pooled features, total loss, d loss / d query features and the MLP gradients (incl. the part through the keys)."""
    from types import SimpleNamespace
    from joligen_b200 import nets_cut
    from oracle import cut_oracle as C
    from oracle import palette_oracle as O
    from oracle.gen_golden_cut import feature_maps
    from oracle.vid_oracle import init_params_from_shapes
    gold = torch.load(os.path.join(golden_dir, "cut_nce.pt"))
    params = init_params_from_shapes(gold["shapes"], gold["wseed"])
    netF = nets_cut.PatchSampleF(use_mlp=True, nc=gold["nc"])
    feat_k = list(feature_maps(gold["kseed"]))
    feat_q = [f.requires_grad_(True) for f in feature_maps(gold["qseed"])]
    opt = SimpleNamespace(alg_cut_nce_T=gold["T"], alg_cut_nce_includes_all_negatives_from_minibatch=False,
                          alg_cut_num_patches=gold["num_patches"])
    with KD.installed():
        netF.data_dependent_initialize(feat_k)
        assert [(k, tuple(v.shape)) for k, v in netF.named_parameters()] == [(k, tuple(s)) for k, s in gold["shapes"]]
        netF.load_state_dict(params)
        crit = nets_cut.PatchNCELoss(opt)
        k_pool, ids_out = netF(feat_k, gold["num_patches"], list(gold["ids"]))
        q_pool, _ = netF(feat_q, gold["num_patches"], ids_out)
        for mine, ref in zip(k_pool + q_pool, gold["k_pool"] + gold["q_pool"]):
            assert rel(mine, ref) < 2e-2
        total = sum((crit(feat_q=fq, feat_k=fk, current_batch=gold["batch"]) * gold["lambda_NCE"]).mean()
                    for fq, fk in zip(q_pool, k_pool)) / len(q_pool)
        assert abs(float(total.detach()) - gold["loss"]) < 2e-2 * abs(gold["loss"])
        total.backward()
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    fk = feature_maps(gold["kseed"])
    fq = [f.requires_grad_(True) for f in feature_maps(gold["qseed"])]
    O.EMULATE_BF16[0] = True
    try:
        kp = C.patch_sample(leaves, fk, gold["num_patches"], gold["ids"])
        qp = C.patch_sample(leaves, fq, gold["num_patches"], gold["ids"])
        C.nce_loss_total(qp, kp, gold["batch"], gold["T"], gold["lambda_NCE"]).backward()
    finally:
        O.EMULATE_BF16[0] = False
    for mine, emu, ref in zip(feat_q, fq, gold["dfeat_q"]):
        assert rel(mine.grad, ref) < max(5e-2, 2.5 * rel(emu.grad, ref)), (rel(mine.grad, ref), rel(emu.grad, ref))
    named = dict(netF.named_parameters())
    for k, ref in gold["grads"].items():
        assert abs(float(named[k].grad.double().norm()) - ref["l2"]) < 5e-2 * ref["l2"] + 1e-6, k


def test_multi_scale_d_on_the_double(golden_dir):
    """nets_projd.MultiScaleD (spectral-norm 4x4 stride-2 convs incl. the power iteration, GroupNorm(c/2) + LeakyReLU,
    4x4 valid conv) vs the reference's golden: logits, hinge loss, parameter and feature gradients, u / v after."""
    import torch.nn.functional as F
    from joligen_b200 import nets_projd
    from oracle import palette_oracle as O
    from oracle import projd_oracle as P
    from oracle.gen_golden_projd import features, seeded_state
    gold = torch.load(os.path.join(golden_dir, "projd_small.pt"))
    net = nets_projd.MultiScaleD(channels=gold["channels"], resolutions=gold["resolutions"], conv=True, feats=None,
                                 num_discs=len(gold["channels"]))
    assert [(k, tuple(v.shape)) for k, v in net.state_dict().items()] == [(k, tuple(s)) for k, s in gold["shapes"]]
    net.load_state_dict(seeded_state(gold["shapes"], gold["wseed"]))
    net = net.train()
    feats = {k: v.requires_grad_(True) for k, v in features(gold["fseed"]).items()}
    with KD.installed():
        logits = net(feats)
        assert logits.shape == gold["logits"].shape and rel(logits, gold["logits"]) < 2e-2
        loss = F.relu(torch.ones_like(logits) - logits).mean()
        assert abs(float(loss.detach()) - gold["loss"]) < 2e-2 * abs(gold["loss"])
        loss.backward()
    named = dict(net.named_parameters())
    scale = max(g["l2"] for g in gold["grads"].values())
    for k, g in gold["grads"].items():
        assert abs(float(named[k].grad.double().norm()) - g["l2"]) < 5e-2 * max(g["l2"], 1e-2 * scale), k
    sd0 = seeded_state(gold["shapes"], gold["wseed"])
    emu_feats = {k: v.requires_grad_(True) for k, v in features(gold["fseed"]).items()}
    O.EMULATE_BF16[0] = True
    try:
        lg = P.multi_scale_d(sd0, emu_feats, gold["channels"], gold["resolutions"], training=True)
        F.relu(1 - lg).mean().backward()
    finally:
        O.EMULATE_BF16[0] = False
    for k, ref in gold["dfeats"].items():
        floor = rel(emu_feats[k].grad, ref)
        assert rel(feats[k].grad, ref) < max(5e-2, 2.5 * floor), (k, rel(feats[k].grad, ref), floor)
    sd = net.state_dict()
    for k, ref in gold["uv_after"].items():     # the power iteration is fp32 torch arithmetic: tight
        assert float((sd[k] - ref).abs().max()) < 1e-5, k


def test_gan_trainer_matches_oracle_on_the_double():
    """trainer_gan.GanTrainer: two optimize_parameters() of the (G) and (D) groups (lsgan, Adam) vs the oracle."""
    from joligen_b200 import nets_gan
    from joligen_b200.trainer_gan import GanTrainer
    from oracle import gan_oracle as G
    from oracle import palette_oracle as O
    ngf, nb, ndf = 16, 2, 16
    gshapes, dshapes = G.resnet_param_shapes(3, 3, ngf, nb), G.nlayer_d_param_shapes(3, ndf, 3)
    gp, dpar = G.init_from_shapes(gshapes, 41), G.init_from_shapes(dshapes, 42)
    netG = nets_gan.ResnetGenerator(3, 3, ngf, n_blocks=nb)
    netD = nets_gan.NLayerDiscriminator(3, ndf, n_layers=3)
    netG.load_state_dict(gp)
    netD.load_state_dict(dpar)
    sG = O.TrainState(params={k: v.clone() for k, v in gp.items()})
    sD = O.TrainState(params={k: v.clone() for k, v in dpar.items()})
    ocG = O.OptimCfg(lr=2e-4, kind="adam", ema_beta=0.999)
    ocD = O.OptimCfg(lr=1e-4, kind="adam", ema_beta=0.999)
    g = torch.Generator().manual_seed(3)
    with KD.installed():
        with mock.patch("torch.cuda.is_available", return_value=True):
            tr = GanTrainer(netG, netD, gan_mode="lsgan", G_lr=2e-4, D_lr=1e-4, optim="adam", device="cpu")
        for step in range(2):
            a = torch.rand(2, 3, 64, 64, generator=g) * 2 - 1
            b = torch.rand(2, 3, 64, 64, generator=g) * 2 - 1
            tr.set_input({"A": a, "B": b})
            lg, ld = tr.optimize_parameters()
            rg, rd = G.gan_train_step(sG, sD, ocG, ocD, a, b, n_blocks=nb)
            assert abs(float(lg) - float(rg)) < 3e-2 * abs(float(rg)), (step, float(lg), float(rg))
            assert abs(float(ld) - float(rd)) < 3e-2 * abs(float(rd)), (step, float(ld), float(rd))


def test_cut_trainer_checkpoint_resume_is_exact(golden_dir):
    """nets' state_dicts + CutTrainer.state_dict() into FRESH nets / a fresh trainer continue exactly like the
    uninterrupted run (Adam moments and step counters of the G, F and D groups)."""
    from oracle.gen_golden_cut_plumbing import batch, patch_ids

    def step(tr, hw, seed):
        a, b = batch(seed)
        ids_a, ids_b = patch_ids(seed + 1, hw)
        tr.set_input({"A": a, "B": b})
        tr.optimize_parameters(patch_ids_A=ids_a, patch_ids_B=ids_b)
        return float(tr.loss_G_tot), float(tr.loss_D_tot)

    with KD.installed():
        gold, tr, nets_ = _build(golden_dir, "cut_plumbing_patchnce.pt")
        hw = gold["cut"]["hw"]
        for s in (500, 510):
            step(tr, hw, s)
        saved = [{k: v.clone() for k, v in n.state_dict().items()} for n in nets_], tr.state_dict()
        want = step(tr, hw, 520)
        _, tr2, nets2 = _build(golden_dir, "cut_plumbing_patchnce.pt")
        with torch.no_grad():
            for n in nets2:
                for p in n.parameters():
                    p.mul_(1.01)     # start elsewhere: everything must come from the checkpoint
        for n, sd in zip(nets2, saved[0]):
            n.load_state_dict(sd)
        tr2.load_state_dict(saved[1])
        got = step(tr2, hw, 520)
        assert got == want
        for n, m in zip(nets_, nets2):
            for (k, v), (_, w) in zip(n.state_dict().items(), m.state_dict().items()):
                assert torch.equal(v, w), k


def test_accelerate_swaps_the_projected_discriminator_heads(golden_dir):
    """accelerate() on a module that HOLDS the reference's MultiScaleD (as ProjectedDiscriminator does next to its frozen
    timm feature network): the heads are swapped, parameters and the spectral-norm buffers adopted, logits and the
    power-iteration state after one training-mode forward == the reference heads themselves (stored)."""
    from oracle import skeleton
    import joligen_b200
    from joligen_b200 import nets_projd
    from oracle.gen_golden_projd import features, seeded_state
    gold = torch.load(os.path.join(golden_dir, "projd_small.pt"))
    acc = skeleton.load(os.path.join(golden_dir, "accel_projd_heads.pt"))
    ref = acc["module"]
    ref.load_state_dict(seeded_state(gold["shapes"], gold["wseed"]))
    ref.train()
    keys = list(ref.state_dict().keys())
    holder = torch.nn.Module()
    holder.feature_network = torch.nn.Identity()          # (stands for the frozen backbone)
    holder.discriminator = ref
    params = dict(holder.discriminator.named_parameters())
    joligen_b200.accelerate(holder)
    fast = holder.discriminator
    assert isinstance(fast, nets_projd.MultiScaleD) and isinstance(holder.feature_network, torch.nn.Identity)
    assert list(fast.state_dict().keys()) == keys
    assert all(p is params[k] for k, p in fast.named_parameters())
    with KD.installed():
        got = fast(features(gold["fseed"]))
    assert rel(got, acc["y"]) < 2e-2 and rel(got, gold["logits"]) < 2e-2
    sd = fast.state_dict()
    for k, b in acc["uv_after"].items():
        assert float((sd[k] - b).abs().max()) < 1e-5, k

