"""Host logic above the C ABI, on the CPU, through the kernel TEST DOUBLE (tests/kernel_double.py).

What this proves (and what it does not): `ops.py` / `nets.py` / `accelerate.py` route the right tensors into the right
kernel arguments — packed weights, channel-slice destinations, residual / FiLM / tap / concat plumbing, statistics
stamps, gradient hand-offs — so that, with every kernel replaced by a torch-CPU restatement of its documented contract,
the stack reproduces the unmodified reference's golden vectors, and the reference's own `PaletteModel` trains with
`accelerate(netG_A)` swapped in.  The CUDA kernels themselves are NOT exercised here (that is `-m gpu`).
"""
import os

import pytest
import torch

import kernel_double as KD

from oracle import ref_stubs  # noqa: E402

REF_MISSING = "needs the reference's own code: build() stages it under oracle/_ref where the checkout is readable"



def rel_l2(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _build(cfg, params):
    from joligen_b200 import nets
    g = nets.build_palette_generator(image_size=cfg.image_size, inner_channel=cfg.inner_channel,
                                     res_blocks=cfg.res_blocks, attn_res=cfg.attn_res,
                                     channel_mults=cfg.channel_mults, num_head_channels=cfg.num_head_channels,
                                     use_scale_shift_norm=cfg.use_scale_shift_norm)
    missing, unexpected = g.load_state_dict(params, strict=False)
    assert not unexpected and all("gammas" in m or "posterior" in m for m in missing)
    return g


def _golden_case(golden_dir, name):
    from oracle import palette_oracle as O
    gold = torch.load(os.path.join(golden_dir, name))
    cfg = O.UNetCfg(**gold["cfg"])
    net = _build(cfg, O.init_params(cfg, gold["wseed"]))
    data = O.synthetic_batch(gold["batch"], cfg.image_size, gold["dseed"])
    torch.manual_seed(gold["rseed"])
    t, u = O.sample_t_gamma(cfg, gold["batch"])
    noise = torch.randn_like(data["gt"])
    return gold, net, data, t, u, noise


def _check_against_golden(gold, net, data, t, u, noise):
    _, noise_hat, w = net(data["gt"], data["cond"], data["mask"], noise, t=t, u=u)
    assert rel_l2(w, gold["min_snr_w"]) < 1e-6
    assert rel_l2(noise_hat, gold["noise_hat"]) < 3e-2  # bf16 storage floor of the deep net (tests/test_gpu_palette.py)
    loss = net.forward_loss(data["gt"], data["cond"], data["mask"], noise=noise, t=t, u=u)
    assert abs(float(loss.detach()) - gold["loss"]) < 1e-2 * abs(gold["loss"])
    loss.backward()
    floor = 1e-3 * max(n for _, n in gold["grad_stats"].values())
    err = ref = 0.0
    for k, p in net.named_parameters():
        assert p.grad is not None, k
        g = p.grad.detach().double()
        _, gnorm = gold["grad_stats"][k]
        assert abs(float(g.norm()) - gnorm) <= 6e-2 * gnorm + floor, k
        if "grads" in gold:
            eb = float((g - gold["grads"][k].double()).norm())
            assert eb <= 6e-2 * gnorm + floor, (k, eb, gnorm)
            err += eb * eb
            ref += gnorm * gnorm
    if "grads" in gold:
        assert (err / ref) ** 0.5 < 3e-2


@pytest.mark.parametrize("name", ["palette_small.pt", "palette_mid.pt"])
def test_generator_host_stack_vs_reference_golden(golden_dir, name):
    """DiffusionGenerator -> PaletteDenoiseFn -> UNet (ResBlocks with FiLM, up / down, attention, concat-in-place, taps,
    fused-statistics stamps, batched emb Linears) on the double == the reference's fp32 vectors at the bf16 floor."""
    gold, net, data, t, u, noise = _golden_case(golden_dir, name)
    with KD.installed():
        _check_against_golden(gold, net, data, t, u, noise)


@pytest.mark.parametrize("mode", ["0", "1"])
def test_groupnorm_fusion_modes_route_the_right_sums(golden_dir, mode, monkeypatch):
    """JG_FUSE_GN=0 (no stamps) and =1 (statistics AND backward sums ride in the conv epilogues): the double checks
    inside groupnorm_fwd / _bwd that the sums handed over describe the tensor they are applied to."""
    from joligen_b200 import ops
    monkeypatch.setattr(ops, "FUSE_GN", [mode != "0"])
    monkeypatch.setattr(ops, "FUSE_STATS", [mode == "1"])
    monkeypatch.setattr(ops, "FUSE_SUMS", [mode == "1"])
    monkeypatch.setattr(ops, "FUSE_SUMS_MAX_C", [1 << 20])
    gold, net, data, t, u, noise = _golden_case(golden_dir, "palette_small.pt")
    with KD.installed():
        _check_against_golden(gold, net, data, t, u, noise)


def test_modulewise_dropin_signatures_nchw():
    """ResBlock / AttentionBlock / UNet keep the reference's NCHW fp32 call signatures (module-wise drop-in)."""
    from joligen_b200 import nets
    torch.manual_seed(0)
    with KD.installed():
        rb = nets.ResBlock(16, 32, 0.0, "groupnorm8", out_channel=24, use_scale_shift_norm=True)
        x = torch.randn(2, 16, 8, 8, requires_grad=True)
        emb = torch.randn(2, 32)
        y = rb(x, emb)
        assert y.shape == (2, 24, 8, 8) and y.dtype == torch.float32
        y.sum().backward()
        assert x.grad is not None and x.grad.shape == x.shape
        # the non-FiLM branch (h + emb_out, then GN -> SiLU)
        rb2 = nets.ResBlock(16, 32, 0.0, "groupnorm4", out_channel=24, use_scale_shift_norm=False)
        y2 = rb2(torch.randn(2, 16, 8, 8), emb)
        assert y2.shape == (2, 24, 8, 8)
        # a width the NHWC layout has to pad (20 -> 24 channels) is refused, not normalised over the padding
        rb3 = nets.ResBlock(16, 32, 0.0, "groupnorm4", out_channel=20, use_scale_shift_norm=False)
        with pytest.raises(NotImplementedError, match="multiples of 8"):
            rb3(torch.randn(2, 16, 8, 8), emb)
        ab = nets.AttentionBlock(16, num_head_channels=8)
        ya = ab(torch.randn(2, 16, 8, 8))
        assert ya.shape == (2, 16, 8, 8)


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
def test_reference_palette_model_trains_with_accelerated_generator(golden_dir):
    """THE drop-in claim: the UNMODIFIED reference's control path (options -> create_model -> setup -> set_input ->
    optimize_parameters(): compute_palette_loss, loss.backward(), AdamW, ema_step with its copy.deepcopy) with
    `model.netG_A = joligen_b200.accelerate(model.netG_A)` — INTEGRATION.md section 2 — reproduces the losses, weights
    and EMA weights of the reference's own two steps (tests/golden/palette_plumbing.pt), seeded identically."""
    from oracle import ref_stubs
    ref_stubs.install()
    from oracle import gen_golden
    from oracle import palette_oracle as O
    import joligen_b200
    from joligen_b200 import nets
    gold = torch.load(os.path.join(golden_dir, "palette_plumbing.pt"))
    model, _ = gen_golden.create_reference_model(gold["size"], gold["batch"])
    cfg = O.UNetCfg(**gold["cfg"])
    model.netG_A.load_state_dict(O.init_params(cfg, gold["wseed"]), strict=False)
    ref_params = dict(model.netG_A.named_parameters())
    model.netG_A = joligen_b200.accelerate(model.netG_A)
    assert isinstance(model.netG_A, nets.DiffusionGenerator)
    assert all(p is ref_params[k] for k, p in model.netG_A.named_parameters())  # the optimizer keeps its tensors
    losses = []
    with KD.installed():
        for step in range(2):
            data = O.synthetic_batch(gold["batch"], gold["size"], gold["data_seeds"][step])
            model.set_input({"A": data["cond"], "B": data["gt"], "B_label_mask": data["mask"],
                             "B_label_cls": torch.zeros(gold["batch"], dtype=torch.long),
                             "A_img_paths": ["a"] * gold["batch"]})
            torch.manual_seed(gold["rng_seeds"][step])
            model.optimize_parameters()
            losses.append(float(model.loss_G_tot.detach()))
    # same seeds => same (t, gamma, noise) draws as the reference (the generator draws in the reference's order)
    for got, want in zip(losses, gold["losses"]):
        assert abs(got - want) < 2e-2 * abs(want), (losses, gold["losses"])
    sd = model.netG_A.state_dict()
    for k, (_, n) in gold["param_stats"].items():
        assert abs(float(sd[k].double().norm()) - n) <= 2e-2 * n + 1e-6, k
    assert isinstance(model.netG_A_ema, nets.DiffusionGenerator)  # ema_step's deepcopy of the accelerated tree
    ema = model.netG_A_ema.state_dict()
    for k, (_, n) in gold["ema_stats"].items():
        assert abs(float(ema[k].double().norm()) - n) <= 2e-2 * n + 1e-6, k
    assert rel_l2(sd["denoise_fn.model.middle_block.1.qkv.weight"], gold["sample_param"]) < 2e-2


def test_double_refuses_ops_it_does_not_restate():
    from joligen_b200 import kernels as K
    with KD.installed():
        with pytest.raises(AssertionError, match="no CPU restatement"):
            K.fill_mask_random(torch.zeros(1, 1, 2, 2), torch.zeros(1, 1, 2, 2), torch.zeros(1, 1, 2, 2))
    assert K.fill_mask_random.__module__ == "joligen_b200.kernels"  # restored


# ---------------------------------------------------------------------------------------------------------------------
# GAN generator / discriminator (config 3)
# ---------------------------------------------------------------------------------------------------------------------
def _emulated_grads(fn, shapes, wseed, x, dy, *args):
    """What bf16 STORAGE alone does to the gradients: the oracle in bf16-storage emulation (leaf gradients)."""
    from oracle import gan_oracle as G
    from oracle import palette_oracle as O
    leaves = {k: v.requires_grad_(True) for k, v in G.init_from_shapes(shapes, wseed).items()}
    O.EMULATE_BF16[0] = True
    try:
        fn(leaves, x, *args).backward(dy)
    finally:
        O.EMULATE_BF16[0] = False
    return {k: v.grad for k, v in leaves.items()}


def _check_grads_at_bf16_floor(named_grads, ref_grads, emu_grads):
    """InstanceNorm backward on these small random nets is ill-conditioned under bf16 storage (the oracle's own
    emulation is ~15 % off the fp32 gradients on the early layers): like tests/test_gpu_gan.py, the path under test must
    be no worse than that floor warrants."""
    gmax = max(float(v.double().norm()) for v in ref_grads.values())
    for k, g in named_grads:
        gref = ref_grads[k].double()
        if float(gref.norm()) < 1e-3 * gmax:  # conv biases in front of an InstanceNorm: true gradient 0
            assert float(g.double().norm()) < 5e-2 * gmax, k
            continue
        e = float((g.double() - gref).norm() / gref.norm())
        e_emu = float((emu_grads[k].double() - gref).norm() / gref.norm())
        assert e <= 1.5 * e_emu + 2e-2, (k, e, e_emu)


def test_gan_nets_host_stack_vs_reference_golden(golden_dir):
    """nets_gan.ResnetGenerator / NLayerDiscriminator / GANLoss on the double vs gan_resnet.pt / gan_nlayerd.pt."""
    from joligen_b200 import nets_gan, ops
    from oracle import gan_oracle as G
    gold = torch.load(os.path.join(golden_dir, "gan_resnet.pt"))
    net = nets_gan.ResnetGenerator(3, 3, gold["ngf"], n_blocks=gold["n_blocks"])
    shapes = G.resnet_param_shapes(3, 3, gold["ngf"], gold["n_blocks"])
    net.load_state_dict(G.init_from_shapes(shapes, gold["wseed"]))
    with KD.installed():
        y = net(gold["x"])
        assert rel_l2(y, gold["y"]) < 3e-2
        y.backward(gold["dy"])
        feats = net.get_feats(gold["x"], gold["feat_ids"])
    emu = _emulated_grads(G.resnet_generator, shapes, gold["wseed"], gold["x"], gold["dy"], gold["n_blocks"])
    _check_grads_at_bf16_floor([(k, p.grad) for k, p in net.named_parameters()], gold["grads"], emu)
    for f, fref in zip(feats, gold["feats"]):
        assert tuple(f.shape) == tuple(fref.shape) and rel_l2(f, fref) < 3e-2
    gold = torch.load(os.path.join(golden_dir, "gan_nlayerd.pt"))
    netd = nets_gan.NLayerDiscriminator(3, gold["ndf"], n_layers=3)
    netd.load_state_dict(G.init_from_shapes(G.nlayer_d_param_shapes(3, gold["ndf"], 3), gold["wseed"]))
    with KD.installed():
        pred = netd(gold["x"])
        assert rel_l2(pred, gold["pred"]) < 3e-2
        crit = nets_gan.GANLoss("lsgan")
        logits = netd.forward_nhwc(ops.to_nhwc(gold["x"]))
        loss_real = crit.forward_nhwc(logits, True)
        assert abs(float(loss_real.detach()) - gold["loss_real"]) < 2e-2 * gold["loss_real"]
        assert abs(float(crit.forward_nhwc(logits, False).detach()) - gold["loss_fake"]) < 2e-2 * gold["loss_fake"]
        hinge = nets_gan.GANLoss("projected")
        assert abs(float(hinge.forward_nhwc(logits, True).detach()) - gold["hinge_real"]) < 2e-2 * gold["hinge_real"]
        loss_real.backward()
    floor = 1e-3 * max(float(v.double().norm()) for v in gold["grads"].values())
    for k, p in netd.named_parameters():
        gref = gold["grads"][k].double()
        assert float((p.grad.double() - gref).norm()) <= 8e-2 * float(gref.norm()) + floor, k


def test_accelerate_swaps_reference_gan_nets_and_matches_their_forward(golden_dir):
    """accelerate() on the reference's own ResnetGenerator / NLayerDiscriminator objects (stored module trees,
    oracle/gen_golden_accelerate.py): parameters adopted, same state_dict keys, and (on the double) the outputs, encoder
    features and every gradient (sampled) of the reference modules evaluating themselves in fp32, at the bf16-storage
    floor."""
    from oracle import gan_oracle as G
    from oracle import skeleton
    from oracle.gen_golden_accelerate import sample
    import joligen_b200
    from joligen_b200 import nets_gan
    cases = (("resnet", nets_gan.ResnetGenerator, G.resnet_param_shapes(3, 3, 16, 2), G.resnet_generator, (2,)),
             ("nlayerd", nets_gan.NLayerDiscriminator, G.nlayer_d_param_shapes(3, 16, 3), G.nlayer_discriminator, (3,)))
    for name, kind, shapes, oracle_fn, oargs in cases:
        gold = skeleton.load(os.path.join(golden_dir, "accel_gan_%s.pt" % name))
        ref = gold["module"]
        ref.load_state_dict(G.init_from_shapes(shapes, 77))
        params, keys = dict(ref.named_parameters()), list(ref.state_dict().keys())
        fast = joligen_b200.accelerate(ref)
        assert isinstance(fast, kind) and list(fast.state_dict().keys()) == keys
        assert all(p is params[k] for k, p in fast.named_parameters())
        x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1))
        dy = torch.randn(gold["y"].shape, generator=torch.Generator().manual_seed(2))
        with KD.installed():
            yf = fast(x)
            assert tuple(yf.shape) == tuple(gold["y"].shape) and rel_l2(yf, gold["y"]) < 3e-2
            yf.backward(dy)
            if kind is nets_gan.ResnetGenerator:
                ff = fast.get_feats(x, [0, 4, 8, 11])
                for a, (shape, b) in zip(ff, gold["feats"]):
                    assert tuple(a.shape) == shape and rel_l2(sample(a), b) < 3e-2
        emu = _emulated_grads(oracle_fn, shapes, 77, x, dy, *oargs)
        _check_grads_at_bf16_floor([(k, sample(p.grad)) for k, p in fast.named_parameters()], gold["grads"],
                                   {k: sample(g) for k, g in emu.items()})
    # variants the mirrors do not implement are refused, not swapped silently
    for ref in skeleton.load(os.path.join(golden_dir, "accel_gan_refused.pt")):
        with pytest.raises((NotImplementedError, RuntimeError)):
            joligen_b200.accelerate(ref)



@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
@pytest.mark.parametrize("nce", [None, "patchnce"])
def test_reference_cut_model_trains_with_accelerated_nets(golden_dir, nce):
    """The reference's cut_model (example_gan_horse2zebra.json, reduced) through its own optimize_parameters() — GAN +
    NCE + identity NCE for (G, F), then D — with netG_A and netD_B_basic swapped by accelerate(): losses of both steps
    vs the reference's own (cut_plumbing*.pt)."""
    from oracle import gen_golden_cut_plumbing as P
    import joligen_b200
    from joligen_b200 import nets_gan
    gold = torch.load(os.path.join(golden_dir, "cut_plumbing.pt" if nce is None else "cut_plumbing_%s.pt" % nce))
    model, _, _, _, _, _ = P.create_reference_model(nce)
    model.netG_A = joligen_b200.accelerate(model.netG_A)
    model.netD_B_basic = joligen_b200.accelerate(model.netD_B_basic)
    assert isinstance(model.netG_A, nets_gan.ResnetGenerator)
    assert isinstance(model.netD_B_basic, nets_gan.NLayerDiscriminator)
    names = ["G_tot", "G_GAN_D_B_basic", "G_NCE", "G_NCE_Y", "D_tot"]
    with KD.installed():
        for step in range(2):
            a, b = P.batch(gold["data_seeds"][step])
            model.set_input({"A": a, "B": b, "A_img_paths": ["a"] * P.BATCH, "B_img_paths": ["b"] * P.BATCH})
            torch.manual_seed(gold["rng_seeds"][step])
            model.optimize_parameters()
            for n in names:
                got, want = float(getattr(model, "loss_" + n).detach()), gold["losses"][step][n]
                # step 0 is a pure forward comparison; step 1 sits behind one Adam update of a GAN (sign-like steps
                # from near-zero gradients): the bounds of tests/test_gpu_widen_cut.py
                assert abs(got - want) < (3e-2 if step == 0 else 7e-2) * abs(want) + 1e-3, (step, n, got, want)
    for k, (_, n) in gold["stats_D"].items():
        if not k.endswith(".bias"):
            assert abs(float(model.netD_B_basic.state_dict()[k].double().norm()) - n) <= 2e-2 * n, k


# ---------------------------------------------------------------------------------------------------------------------
# INTEGRATION.md section 2 under DistributedDataParallel (what BaseModel.parallelize builds, base_model.py:725-737) with
# gradient accumulation (train_iter_size = 2: the first micro-step under no_sync, base_model.py:1313-1315), two gloo
# ranks on the CPU through the double.  Pins (ADVICE r1) that EVERY parameter gradient of the B200 modules reaches
# autograd's AccumulateGrad — on the first and on the second micro-step, when .grad already exists — so the reducer
# hooks fire for the convolution weights too.  (tests/test_gpu_multi.py runs the same on the real kernels.)
# ---------------------------------------------------------------------------------------------------------------------
_DDP_CFG = dict(image_size=32, inner_channel=32, channel_mults=(1, 2), res_blocks=(1, 1), attn_res=(2,),
                num_head_channels=16)


def _ddp_double_worker(rank, world, port, out):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(2)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from joligen_b200 import nets
    from oracle import palette_oracle as O
    cfg = O.UNetCfg(**_DDP_CFG)

    def make():
        net = nets.build_palette_generator(**_DDP_CFG)
        net.load_state_dict(O.init_params(cfg, 50), strict=False)
        return net

    def draw(seed):
        data = O.synthetic_batch(2, cfg.image_size, seed)
        torch.manual_seed(seed + 7)
        t, u = O.sample_t_gamma(cfg, 2)
        return data, torch.randn_like(data["gt"]), t, u

    def loss_of(model, d):
        data, noise, t, u = d
        _, noise_hat, _ = model(data["gt"], data["cond"], data["mask"], noise, t=t, u=u)
        return torch.nn.functional.mse_loss(noise_hat, noise)

    draws = {(r, m): draw(5000 + 10 * r + m) for r in range(world) for m in range(2)}
    with KD.installed():
        ddp = DDP(make())
        with ddp.no_sync():
            (loss_of(ddp, draws[(rank, 0)]) / 2).backward()
        (loss_of(ddp, draws[(rank, 1)]) / 2).backward()
        got = {k: p.grad.detach().clone() for k, p in ddp.module.named_parameters() if p.grad is not None}
        res = {"n_grads": len(got), "n_params": sum(1 for _ in ddp.module.parameters())}
        if rank == 0:
            solo = make()
            for r in range(world):
                for m in range(2):
                    (loss_of(solo, draws[(r, m)]) / (2 * world)).backward()
            worst, worst_k = 0.0, None
            for k, p in solo.named_parameters():
                ref = p.grad.detach().double()
                e = float((got[k].double() - ref).norm() / (ref.norm() + 1e-12))
                if e > worst and float(ref.norm()) > 1e-6:
                    worst, worst_k = e, k
            res["worst"], res["worst_k"] = worst, worst_k
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_ddp_wrapped_modules_with_gradient_accumulation_on_the_double():
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_ddp_double_worker, args=(2, port, out), nprocs=2, join=True)
    a, b = out[0], out[1]
    assert a["n_grads"] == a["n_params"] == b["n_grads"]
    # DDP's mean over ranks of the accumulated micro-step gradients == the plain sum / (2 * world) on one model; a
    # parameter whose gradient skipped the reducer would hold its rank-local value (different data: error ~ 1)
    assert a["worst"] < 1e-3, (a["worst_k"], a["worst"])


# ---------------------------------------------------------------------------------------------------------------------
# --G_unet_mha_vit_efficient (efficient=True: skip weight 1/sqrt(2), up-blocks convolve BEFORE upsampling) and the
# non-FiLM ResBlock: the oracle vs the reference directly, the host stack vs the oracle and vs the reference
# ---------------------------------------------------------------------------------------------------------------------
_VARIANT_BASE = dict(image_size=32, inner_channel=32, channel_mults=(1, 2), res_blocks=(1, 1), attn_res=(2,),
                     num_head_channels=16)


@pytest.mark.parametrize("variant", [dict(efficient=True), dict(use_scale_shift_norm=False)])
def test_unet_variants_oracle_host_stack_and_reference_agree(variant, golden_dir):
    """The reference generator of each variant (stored module tree and its fp32 forward / gradients,
    oracle/gen_golden_accelerate.py) vs the oracle, and accelerate() of it on the double."""
    from oracle import palette_oracle as O
    from oracle import skeleton
    from oracle.gen_golden_accelerate import UNET_VARIANT_BASE, sample
    import joligen_b200
    cfg = O.UNetCfg(**UNET_VARIANT_BASE, **variant)
    params = O.init_params(cfg, 5)
    gold = skeleton.load(os.path.join(golden_dir, "accel_unet_%s.pt" % ("efficient" if cfg.efficient else
                                                                        "no_scale_shift")))
    ref = gold["module"]
    assert [(k, tuple(v.shape)) for k, v in ref.named_parameters()] == list(O.generator_param_shapes(cfg).items())
    ref.load_state_dict(params, strict=False)
    nh_r, ref_grads = gold["noise_hat"], gold["grads"]
    data = O.synthetic_batch(2, cfg.image_size, 9)
    torch.manual_seed(1)
    t, u = O.sample_t_gamma(cfg, 2)
    noise = torch.randn_like(data["gt"])
    # the reference drew the same noise with the same seed (its forward draws t, u, then the noise)
    assert torch.equal(gold["noise"], noise)
    # (1) the oracle restates the reference (fp32)
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    _, nh_o, _ = O.diffusion_forward(leaves, data["gt"], data["cond"], data["mask"], noise, t, u, cfg)
    assert rel_l2(nh_o, nh_r) < 1e-4
    O.palette_loss(noise, nh_o, data["mask"]).backward()
    for k in ref_grads:
        assert rel_l2(sample(leaves[k].grad), ref_grads[k]) < 1e-3 or float(ref_grads[k].norm()) < 1e-6, k
    # (2) the accelerated reference net on the double, seeded the same way, at the bf16 floor of THIS net (measured: the
    # oracle with the CUDA path's rounding points vs fp32; the 1/sqrt(2) skip weight makes the efficient variant noisier)
    emu = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    O.EMULATE_BF16[0] = True
    try:
        _, nh_e, _ = O.diffusion_forward(emu, data["gt"], data["cond"], data["mask"], noise, t, u, cfg)
        O.palette_loss(noise, nh_e, data["mask"]).backward()
    finally:
        O.EMULATE_BF16[0] = False
    floor = rel_l2(nh_e, nh_r)
    gerr = gnrm = 0.0
    for k, q in ref_grads.items():
        gerr += float((sample(emu[k].grad).double() - q.double()).norm()) ** 2
        gnrm += float(q.double().norm()) ** 2
    gfloor = (gerr / gnrm) ** 0.5
    fast = joligen_b200.accelerate(ref)
    fast.zero_grad()
    with KD.installed():
        torch.manual_seed(1)
        noise_f, nh_f, _ = fast(data["gt"], data["cond"], data["mask"], None, None, None)
        assert torch.equal(noise_f, noise) and rel_l2(nh_f, nh_r) < max(3e-2, 1.5 * floor), (rel_l2(nh_f, nh_r), floor)
        torch.nn.functional.mse_loss(noise_f * data["mask"].clamp(0, 1), nh_f * data["mask"].clamp(0, 1)).backward()
    err = nrm = 0.0
    for k, p in fast.named_parameters():
        q = ref_grads[k]
        err += float((sample(p.grad).double() - q.double()).norm()) ** 2
        nrm += float(q.double().norm()) ** 2
    assert (err / nrm) ** 0.5 < max(4e-2, 1.5 * gfloor), ((err / nrm) ** 0.5, gfloor)



@pytest.mark.parametrize("norm", ["instancenorm", "layernorm", "groupnorm"])
def test_accelerate_rebuilds_the_reference_norm_variant(norm, golden_dir):
    """--G_unet_mha_norm_layer instancenorm (GroupNorm(C, C): the group count follows each block's width) / layernorm
    (GroupNorm(1, C)) / groupnorm N: accelerate() must rebuild every block's normalisation, not the first block's group
    count everywhere — checked structurally and against the reference's own forward (stored)."""
    from oracle import skeleton
    import torch.nn as nn
    import joligen_b200
    gold = skeleton.load(os.path.join(golden_dir, "accel_norm_%s.pt" % norm))
    ref = skeleton.seed_(gold["module"], 3)
    groups = lambda m: [(g.num_groups, g.num_channels) for g in m.modules() if isinstance(g, nn.GroupNorm)]  # noqa: E731
    want_groups = groups(ref)
    fast = joligen_b200.accelerate(ref)
    assert groups(fast) == want_groups
    with KD.installed():
        got = fast(gold["x"], gold["emb"])
    assert rel_l2(got, gold["y"]) < 4e-2, rel_l2(got, gold["y"])



@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
def test_reference_palette_inference_with_accelerated_generator():
    """PaletteModel.inference (palette_model.py:622-760: set_new_noise_schedule on the denoiser, set_new_sampling_method,
    netG.restoration(y_cond=, y_t=, y_0=, mask=, sample_num=, cls=, ddim_num_steps=, ddim_eta=)) on the accelerated
    generator == the reference sampling itself with the same seeds (8 reverse steps)."""
    from oracle import ref_stubs
    ref_stubs.install()
    from oracle import gen_golden
    from oracle import palette_oracle as O
    import contextlib
    import joligen_b200
    outs = []
    for fast in (False, True):
        model, _ = gen_golden.create_reference_model(32, 2, extra={"G_diff_n_timestep_test": 8})
        model.netG_A.load_state_dict(O.init_params(O.UNetCfg(**gen_golden.SMALL), 21), strict=False)
        if fast:
            model.netG_A = joligen_b200.accelerate(model.netG_A)
        data = O.synthetic_batch(2, 32, 100)
        torch.manual_seed(7)
        model.set_input({"A": data["cond"], "B": data["gt"], "B_label_mask": data["mask"],
                         "B_label_cls": torch.zeros(2, dtype=torch.long), "A_img_paths": ["a"] * 2})
        with (KD.installed() if fast else contextlib.nullcontext()), torch.no_grad():
            torch.manual_seed(8)
            model.inference(2)
        outs.append((model.output.clone(), model.visuals.clone()))
    assert outs[0][0].shape == outs[1][0].shape and outs[0][1].shape == outs[1][1].shape
    assert rel_l2(outs[1][0], outs[0][0]) < 3e-2 and rel_l2(outs[1][1], outs[0][1]) < 3e-2


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
def test_reference_checkpoints_interchange_with_accelerated_nets():
    """BaseModel.save_networks / load_networks (base_model.py:824-868, 957-1103) on a model whose netG_A was accelerated:
    the files load into an UNMODIFIED reference net (all keys matched), and into another accelerated model — whose
    convolutions then run on the loaded weights (the bf16 copies are re-packed)."""
    from oracle import ref_stubs
    ref_stubs.install()
    from oracle import gen_golden
    from oracle import palette_oracle as O
    import joligen_b200
    model, _ = gen_golden.create_reference_model(32, 2)
    model.netG_A.load_state_dict(O.init_params(O.UNetCfg(**gen_golden.SMALL), 21), strict=False)
    model.netG_A = joligen_b200.accelerate(model.netG_A)
    data = O.synthetic_batch(2, 32, 100)
    batch = {"A": data["cond"], "B": data["gt"], "B_label_mask": data["mask"],
             "B_label_cls": torch.zeros(2, dtype=torch.long), "A_img_paths": ["a"] * 2}
    x, emb = torch.randn(2, 6, 32, 32), torch.randn(2, 32)
    with KD.installed():
        model.set_input(batch)
        model.optimize_parameters()
        os.makedirs(model.save_dir, exist_ok=True)
        model.save_networks("latest")
        assert sorted(os.listdir(model.save_dir)) == ["latest_net_G_A.pth", "latest_net_G_A_ema.pth"]
        plain, _ = gen_golden.create_reference_model(32, 2)
        for name in ("latest_net_G_A.pth", "latest_net_G_A_ema.pth"):
            res = plain.netG_A.load_state_dict(torch.load(os.path.join(model.save_dir, name)))
            assert not res.missing_keys and not res.unexpected_keys
        other, _ = gen_golden.create_reference_model(32, 2)
        other.netG_A = joligen_b200.accelerate(other.netG_A)
        before = other.netG_A.denoise_fn.model(x, emb)       # packs the (different) initial weights
        other.save_dir = model.save_dir
        other.load_networks("latest")
        after = other.netG_A.denoise_fn.model(x, emb)
        want = model.netG_A.denoise_fn.model(x, emb)
    assert torch.equal(after, want) and not torch.equal(before, want)
    # the reference net evaluating the same checkpoint itself, fp32
    plain.netG_A.load_state_dict(torch.load(os.path.join(model.save_dir, "latest_net_G_A.pth")))
    with torch.no_grad():
        assert rel_l2(want, plain.netG_A.denoise_fn.model(x, emb)) < 3e-2


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
def test_train_launcher_hook_accelerates_the_models_train_py_creates():
    """joligen_b200.train: the create_model hook (what `python -m joligen_b200.train` installs in every rank) swaps the
    nets of the models joliGEN's own train.py builds — palette_model and cut_model — and leaves the rest alone."""
    from oracle import ref_stubs
    ref_stubs.install()
    import train as ref_train
    import models
    from joligen_b200 import nets, nets_gan
    from joligen_b200 import train as launcher
    saved = ref_train.create_model, models.create_model
    try:
        launcher.install_hook()
        launcher.install_hook()   # idempotent
        from oracle import gen_golden, gen_golden_cut_plumbing
        model, _ = gen_golden.create_reference_model(32, 2)           # its `from models import create_model` is hooked
        assert isinstance(model.netG_A, nets.DiffusionGenerator)
        opt_params = {id(p) for g in model.optimizer_G.param_groups for p in g["params"]}
        assert {id(p) for p in model.netG_A.parameters()} == opt_params   # the optimizer built before the swap still applies
        with KD.installed():   # cut_model's data_dependent_initialize runs the (now accelerated) generator
            cut, _, _, _, _, _ = gen_golden_cut_plumbing.create_reference_model("patchnce")
        assert isinstance(cut.netG_A, nets_gan.ResnetGenerator) and isinstance(cut.netD_B_basic, nets_gan.NLayerDiscriminator)
        assert type(cut.netF).__module__.startswith("models.")          # no mirror: stays the reference's
        # the spawn target resolves to the reference's train_gpu in a fresh interpreter (no recursion on itself)
        assert launcher._ORIG_TRAIN_GPU is None and ref_train.train_gpu.__module__ == "train"
    finally:
        ref_train.create_model, models.create_model = saved
        ref_train._jg_hooked = False


@pytest.mark.parametrize("padding_type", ["replicate", "zeros"])
def test_accelerate_resnet_generator_padding_types(padding_type, golden_dir):
    """--G_padding_type replicate / zeros (resnet_generator.py:42-50, 328-336): accelerate() reads it off the layers,
    the mirror runs nn.ReplicationPad2d through jg_pad2d (mode 1) / the zero padding inside the convolution — output,
    encoder features and input gradient vs the reference module itself (stored)."""
    from oracle import gan_oracle as G
    from oracle import skeleton
    from oracle.gen_golden_accelerate import sample
    import joligen_b200
    from joligen_b200 import nets_gan
    gold = skeleton.load(os.path.join(golden_dir, "accel_resnet_padding_%s.pt" % padding_type))
    ref = gold["module"]
    seeded = list(G.init_from_shapes(G.resnet_param_shapes(3, 3, 16, 2), 77).values())
    ref.load_state_dict(dict(zip(ref.state_dict().keys(), seeded)))   # (the layer indices shift without pad layers)
    ref_layers = [type(m).__name__ for m in ref.decoder.model]
    fast = joligen_b200.accelerate(ref)
    assert isinstance(fast, nets_gan.ResnetGenerator)
    assert [type(m).__name__ for m in fast.decoder.model] == ref_layers
    x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1))
    xf = x.clone().requires_grad_(True)
    dy = torch.randn(gold["y"].shape, generator=torch.Generator().manual_seed(2))
    with KD.installed():
        yf = fast(xf)
        assert rel_l2(yf, gold["y"]) < 3e-2
        yf.backward(dy)
        for a, (shape, b) in zip(fast.get_feats(x, [0, 4, 8, 11]), gold["feats"]):
            assert tuple(a.shape) == shape and rel_l2(sample(a), b) < 3e-2
    assert rel_l2(xf.grad, gold["x_grad"]) < 0.3   # (InstanceNorm backward under bf16 storage: see the floor tests above)



def test_accelerate_wavelet_space_unet_vs_reference(golden_dir):
    """--train_feat_wavelet (UNet(freq_space=True), unet_generator_attn.py:467-473, 69-96, 113-140): the net works on
    the Haar bands of its input / output and resamples in pixel space (inverse transform -> resample -> transform).
    The mirror composes jg_haar with the layout / resample kernels; accelerate() adopts the filter buffers — output and
    input gradient vs the reference's own forward / backward (stored)."""
    from oracle import skeleton
    import joligen_b200
    from joligen_b200 import nets
    gold = skeleton.load(os.path.join(golden_dir, "accel_wavelet_unet.pt"))
    ref = skeleton.seed_(gold["module"], 3)
    keys = list(ref.state_dict().keys())
    fast = joligen_b200.accelerate(ref)
    assert isinstance(fast, nets.UNet) and fast.freq_space and list(fast.state_dict().keys()) == keys
    assert (fast.in_channel, fast.out_channel) == (6, 3)
    xf = gold["x"].clone().requires_grad_(True)
    want = gold["y"]
    with KD.installed():
        got = fast(xf, gold["emb"])
        assert tuple(got.shape) == tuple(want.shape) == (1, 3, 32, 32)
        assert rel_l2(got, want) < 4e-2, rel_l2(got, want)
        got.backward(gold["dy"])
    assert rel_l2(xf.grad, gold["x_grad"]) < 0.1, rel_l2(xf.grad, gold["x_grad"])



def test_accelerate_wavelet_space_discriminator_vs_reference(golden_dir):
    """NLayerDiscriminator(freq_space=True) (discriminators.py:40-46, 112-117): the PatchGAN reads the Haar bands."""
    from oracle import skeleton
    import joligen_b200
    from joligen_b200 import nets_gan, ops
    gold = skeleton.load(os.path.join(golden_dir, "accel_wavelet_nlayerd.pt"))
    ref = skeleton.seed_(gold["module"], 4)
    keys = list(ref.state_dict().keys())
    fast = joligen_b200.accelerate(ref)
    assert isinstance(fast, nets_gan.NLayerDiscriminator) and fast.freq_space and list(fast.state_dict().keys()) == keys
    x, want = gold["x"], gold["y"]
    with KD.installed():
        got = fast(x)
        got2 = ops.to_nchw(fast.forward_nhwc(ops.to_nhwc(x)), 1)     # the trainers' NHWC entry point
    assert tuple(got.shape) == tuple(want.shape) and rel_l2(got, want) < 3e-2 and rel_l2(got2, want) < 3e-2



def test_accelerate_spectral_norm_discriminator_vs_reference(golden_dir):
    """--D_spectral: NLayerDiscriminator of torch-spectral_norm-wrapped convolutions (`weight_orig`, `weight_u`,
    `weight_v` in the state_dict).  The wrapper's pre-forward hook never runs on the B200 path: the mirror does the power
    iteration and the normalisation itself (nets_projd._sn_weight) — logits, the last layer's gradient and the u / v
    buffers after one training-mode forward vs the reference module (stored)."""
    from oracle import skeleton
    from oracle.gen_golden_accelerate import sample
    import joligen_b200
    from joligen_b200 import nets_gan
    gold = skeleton.load(os.path.join(golden_dir, "accel_spectral_nlayerd.pt"))
    ref = skeleton.seed_(gold["module"], 2).train()
    keys = list(ref.state_dict().keys())
    fast = joligen_b200.accelerate(ref)
    assert isinstance(fast, nets_gan.NLayerDiscriminator) and list(fast.state_dict().keys()) == keys
    assert any(k.endswith("weight_orig") for k in keys) and any(k.endswith("weight_u") for k in keys)
    with KD.installed():
        got = fast(gold["x"])
        assert rel_l2(got, gold["y"]) < 3e-2, rel_l2(got, gold["y"])
        got.backward(gold["dy"])
    sd = fast.state_dict()
    for k, b in gold["uv_after"].items():   # the power iteration is fp32 torch arithmetic on both sides
        assert float((sd[k] - b).abs().max()) < 1e-5, k
    last = [k for k in keys if k.endswith("weight_orig")][-1]
    assert rel_l2(sample(dict(fast.named_parameters())[last].grad), gold["grads"][last]) < 3e-2



def test_accelerate_spectral_norm_generator_vs_reference(golden_dir):
    """--G_spectral: ResnetGenerator whose convolutions AND transposed convolutions are spectral_norm-wrapped (the matrix
    rows of a ConvTranspose2d are its OUTPUT channels: dim 1) — output, the u / v buffers after one training-mode
    forward and the gradient of a transposed-convolution weight vs the reference module (stored)."""
    from oracle import skeleton
    from oracle.gen_golden_accelerate import sample
    import joligen_b200
    from joligen_b200 import nets_gan
    gold = skeleton.load(os.path.join(golden_dir, "accel_spectral_resnet.pt"))
    ref = skeleton.seed_(gold["module"], 4).train()
    keys = list(ref.state_dict().keys())
    fast = joligen_b200.accelerate(ref)
    assert isinstance(fast, nets_gan.ResnetGenerator) and list(fast.state_dict().keys()) == keys
    # wrapped: stem, down- and up-sampling layers; NOT wrapped: the ResnetBlocks (a reference quirk) and the 7x7 head
    assert "decoder.model.0.weight_orig" in keys and "decoder.model.7.weight" in keys
    assert "encoder.model.10.conv_block.1.weight" in keys
    with KD.installed():
        got = fast(gold["x"])
        assert rel_l2(got, gold["y"]) < 3e-2, rel_l2(got, gold["y"])
        got.backward(gold["dy"])
    sd = fast.state_dict()
    for k, b in gold["uv_after"].items():
        assert float((sd[k] - b).abs().max()) < 1e-5, k
    gf = sample(dict(fast.named_parameters())["decoder.model.3.weight_orig"].grad)
    gr = gold["grads"]["decoder.model.3.weight_orig"]
    assert rel_l2(gf, gr) < 0.15, rel_l2(gf, gr)

