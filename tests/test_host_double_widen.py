"""Host logic of the widening rows on the CPU through the kernel TEST DOUBLE (tests/kernel_double.py): samplers,
class / mask conditioning, the reference-image UNet, the video UNet — the same comparisons tests/test_gpu_*.py make on
the real kernels, against the same golden vectors of the unmodified reference.  See tests/test_host_double.py for
what a pass does and does not prove."""
import os

import pytest
import torch

import kernel_double as KD

from oracle import ref_stubs  # noqa: E402

REF_MISSING = "needs the reference's own code: build() stages it under oracle/_ref where the checkout is readable"


def rel_l2(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


class _Emulated:
    """oracle.palette_oracle.EMULATE_BF16 for the duration of a with-block"""

    def __enter__(self):
        from oracle import palette_oracle as O
        O.EMULATE_BF16[0] = True

    def __exit__(self, *a):
        from oracle import palette_oracle as O
        O.EMULATE_BF16[0] = False


def test_ddpm_and_ddim_samplers_on_the_double(golden_dir):
    """restoration_ddpm / restoration (ddim): forward-only UNet + one fused step per reverse step (jg_ddpm_step)."""
    from joligen_b200 import nets
    from oracle import palette_oracle as O
    gold = torch.load(os.path.join(golden_dir, "palette_sampling.pt"))
    cfg = O.UNetCfg(**gold["cfg"])
    params = O.init_params(cfg, gold["wseed"])
    data = O.synthetic_batch(gold["batch"], cfg.image_size, gold["dseed"])
    torch.manual_seed(gold["rseed"])
    y_t0 = torch.randn_like(data["gt"])
    noises = {i: torch.randn_like(data["gt"]) for i in reversed(range(1, cfg.n_timestep_test))}
    g = nets.build_palette_generator(image_size=cfg.image_size, inner_channel=cfg.inner_channel,
                                     res_blocks=cfg.res_blocks, attn_res=cfg.attn_res,
                                     channel_mults=cfg.channel_mults, num_head_channels=cfg.num_head_channels,
                                     n_timestep_test=cfg.n_timestep_test)
    g.load_state_dict(params, strict=False)
    m = data["mask"].clamp(0, 1).bool().expand_as(data["gt"])
    with KD.installed():
        y, ret = g.restoration_ddpm(data["cond"], y_t=y_t0, y_0=data["gt"], mask=data["mask"],
                                    sample_num=gold["sample_num"], noise_fn=lambda i, shape: noises[i])
        g.sampling_method = "ddim"
        yd, retd = g.restoration(data["cond"], y_t=y_t0, y_0=data["gt"], mask=data["mask"],
                                 sample_num=gold["sample_num"], ddim_num_steps=gold["ddim_steps"],
                                 ddim_eta=gold["ddim_eta"])
    assert ret.shape == gold["ret_arr"].shape and retd.shape == gold["ret_arr_ddim"].shape
    assert torch.equal(y[~m], data["gt"][~m]) and torch.equal(yd[~m], data["gt"][~m])  # outside the mask: y_0 exactly
    with _Emulated(), torch.no_grad():
        yo, reto = O.restoration_ddpm(params, data["cond"], y_t0, data["gt"], data["mask"], noises, cfg,
                                      gold["sample_num"])
        ydo, _ = O.restoration_ddim(params, data["cond"], y_t0, data["gt"], data["mask"], cfg, gold["sample_num"],
                                    num_steps=gold["ddim_steps"], eta=gold["ddim_eta"])
    assert rel_l2(y, gold["y"]) < max(3e-2, 2.5 * rel_l2(yo, gold["y"]))
    assert rel_l2(ret, gold["ret_arr"]) < max(3e-2, 2.5 * rel_l2(reto, gold["ret_arr"]))
    assert rel_l2(yd, gold["y_ddim"]) < max(3e-2, 2.5 * rel_l2(ydo, gold["y_ddim"]))


@pytest.mark.parametrize("conditioning", ["class", "mask", "class_mask"])
def test_conditioned_generator_on_the_double(golden_dir, conditioning):
    """--alg_diffusion_cond_embed class / mask / class_mask: LabelEmbedder + per-pixel mask embedding written into the
    UNet input, nn.Embedding(max_norm=1)'s in-place renormalisation, scatter-add backward."""
    from joligen_b200 import nets
    from oracle import palette_oracle as O
    from oracle.gen_golden_cond import BASE, cond_batch, cond_cfg, cond_params
    g = torch.load(os.path.join(golden_dir, "palette_cond_%s.pt" % conditioning))
    cfg = cond_cfg(conditioning, g["nclasses"])
    params = cond_params(cfg, g["wseed"])
    net = nets.build_palette_generator(conditioning=conditioning, nclasses=g["nclasses"], **BASE)
    missing, unexpected = net.load_state_dict(params, strict=False)
    assert not unexpected and all("gammas" in m or "posterior" in m for m in missing)
    data = cond_batch(cfg, g["batch"], g["dseed"])
    torch.manual_seed(g["rseed"])
    t, u = O.sample_t_gamma(cfg, g["batch"])
    noise = torch.randn_like(data["gt"])
    cls = data["cls"] if "class" in conditioning else None
    with KD.installed():
        _, noise_hat, _ = net(data["gt"], data["cond"], data["mask"], noise, cls=cls, t=t, u=u)
        assert rel_l2(noise_hat, g["noise_hat"]) < 4e-2
        sd = net.state_dict()
        for k, ref in g["tables_after"].items():
            assert torch.allclose(sd[k], ref, atol=1e-6), k
        net.load_state_dict(params, strict=False)
        loss = net.forward_loss(data["gt"], data["cond"], data["mask"], noise=noise, cls=cls, t=t, u=u)
        assert abs(float(loss.detach()) - g["loss"]) < 1e-2 * abs(g["loss"])
        loss.backward()
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    with _Emulated():
        _, nh_e, _ = O.diffusion_forward(leaves, data["gt"], data["cond"], data["mask"], noise, t, u, cfg, cls=cls)
        O.palette_loss(noise, nh_e, data["mask"]).backward()
    floor = 1e-3 * max(n for _, n in g["grad_stats"].values())
    named = dict(net.named_parameters())
    for k, p in named.items():
        assert p.grad is not None, k
        _, gnorm = g["grad_stats"][k]
        emu = abs(float(leaves[k].grad.double().norm()) - gnorm) / (gnorm + 1e-30)
        assert abs(float(p.grad.double().norm()) - gnorm) <= max(6e-2, 2.5 * emu) * gnorm + floor, k
    for k, ref in g["grads"].items():
        rn = float(ref.double().norm())
        emu = float((leaves[k].grad.double() - ref.double()).norm()) / rn
        assert float((named[k].grad.double() - ref.double()).norm()) <= max(6e-2, 2.5 * emu) * rn + floor, (k, emu)


def _check_unet_grads(named, leaves, gold):
    scale = max(g["l2"] for g in gold["grads"].values())
    for k, g in gold["grads"].items():
        mine = named[k].grad.detach().double()
        ref = leaves[k].grad.double()
        err = float((mine - ref).norm()) / max(float(ref.norm()), 2e-2 * scale)
        emu = abs(float(ref.norm()) - g["l2"]) / max(g["l2"], 2e-2 * scale)  # emulation vs fp32 reference
        assert err < max(8e-2, 3 * emu), (k, err, emu)


def test_refattn_unet_on_the_double(golden_dir):
    """UNetGeneratorRefAttn: two UNets, every attention block of the main one attends to its own and to the reference
    UNet's keys / values (mix_qkv, both results in the halves of one buffer, proj_out 2C -> C)."""
    from oracle import palette_oracle as O
    from oracle import ref_oracle as R
    from oracle.gen_golden_ref import inputs
    from oracle.vid_oracle import init_params_from_shapes
    from test_ref_oracle import build_b200
    gold = torch.load(os.path.join(golden_dir, "refattn_small.pt"))
    cfg = O.UNetCfg(**gold["cfg"])
    params = init_params_from_shapes(gold["shapes"], gold["wseed"])
    x, ref, emb, gy = inputs(cfg, gold["batch"], gold["dseed"])
    net = build_b200(cfg)
    missing, unexpected = net.load_state_dict(params, strict=False)
    assert not missing and not unexpected
    with KD.installed():
        y = net(x, emb, ref)
        (y * gy).sum().backward()
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    with _Emulated():
        yo = R.unet_ref_forward(leaves, x, emb, ref, cfg)
        (yo * gy).sum().backward()
    floor = rel_l2(yo, gold["y"])
    assert rel_l2(y, gold["y"]) < max(3e-2, 2 * floor) and rel_l2(y, yo) < max(3e-2, 2 * floor)
    _check_unet_grads(dict(net.named_parameters()), leaves, gold)


def test_video_unet_on_the_double(golden_dir):
    """UNetVid: clips folded to B*F frames, per-clip embeddings repeated per frame, MotionModules (LayerNorm + frame
    positional encoding, temporal attention over the frames of each pixel, GEGLU feed-forward) as 1x1 convolutions."""
    from joligen_b200 import nets_vid
    from oracle import vid_oracle as V
    from oracle.gen_golden_vid import inputs
    gold = torch.load(os.path.join(golden_dir, "vid_small.pt"))
    cfg = V.VidCfg(**gold["cfg"])
    params = V.init_params_from_shapes(gold["shapes"], gold["wseed"])
    x, emb, gy = inputs(cfg, gold["batch"], gold["frames"], gold["dseed"])
    net = nets_vid.UNetVid(image_size=cfg.image_size, in_channel=cfg.in_channel, inner_channel=cfg.inner_channel,
                           out_channel=cfg.out_channel, res_blocks=list(cfg.res_blocks), attn_res=list(cfg.attn_res),
                           tanh=False, n_timestep_train=cfg.n_timestep_train, n_timestep_test=cfg.n_timestep_test,
                           norm="groupnorm", group_norm_size=cfg.group_norm_size, cond_embed_dim=cfg.cond_embed_dim,
                           channel_mults=cfg.channel_mults, num_heads=cfg.num_heads,
                           num_head_channels=cfg.num_head_channels, max_sequence_length=cfg.max_sequence_length,
                           num_attention_heads=cfg.num_attention_heads,
                           num_transformer_blocks=cfg.num_transformer_blocks)
    missing, unexpected = net.load_state_dict(params, strict=False)
    assert not unexpected and all(m.endswith("pos_encoder.pe") for m in missing)
    with KD.installed():
        y = net(x, emb)
        (y * gy).sum().backward()
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    with _Emulated():
        yo = V.unet_vid_forward(V.add_buffers(leaves, cfg), x, emb, cfg)
        (yo * gy).sum().backward()
    floor = rel_l2(yo, gold["y"])
    assert rel_l2(y, gold["y"]) < max(3e-2, 2 * floor) and rel_l2(y, yo) < max(3e-2, 2 * floor)
    _check_unet_grads(dict(net.named_parameters()), leaves, gold)


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
@pytest.mark.parametrize("which", ["ref", "vid"])
def test_reference_palette_model_cfg4_cfg5_trains_with_accelerated_generator(golden_dir, which):
    """The unmodified reference's control path for BASELINE config 4 (unet_mha_ref_attn with ref_A) and config 5
    (unet_vid, 3-frame clips) with `accelerate(netG_A)`: two optimize_parameters() vs the reference's own
    (refattn_plumbing.pt / vid_plumbing.pt), seeded identically (the video noise is drawn on the folded clip)."""
    from oracle import ref_stubs
    ref_stubs.install()
    from oracle import gen_golden_plumbing45 as P
    import joligen_b200
    from joligen_b200 import nets, nets_ref, nets_vid
    gold = torch.load(os.path.join(golden_dir, "vid_plumbing.pt" if which == "vid" else "refattn_plumbing.pt"))
    model, _, _, _, _ = P.create_reference_model(which)
    ref_params = dict(model.netG_A.named_parameters())
    model.netG_A = joligen_b200.accelerate(model.netG_A)
    assert isinstance(model.netG_A, nets.DiffusionGenerator)
    assert isinstance(model.netG_A.denoise_fn.model, nets_vid.UNetVid if which == "vid" else nets_ref.UNetGeneratorRefAttn)
    assert all(p is ref_params[k] for k, p in model.netG_A.named_parameters())
    losses = []
    with KD.installed():
        for step in range(2):
            data = P.batch(which, gold["data_seeds"][step])
            model.set_input(dict(data, A_img_paths=["a"] * P.BATCH, B_label_cls=torch.zeros(P.BATCH, dtype=torch.long)))
            torch.manual_seed(gold["rng_seeds"][step])
            model.optimize_parameters()
            losses.append(float(model.loss_G_tot.detach()))
    for got, want in zip(losses, gold["losses"]):
        assert abs(got - want) < 3e-2 * abs(want), (losses, gold["losses"])
    sd, ema = model.netG_A.state_dict(), model.netG_A_ema.state_dict()
    for k, (_, n) in gold["param_stats"].items():
        assert abs(float(sd[k].double().norm()) - n) <= 2e-2 * n + 1e-6, k
    for k, (_, n) in gold["ema_stats"].items():
        assert abs(float(ema[k].double().norm()) - n) <= 2e-2 * n + 1e-6, k


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
@pytest.mark.parametrize("which", ["ref", "vid"])
def test_reference_inference_cfg4_cfg5_with_accelerated_generator(which):
    """PaletteModel.inference for the reference-image UNet (its `use_ref` branch: restoration(..., ref=cur_ref)) and for
    video clips (5-D y_cond / y_t / mask: B*F frames through the UNet and the step kernel, one noise level per clip, the
    draws in the reference's 5-D shape) on the accelerated generator == the reference's own sampling, same seeds."""
    import contextlib
    from oracle import ref_stubs
    ref_stubs.install()
    from oracle import gen_golden_plumbing45 as P
    from models.modules.diffusion_utils import set_new_noise_schedule
    import joligen_b200
    outs = []
    for fast in (False, True):
        model, _, _, _, _ = P.create_reference_model(which)
        model.netG_A.denoise_fn.model.beta_schedule["test"]["n_timestep"] = 6
        set_new_noise_schedule(model.netG_A.denoise_fn.model, "test")
        if fast:
            model.netG_A = joligen_b200.accelerate(model.netG_A)
        torch.manual_seed(7)
        model.set_input(dict(P.batch(which, 200), A_img_paths=["a"] * P.BATCH,
                             B_label_cls=torch.zeros(P.BATCH, dtype=torch.long)))
        with (KD.installed() if fast else contextlib.nullcontext()), torch.no_grad():
            torch.manual_seed(8)
            model.inference(2)
        outs.append(model.fake_B.clone())
    assert outs[0].shape == outs[1].shape and outs[0].dim() == (5 if which == "vid" else 4)
    assert rel_l2(outs[1], outs[0]) < 3e-2, rel_l2(outs[1], outs[0])


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
@pytest.mark.parametrize("cond", ["class", "class_mask"])
def test_reference_palette_model_with_conditioning_trains_with_accelerated_generator(cond):
    """--alg_diffusion_cond_embed class / class_mask (example_ddpm_mario.json ships `class`) through the reference's own
    optimize_parameters(): B_label_cls / the semantic mask reach the accelerated generator's label embeddings; two steps
    of the accelerated model == two steps of the untouched one, same seeds."""
    import contextlib
    import copy
    from oracle import ref_stubs
    ref_stubs.install()
    from oracle import gen_golden
    from oracle import palette_oracle as O
    import joligen_b200
    losses = []
    for fast in (False, True):
        torch.manual_seed(3)
        model, _ = gen_golden.create_reference_model(32, 2, extra={"alg_diffusion_cond_embed": cond,
                                                                   "f_s_semantic_nclasses": 4, "cls_semantic_nclasses": 4,
                                                                   "alg_diffusion_dropout_prob": 0.0})
        with torch.no_grad():   # de-zero the reference's zero-initialised convolutions
            g = torch.Generator().manual_seed(11)
            for p in model.netG_A.parameters():
                if float(p.abs().max()) == 0.0:
                    p.copy_(torch.randn(p.shape, generator=g) * 0.05)
        if fast:
            model.netG_A = joligen_b200.accelerate(model.netG_A)
            assert model.netG_A.denoise_fn.conditioning == cond
        ls = []
        with (KD.installed() if fast else contextlib.nullcontext()):
            for step in range(2):
                data = O.synthetic_batch(2, 32, 100 + step)
                mask = (data["mask"] * torch.tensor([1, 2]).view(2, 1, 1, 1)).long()
                model.set_input({"A": data["cond"], "B": data["gt"], "B_label_mask": mask,
                                 "B_label_cls": torch.tensor([1, 2]), "A_img_paths": ["a"] * 2})
                torch.manual_seed(1000 + step)
                model.optimize_parameters()
                ls.append(float(model.loss_G_tot.detach()))
        losses.append(ls)
    for got, want in zip(losses[1], losses[0]):
        assert abs(got - want) < 2e-2 * abs(want), losses
