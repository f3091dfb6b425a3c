"""Goldens for accelerate() on modules built by the UNMODIFIED reference (TEST INFRASTRUCTURE — see oracle/__init__.py).

    python -m oracle.gen_golden_accelerate       # writes tests/golden/accel_*.pt (needs the reference tree)

Each file holds a reference module as built (oracle/skeleton.py: the reference's classes as named stand-ins, every
attribute, parameter and buffer kept), the inputs, and what the reference modules computed from them in fp32 on the
CPU: outputs, encoder features and gradients (a fixed, seeded sample of each: `sample`) and the spectral-norm buffers after a
training-mode forward.  Weights are seeded (oracle/skeleton.py: seed_, or the oracles' seeded state_dicts).
tests/test_host_double.py and tests/test_host_double_cut.py swap the stored modules
with accelerate() and compare the B200 mirrors against those values.
"""
import copy
import functools
import os
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_stubs  # noqa: E402
from oracle import skeleton  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
UNET_VARIANT_BASE = dict(image_size=32, inner_channel=32, channel_mults=(1, 2), res_blocks=(1, 1), attn_res=(2,),
                         num_head_channels=16)


def _instance_norm():
    return functools.partial(nn.InstanceNorm2d, affine=False, track_running_stats=False)


def _save(name, obj):
    skeleton.save(obj, os.path.join(GOLDEN, "accel_%s.pt" % name))


def sample(t, n=1024):
    """A fixed, seeded sample of n elements of t (all of them when t is smaller): stored gradients stay small."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= n:
        return flat.clone()
    return flat[sample_index(flat.numel(), n)]


def sample_index(numel, n=1024):
    return torch.randperm(numel, generator=torch.Generator().manual_seed(0))[:n]


def _grads(m):
    return {k: sample(p.grad) for k, p in m.named_parameters() if p.grad is not None}


def gen_gan_nets():
    from models.modules.discriminators import NLayerDiscriminator
    from models.modules.resnet_architecture.resnet_generator import ResnetGenerator
    from oracle import gan_oracle as G
    norm = _instance_norm()
    for name, ref, shapes in (
            ("resnet", ResnetGenerator(3, 3, 16, norm_layer=norm, use_dropout=False, n_blocks=2),
             G.resnet_param_shapes(3, 3, 16, 2)),
            ("nlayerd", NLayerDiscriminator(3, 16, n_layers=3, norm_layer=norm), G.nlayer_d_param_shapes(3, 16, 3))):
        ref.load_state_dict(G.init_from_shapes(shapes, 77))
        keep = copy.deepcopy(ref)
        x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1))
        y = ref(x)
        dy = torch.randn(y.shape, generator=torch.Generator().manual_seed(2))
        y.backward(dy)
        case = {"module": keep, "y": y.detach(), "grads": _grads(ref)}
        if name == "resnet":
            with torch.no_grad():
                case["feats"] = [(tuple(f.shape), sample(f)) for f in ref.get_feats(x, [0, 4, 8, 11])]
        _save("gan_" + name, case)
    # variants the mirrors do not implement (accelerate() must refuse them)
    _save("gan_refused", [ResnetGenerator(3, 3, 16, norm_layer=nn.BatchNorm2d, n_blocks=2),
                          ResnetGenerator(3, 3, 16, norm_layer=norm, n_blocks=2, mobile=True),
                          NLayerDiscriminator(3, 16, n_layers=3, norm_layer=norm, use_dropout=True)])


def gen_unet_variant(name, variant):
    from oracle import palette_oracle as O
    from models.modules.diffusion_generator import DiffusionGenerator
    from models.modules.palette_denoise_fn import PaletteDenoiseFn
    from models.modules.unet_generator_attn.unet_generator_attn import UNet
    cfg = O.UNetCfg(**UNET_VARIANT_BASE, **variant)
    unet = UNet(image_size=cfg.image_size, in_channel=cfg.in_channel, inner_channel=cfg.inner_channel,
                out_channel=cfg.out_channel, res_blocks=list(cfg.res_blocks), attn_res=list(cfg.attn_res), tanh=False,
                n_timestep_train=cfg.n_timestep_train, n_timestep_test=cfg.n_timestep_test, norm="groupnorm",
                group_norm_size=cfg.group_norm_size, cond_embed_dim=cfg.cond_embed_dim, channel_mults=cfg.channel_mults,
                num_heads=cfg.num_heads, num_head_channels=cfg.num_head_channels, efficient=cfg.efficient,
                use_scale_shift_norm=cfg.use_scale_shift_norm)
    ref = DiffusionGenerator(denoise_fn=PaletteDenoiseFn(model=unet, cond_embed_dim=cfg.cond_embed_dim, ref_embed_net="",
                                                         conditioning="", nclasses=2),
                             sampling_method="ddpm", image_size=cfg.image_size, G_ngf=cfg.inner_channel,
                             loading_backward_compatibility=False)
    ref.load_state_dict(O.init_params(cfg, 5), strict=False)
    keep = copy.deepcopy(ref)
    data = O.synthetic_batch(2, cfg.image_size, 9)
    torch.manual_seed(1)
    noise, noise_hat, _ = ref(data["gt"], data["cond"], data["mask"], None, None, None)
    torch.nn.functional.mse_loss(noise * data["mask"].clamp(0, 1), noise_hat * data["mask"].clamp(0, 1)).backward()
    _save("unet_" + name, {"module": keep, "noise": noise.detach(), "noise_hat": noise_hat.detach(),
                           "grads": _grads(ref)})


def gen_norm_variants():
    from models.modules.unet_generator_attn.unet_generator_attn import UNet
    for norm in ("instancenorm", "layernorm", "groupnorm"):
        torch.manual_seed(0)
        ref = UNet(image_size=32, in_channel=6, inner_channel=32, out_channel=3, res_blocks=[1, 1], attn_res=[2],
                   tanh=False, n_timestep_train=2000, n_timestep_test=1000, norm=norm, group_norm_size=8,
                   cond_embed_dim=32, channel_mults=(1, 2), num_heads=1, num_head_channels=16)
        skeleton.seed_(ref, 3)
        keep = copy.deepcopy(ref)
        x = torch.randn(2, 6, 32, 32)
        emb = torch.randn(2, 32)
        with torch.no_grad():
            _save("norm_" + norm, {"module": keep, "x": x, "emb": emb, "y": ref(x, emb)})


def gen_resnet_padding():
    from models.modules.resnet_architecture.resnet_generator import ResnetGenerator
    from oracle import gan_oracle as G
    for padding_type in ("replicate", "zeros"):
        ref = ResnetGenerator(3, 3, 16, norm_layer=_instance_norm(), use_dropout=False, n_blocks=2,
                              padding_type=padding_type)
        seeded = list(G.init_from_shapes(G.resnet_param_shapes(3, 3, 16, 2), 77).values())
        ref.load_state_dict(dict(zip(ref.state_dict().keys(), seeded)))
        keep = copy.deepcopy(ref)
        x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1))
        xr = x.clone().requires_grad_(True)
        y = ref(xr)
        dy = torch.randn(y.shape, generator=torch.Generator().manual_seed(2))
        y.backward(dy)
        with torch.no_grad():
            feats = [(tuple(f.shape), sample(f)) for f in ref.get_feats(x, [0, 4, 8, 11])]
        _save("resnet_padding_" + padding_type,
              {"module": keep, "y": y.detach(), "x_grad": xr.grad, "feats": feats})


def gen_wavelet():
    from models.modules.discriminators import NLayerDiscriminator
    from models.modules.unet_generator_attn.unet_generator_attn import UNet
    torch.manual_seed(0)
    ref = UNet(image_size=32, in_channel=6, inner_channel=32, out_channel=3, res_blocks=[1, 1], attn_res=[2], tanh=False,
               n_timestep_train=2000, n_timestep_test=1000, norm="groupnorm", group_norm_size=8, cond_embed_dim=32,
               channel_mults=(1, 2), num_heads=1, num_head_channels=16, freq_space=True)
    skeleton.seed_(ref, 3)
    keep = copy.deepcopy(ref)
    x = torch.randn(1, 6, 32, 32)
    emb = torch.randn(1, 32)
    xr = x.clone().requires_grad_(True)
    y = ref(xr, emb)
    dy = torch.randn_like(y)
    y.backward(dy)
    unet = {"module": keep, "x": x, "emb": emb, "dy": dy, "y": y.detach(), "x_grad": xr.grad}
    torch.manual_seed(1)
    ref = skeleton.seed_(NLayerDiscriminator(3, 16, n_layers=3, norm_layer=_instance_norm(), freq_space=True), 4)
    keep = copy.deepcopy(ref)
    x = torch.randn(2, 3, 128, 128)
    with torch.no_grad():
        disc = {"module": keep, "x": x, "y": ref(x)}
    _save("wavelet_unet", unet)
    _save("wavelet_nlayerd", disc)


def gen_spectral():
    from models.modules.discriminators import NLayerDiscriminator
    from models.modules.resnet_architecture.resnet_generator import ResnetGenerator
    for name, seed, build, size in (
            ("nlayerd", 2, lambda: NLayerDiscriminator(3, 16, n_layers=3, norm_layer=_instance_norm(), use_spectral=True),
             96),
            ("resnet", 4, lambda: ResnetGenerator(3, 3, 16, norm_layer=_instance_norm(), use_dropout=False, n_blocks=2,
                                                  use_spectral=True), 64)):
        torch.manual_seed(seed)
        ref = skeleton.seed_(build(), seed).train()
        keep = copy.deepcopy(ref)
        x = torch.randn(2, 3, size, size)
        y = ref(x)
        dy = torch.randn_like(y)
        y.backward(dy)
        _save("spectral_" + name, {"module": keep, "x": x, "dy": dy, "y": y.detach(), "grads": _grads(ref),
                                   "uv_after": {k: v.detach().clone() for k, v in ref.state_dict().items()
                                                if k.endswith(("weight_u", "weight_v"))}})


def gen_projected_heads():
    from models.modules.projected_d.discriminator import MultiScaleD
    from oracle.gen_golden_projd import CHANNELS, RESOLUTIONS, features, seeded_state
    gold = torch.load(os.path.join(GOLDEN, "projd_small.pt"))
    ref = MultiScaleD(channels=CHANNELS, resolutions=RESOLUTIONS, conv=True, feats=None, num_discs=2, proj_type=2, cond=0)
    ref.load_state_dict(seeded_state(gold["shapes"], gold["wseed"]))
    ref.train()
    keep = copy.deepcopy(ref)
    with torch.no_grad():
        y = ref(features(gold["fseed"]))
    _save("projd_heads", {"module": keep, "y": y, "uv_after": {k: v.clone() for k, v in ref.state_dict().items()
                                                               if k.endswith(("weight_u", "weight_v"))}})


def main():
    ref_stubs.install()
    torch.set_num_threads(4)
    gen_gan_nets()
    gen_unet_variant("efficient", dict(efficient=True))
    gen_unet_variant("no_scale_shift", dict(use_scale_shift_norm=False))
    gen_norm_variants()
    gen_resnet_padding()
    gen_wavelet()
    gen_spectral()
    gen_projected_heads()


if __name__ == "__main__":
    main()
