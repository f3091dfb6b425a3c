"""accelerate() on a network built by the UNMODIFIED reference (only where /root/reference exists,
i.e. in the build container): the swapped tree shares the reference's Parameter objects and keeps
its state_dict keys.  (CPU only: no kernels are launched.)"""
import os

import pytest
import torch

from oracle import ref_stubs  # noqa: E402

REF_MISSING = "needs the reference's own code: build() stages it under oracle/_ref where the checkout is readable"



@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
def test_accelerate_adopts_reference_parameters():
    from oracle import ref_stubs
    ref_stubs.install()
    from oracle import gen_golden
    from oracle import palette_oracle as O
    from joligen_b200 import accelerate, nets
    cfg = O.UNetCfg(**gen_golden.SMALL)
    ref_net = gen_golden.build_reference_generator(cfg)
    ref_params = dict(ref_net.named_parameters())
    ref_keys = list(ref_net.state_dict().keys())
    fast = accelerate(ref_net)
    assert isinstance(fast, nets.DiffusionGenerator)
    assert list(fast.state_dict().keys()) == ref_keys
    for k, p in fast.named_parameters():
        assert p is ref_params[k]  # same Parameter objects: optimizers / DDP built on the reference still apply
    # a reference wrapper that merely CONTAINS a UNet gets the child swapped in place
    holder = torch.nn.Module()
    holder.netG = gen_golden.build_reference_generator(cfg).denoise_fn.model
    accelerate(holder)
    assert isinstance(holder.netG, nets.UNet)


@pytest.mark.skipif(not ref_stubs.available(), reason=REF_MISSING)
def test_accelerate_video_and_reference_attention_unets():
    """Rows a-16..a-18: the reference's UNetVid / UNetGeneratorRefAttn objects are swapped for the B200 mirrors,
    which adopt the reference's Parameter objects (incl. the MotionModule's positional-encoding buffers)."""
    from oracle import ref_stubs
    ref_stubs.install()
    from oracle import gen_golden_ref, gen_golden_vid
    from oracle import palette_oracle as O
    from oracle import vid_oracle as V
    from joligen_b200 import accelerate, nets_ref, nets_vid
    ref_vid = gen_golden_vid.build_reference(V.VidCfg(**gen_golden_vid.CFG))
    params, keys = dict(ref_vid.named_parameters()), list(ref_vid.state_dict().keys())
    fast = accelerate(ref_vid)
    assert isinstance(fast, nets_vid.UNetVid) and list(fast.state_dict().keys()) == keys
    assert all(p is params[k] for k, p in fast.named_parameters())
    ref_ra = gen_golden_ref.build_reference(O.UNetCfg(**gen_golden_ref.CFG))
    params, keys = dict(ref_ra.named_parameters()), list(ref_ra.state_dict().keys())
    fast = accelerate(ref_ra)
    assert isinstance(fast, nets_ref.UNetGeneratorRefAttn) and list(fast.state_dict().keys()) == keys
    assert all(p is params[k] for k, p in fast.named_parameters())
    # whole generators (cfg 4 / cfg 5): DiffusionGenerator(PaletteDenoiseFn(<those UNets>))
    from models.modules.diffusion_generator import DiffusionGenerator
    from models.modules.palette_denoise_fn import PaletteDenoiseFn
    from joligen_b200 import nets
    for unet, kind, nargs in ((gen_golden_vid.build_reference(V.VidCfg(**gen_golden_vid.CFG)), nets_vid.UNetVid, 2),
                              (gen_golden_ref.build_reference(O.UNetCfg(**gen_golden_ref.CFG)),
                               nets_ref.UNetGeneratorRefAttn, 3)):
        dn = PaletteDenoiseFn(model=unet, cond_embed_dim=32, ref_embed_net="", conditioning="", nclasses=2)
        gen = DiffusionGenerator(denoise_fn=dn, sampling_method="ddpm", image_size=32, G_ngf=64,
                                 loading_backward_compatibility=False)
        params, keys = dict(gen.named_parameters()), list(gen.state_dict().keys())
        fast = accelerate(gen)
        assert isinstance(fast, nets.DiffusionGenerator) and isinstance(fast.denoise_fn.model, kind)
        assert fast.denoise_fn.model_nargs == nargs == dn.model_nargs
        assert list(fast.state_dict().keys()) == keys
        assert all(p is params[k] for k, p in fast.named_parameters())
