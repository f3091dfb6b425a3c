"""Host-side logic of the B200 path that needs no GPU: flat parameter buffers, strided-view acceptance, concat
geometry, weight-tile accounting of the batched pack / unpack launches, gradient-stamp slicing."""
import torch
import torch.nn as nn


def test_flat_params_views_alignment_and_rebind():
    from joligen_b200.trainer import FlatParams
    net = nn.Sequential(nn.Linear(5, 7), nn.Conv2d(3, 6, 3), nn.GroupNorm(2, 6))
    before = {k: v.detach().clone() for k, v in net.named_parameters()}
    flat = FlatParams(net)
    assert flat.total % 64 == 0 and all(o % 64 == 0 for o in flat.offsets)   # 256-byte aligned slices
    for (k, p), o in zip(net.named_parameters(), flat.offsets):
        assert torch.equal(p.detach(), before[k])                            # values kept
        assert p.data_ptr() == flat.data.data_ptr() + 4 * o                  # parameters ARE views of the buffer
        assert p.grad.data_ptr() == flat.grad.data_ptr() + 4 * o
    # an optimizer-style in-place update of the flat buffer is visible through the module
    flat.data.add_(1.0)
    assert torch.allclose(net[0].weight.detach(), before["0.weight"] + 1.0)
    # autograd accumulates into the flat gradient; a dropped .grad is re-bound to the same slice
    net[0](torch.ones(2, 5)).sum().backward()
    assert float(flat.grad.abs().sum()) > 0
    net[0].weight.grad = None
    flat.rebind_grads()
    assert net[0].weight.grad.data_ptr() == flat.grad.data_ptr() + 4 * flat.offsets[0]
    un = flat.unflatten(flat.data)
    assert list(un.keys()) == [k for k, _ in net.named_parameters()]
    assert all(un[k].shape == p.shape for k, p in net.named_parameters())


def test_rows_accepts_channel_slices_and_copies_the_rest():
    from joligen_b200.ops import _rows
    buf = torch.zeros(2, 4, 4, 32, dtype=torch.bfloat16)
    assert _rows(buf) is buf
    s = buf[..., 8:24]                       # channel slice: unit channel stride, uniform row stride, aligned start
    assert _rows(s) is s
    assert _rows(buf[..., 4:20]).is_contiguous()          # start not 16-byte aligned -> copied
    assert _rows(buf[:, ::2]).is_contiguous()             # rows not uniformly strided -> copied
    assert _rows(buf.permute(0, 3, 1, 2)).is_contiguous()  # NCHW view -> copied
    odd = torch.zeros(2, 4, 4, 20, dtype=torch.bfloat16)[..., :16]   # row stride 20: not a multiple of 8
    assert _rows(odd).is_contiguous()


def test_colsum_stamp_follows_channel_slices_and_dies_with_inplace_updates():
    from joligen_b200.ops import _slice_with_stamp
    d = torch.zeros(1, 2, 2, 16)
    colsum = torch.arange(16.0)
    d._jg_colsum = (colsum, d._version)
    v = _slice_with_stamp(d, 8, 16)
    assert torch.equal(v._jg_colsum[0], colsum[8:16]) and v._jg_colsum[1] == v._version
    d.add_(1.0)                               # autograd accumulated another gradient INTO d: the sums are stale
    assert not hasattr(_slice_with_stamp(d, 0, 8), "_jg_colsum")


def test_weight_tile_accounting():
    """jg_weight_tiles (host function of the C ABI) = the grid of the batched pack / unpack kernels: 32 co x 32 ci x 9
    taps per tile, and for 1x1 weights 32 co x (9 x 32) ci."""
    from joligen_b200 import lib
    l = lib.load()
    assert l.jg_weight_tiles(64, 64, 9) == 2 * 2 * 1
    assert l.jg_weight_tiles(128, 192, 9) == 4 * 6
    assert l.jg_weight_tiles(64, 64, 16) == 2 * 2 * 2          # 4x4 filters: two tap chunks
    assert l.jg_weight_tiles(64, 6, 9) == 2 * 1                # ragged Cin
    assert l.jg_weight_tiles(512, 512, 1) == 16 * 2            # 1x1: 288-channel ci spans
    assert l.jg_weight_tiles(4096, 512, 1) == 128 * 2
    assert l.jg_weight_tiles(64, 288, 1) == 2 and l.jg_weight_tiles(64, 289, 1) == 4


def test_concat_geometry_and_token_grid():
    from joligen_b200 import nets
    from joligen_b200.nets_cut import _token_grid
    g = nets.build_palette_generator(image_size=32, inner_channel=32, channel_mults=(1, 2), res_blocks=(1, 1),
                                     attn_res=(2,), num_head_channels=16)
    unet = g.denoise_fn.model
    assert unet.input_blocks[1].out_geometry(32, 32) == (32, 32, 32)         # ResBlock keeps the size
    assert unet.input_blocks[2].out_geometry(32, 32) == (16, 16, 32)         # downsampling ResBlock
    assert unet.input_blocks[0].out_geometry(32, 32) is None                 # plain conv: no view destination
    assert unet.output_blocks[-1].out_geometry(32, 32) == (32, 32, 32)
    assert unet.output_blocks[1].out_geometry(16, 16) == (32, 32, 64)        # ResBlock + attention + upsample
    assert _token_grid(4096) == (256, 16) and _token_grid(24) == (3, 8) and _token_grid(7) == (7, 1)


def test_denoise_fn_argument_count_drives_the_reference_image_path():
    from joligen_b200 import nets, nets_ref, nets_vid
    kw = dict(image_size=16, in_channel=6, inner_channel=32, out_channel=3, res_blocks=[1, 1], attn_res=[2],
              tanh=False, n_timestep_train=10, n_timestep_test=5, norm="groupnorm", group_norm_size=32,
              cond_embed_dim=32, channel_mults=(1, 2), num_head_channels=16)
    assert nets.PaletteDenoiseFn(nets.UNet(**kw), 32).model_nargs == 2
    assert nets.PaletteDenoiseFn(nets_vid.UNetVid(**kw), 32).model_nargs == 2
    dn = nets.PaletteDenoiseFn(nets_ref.UNetGeneratorRefAttn(**kw), 32)
    assert dn.model_nargs == 3
    import pytest
    with pytest.raises(RuntimeError):
        dn.pack_ref(None)                     # the three-argument UNet needs the reference image
    assert nets.PaletteDenoiseFn(nets.UNet(**kw), 32).pack_ref(None) is None


def test_no_undefined_names_in_the_package():
    """A forgotten import in a rarely taken branch is exactly what no GPU test reaches (nets.py once used `F.pad`
    without importing `F`): tools/undefined_names.py resolves every loaded name of every product module."""
    import glob
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("undefined_names", os.path.join(root, "tools", "undefined_names.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    files = sorted(glob.glob(os.path.join(root, "joligen_b200", "*.py"))) + [
        os.path.join(root, "bench.py"), os.path.join(root, "__graft_entry__.py"),
        os.path.join(root, "baseline", "ref_runner.py"), os.path.join(root, "oracle", "install_ref.py")]
    bad = []
    for f in files:
        bad += ["%s:%d %s" % (os.path.relpath(f, root), line, name) for line, name in mod.check_source(open(f).read(), f)]
    assert not bad, bad


def test_checkers_are_imported_only_where_the_contract_allows():
    """oracle/ (the CPU restatement) and tests/kernel_double.py are CHECKERS: only tests/, __graft_entry__.smoke() and
    bench.py's CPU-baseline legs may import them — never the product package, the tools, or the reference arm's runner."""
    import glob
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    allowed = {"bench.py", "__graft_entry__.py"}
    bad = []
    for f in glob.glob(os.path.join(root, "**", "*.py"), recursive=True):
        rel = os.path.relpath(f, root)
        if rel.startswith(("tests" + os.sep, "oracle" + os.sep)) or rel in allowed:
            continue
        src = open(f).read()
        if re.search(r"^\s*(from|import)\s+(oracle|kernel_double)\b", src, re.M):
            bad.append(rel)
    assert not bad, bad
    # the product package never mentions the double
    for f in glob.glob(os.path.join(root, "joligen_b200", "*.py")):
        assert "kernel_double" not in open(f).read(), f
