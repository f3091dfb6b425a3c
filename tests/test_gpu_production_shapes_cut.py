"""Parity of the kernels the CUT benchmark step runs (bench.py --config 3: resnet_9blocks G, NLayerDiscriminator D,
PatchSampleF + MoNCE, 256x256, batch 4 per GPU), at the shapes that step runs them at.  The conv launchers pick a
kernel (generic implicit GEMM, halo, halo pair) and a template variant from the geometry, so toy shapes do not reach
the variants the benchmark uses: 7x7 filters on the reflect-padded 262x262 image, stride-2 4x4 and 3x3 filters, the
ResnetBlock's pad-0 3x3 on 66x66, the discriminator's ragged 32 -> 31 -> 30 maps, transposed convolutions.

Every case goes through the same ops the nets call (ops.reflection_pad, ops.conv_act, ops.conv_transpose2d, ...).
Reference: float64 torch on the same bf16-rounded operands.  Tolerances, as in test_gpu_production_shapes.py:
bf16 outputs within 1e-2 of the tensor's max, fp32 weight / bias gradients within 1e-3, scalar losses within 1e-5,
index / pad / copy work bit-exact.  The weight-gradient kernels read the activation gradient as ConvActFn stores it
(bf16, after act_bwd), so the dW / db reference starts from that stored operand; the dx reference is the plain
float64 chain.

test_cases_match_the_benchmark_step runs without a GPU: it records the kernel geometries of one bench.py config-3 step
on the kernel double and checks that the case lists below are exactly those geometries.
"""
import math
import os
import sys

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

BATCH = 4
SIZE = 256
NGF = NDF = 64

# (name, kind, cin, cout, k, stride, pad, reflect, act, input size): every distinct convolution of the config-3 step.
# kind "conv" = nn.Conv2d (+ the activation fused into its epilogue), "convT" = nn.ConvTranspose2d(3, s2, p1, op1);
# reflect = the ReflectionPad2d in front of it; input size = the map before that pad.
CONV_LAYERS = [
    ("G_stem", "conv", 3, NGF, 7, 1, 0, 3, "none", SIZE),
    ("G_down1", "conv", NGF, 2 * NGF, 3, 2, 1, 0, "none", SIZE),
    ("G_down2", "conv", 2 * NGF, 4 * NGF, 3, 2, 1, 0, "none", SIZE // 2),
    ("G_block", "conv", 4 * NGF, 4 * NGF, 3, 1, 0, 1, "none", SIZE // 4),
    ("G_up1", "convT", 4 * NGF, 2 * NGF, 3, 2, 1, 0, "none", SIZE // 4),
    ("G_up2", "convT", 2 * NGF, NGF, 3, 2, 1, 0, "none", SIZE // 2),
    ("G_out", "conv", NGF, 3, 7, 1, 0, 3, "tanh", SIZE),
    ("D_0", "conv", 3, NDF, 4, 2, 1, 0, "lrelu", SIZE),
    ("D_1", "conv", NDF, 2 * NDF, 4, 2, 1, 0, "none", SIZE // 2),
    ("D_2", "conv", 2 * NDF, 4 * NDF, 4, 2, 1, 0, "none", SIZE // 4),
    ("D_3", "conv", 4 * NDF, 8 * NDF, 4, 1, 1, 0, "none", SIZE // 8),
    ("D_4", "conv", 8 * NDF, 1, 4, 1, 1, 0, "none", SIZE // 8 - 1),
]
# G runs on cat(real_A, real_B) in the step (identity NCE: batch 8), its encoder alone on batch 4 for the NCE features,
# and on batch 1 in PatchSampleF's data_dependent_initialize
CONV_CASES = ([(n,) + layer for layer in CONV_LAYERS if layer[0].startswith("G") for n in (BATCH, 2 * BATCH, 1)]
              + [(BATCH,) + layer for layer in CONV_LAYERS if layer[0].startswith("D")])

# (C, size, act): every InstanceNorm (GroupNorm with groups == C) of the step; the ResnetBlock's second norm has no act
NORM_SHAPES = [(NGF, SIZE, "relu"), (2 * NGF, SIZE // 2, "relu"), (4 * NGF, SIZE // 4, "relu"),
               (4 * NGF, SIZE // 4, "none"), (2 * NDF, SIZE // 4, "lrelu"), (4 * NDF, SIZE // 8, "lrelu"),
               (8 * NDF, SIZE // 8 - 1, "lrelu")]
OFFSETS = [0.0, 4.0, 16.0]  # per-channel mean offset in standard deviations

# (C stored, size, pad): the reflection pads (image 3 -> 8 channels and the decoder's 64 channels at 256, ResnetBlocks)
PAD_CASES = [(8, SIZE, 3), (NGF, SIZE, 3), (4 * NGF, SIZE // 4, 1)]

NCE_LAYERS = [0, 4, 8, 12, 16]
NUM_PATCHES = 256
NC = 256
# (real channels, stored channels, size) of the encoder outputs at NCE_LAYERS: the padded image, the first stride-2
# conv, the second one's InstanceNorm+ReLU, ResnetBlocks 3 and 7
NCE_FEATS = [(3, 8, SIZE + 6), (2 * NGF, 2 * NGF, SIZE // 2), (4 * NGF, 4 * NGF, SIZE // 4),
             (4 * NGF, 4 * NGF, SIZE // 4), (4 * NGF, 4 * NGF, SIZE // 4)]


def _acts():
    from joligen_b200 import lib as L
    return {"none": L.ACT_NONE, "relu": L.ACT_RELU, "lrelu": L.ACT_LRELU02, "tanh": L.ACT_TANH}


@pytest.fixture(scope="module")
def K():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from joligen_b200 import kernels
    from joligen_b200 import lib
    assert lib.load().jg_check_device() == 0, lib.load().jg_last_error()
    return kernels


def rel(a, b):
    a, b = a.double(), b.double().to(a.device)
    return float((a - b).abs().max()) / (float(b.abs().max()) + 1e-30)


def close(what, a, b, tol):
    """rel(a, b) < tol; the error is printed (pytest -s) so that a run lists every margin"""
    err = rel(a, b)
    print("PARITY %-40s %.2e  (tol %.0e)" % (what, err, tol))
    assert err < tol, (what, err, tol)


def _nhwc(t_nchw, c8=None):
    """NCHW -> NHWC bf16, channels zero-padded to c8"""
    n, c, h, w = t_nchw.shape
    out = torch.zeros((n, h, w, c8 or c), dtype=torch.bfloat16, device=t_nchw.device)
    out[..., :c] = t_nchw.permute(0, 2, 3, 1).to(torch.bfloat16)
    return out


def _nchw(t_nhwc, c=None):
    t = t_nhwc.double().permute(0, 3, 1, 2)
    return t if c is None else t[:, :c]


def _act64(u, act):
    if act == "relu":
        return F.relu(u)
    if act == "lrelu":
        return F.leaky_relu(u, 0.2)
    if act == "tanh":
        return torch.tanh(u)
    return u


def _act_grad64(y, act):
    """d act / d u as a function of the activation's output (what act_bwd reads)"""
    if act == "relu":
        return (y > 0).double()
    if act == "lrelu":
        return torch.where(y > 0, 1.0, 0.2).double()
    if act == "tanh":
        return 1.0 - y * y
    return torch.ones_like(y)


def _c8(c):
    return (c + 7) // 8 * 8


def _make_module(kind, cin, cout, k, stride, pad, device):
    if kind == "convT":
        return nn.ConvTranspose2d(cin, cout, k, stride=stride, padding=pad, output_padding=1).to(device)
    return nn.Conv2d(cin, cout, k, stride=stride, padding=pad).to(device)


def _run_layer(layer_mod, kind, stride, pad, reflect, act, x_d):
    """the layer exactly as nets_gan._SeqRunner calls it"""
    from joligen_b200 import ops
    from joligen_b200.nets import ConvPack
    packed = ConvPack(layer_mod).get()
    h = ops.reflection_pad(x_d, reflect) if reflect else x_d
    if kind == "convT":
        return ops.conv_transpose2d(h, layer_mod.weight, layer_mod.bias, packed, pad=pad)
    return ops.conv_act(h, layer_mod.weight, layer_mod.bias, packed, stride=stride, pad=pad, act=_acts()[act])


@pytest.mark.gpu
@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "n%d_%s" % (c[0], c[1]))
def test_conv_cut_production_shape(K, case):
    """forward (+bias, +fused activation), dx, dW, db of one layer; padded output / input channels exactly zero"""
    n, name, kind, cin, cout, k, stride, pad, reflect, act, size = case
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(CONV_LAYERS.index(case[1:]) * 10 + n)
    rnd = lambda *shape: torch.randn(*shape, generator=g, device=dev, dtype=torch.float64)  # noqa: E731
    mod = _make_module(kind, cin, cout, k, stride, pad, dev)
    fan_in = mod.weight[0].numel() if kind == "conv" else cin * k * k
    with torch.no_grad():
        mod.weight.copy_((rnd(*mod.weight.shape) / math.sqrt(fan_in)).bfloat16())
        mod.bias.copy_(0.1 * rnd(cout))
    x = rnd(n, cin, size, size).bfloat16().double()

    # float64 reference
    xr = x.clone().requires_grad_(True)
    wr = mod.weight.detach().double().requires_grad_(True)
    br = mod.bias.detach().double().requires_grad_(True)
    h = F.pad(xr, (reflect,) * 4, mode="reflect") if reflect else xr
    if kind == "convT":
        u = F.conv_transpose2d(h, wr, br, stride=stride, padding=pad, output_padding=1)
    else:
        u = F.conv2d(h, wr, br, stride=stride, padding=pad)
    ref = _act64(u, act)
    dy = rnd(*ref.shape).bfloat16().double()
    ref.backward(dy)

    # the ops
    cin8, cout8 = _c8(cin), _c8(cout)
    x_d = _nhwc(x, cin8).requires_grad_(True)
    y = _run_layer(mod, kind, stride, pad, reflect, act, x_d)
    assert tuple(y.shape) == (n, ref.shape[2], ref.shape[3], cout8)
    close("y", _nchw(y, cout), ref.detach(), 1e-2)
    if cout8 != cout:
        assert float(y[..., cout:].float().abs().max()) == 0.0
    y.backward(_nhwc(dy, cout8))
    close("dx", _nchw(x_d.grad, cin), xr.grad, 1e-2)
    if cin8 != cin:
        assert float(x_d.grad[..., cin:].float().abs().max()) == 0.0
    dw_ref, db_ref = wr.grad, br.grad
    if act != "none":
        # the weight-gradient kernels read bf16(dy * act'(y)) as act_bwd stored it
        gs = (dy * _act_grad64(_nchw(y, cout), act)).bfloat16().double()
        dw_ref = torch.nn.grad.conv2d_weight(h.detach(), (cout, cin, k, k), gs, stride=stride, padding=pad)
        db_ref = gs.sum(dim=(0, 2, 3))
    close("dW", mod.weight.grad, dw_ref, 1e-3)
    close("db", mod.bias.grad, db_ref, 1e-3)


def _offset_input(g, n, c, size, offset, dev):
    """bf16 activations with a per-channel mean of `offset` standard deviations (std 0.5..2 per channel)"""
    std = 0.5 + 1.5 * torch.rand(1, c, 1, 1, generator=g, device=dev, dtype=torch.float64)
    sign = torch.where(torch.rand(1, c, 1, 1, generator=g, device=dev) < 0.5, -1.0, 1.0).double()
    z = torch.randn(n, c, size, size, generator=g, device=dev, dtype=torch.float64)
    return (std * (z + sign * offset)).bfloat16().double()


@pytest.mark.gpu
@pytest.mark.parametrize("offset", OFFSETS, ids=lambda o: "off%g" % o)
@pytest.mark.parametrize("shape", NORM_SHAPES, ids=lambda s: "c%d_%d_%s" % s)
def test_instance_norm_cut_production_shape(K, shape, offset):
    """InstanceNorm + act forward / backward through ops.group_norm (groups == C, no affine), the stand-alone chan_stats
    pass, and the statistics fused into a conv epilogue feeding the same norm"""
    from joligen_b200 import ops
    c, size, act = shape
    n, dev = BATCH, "cuda"
    g = torch.Generator(device=dev).manual_seed(c * 31 + size + int(offset))
    x = _offset_input(g, n, c, size, offset, dev)
    xr = x.clone().requires_grad_(True)
    ref = _act64(F.instance_norm(xr, eps=1e-5), act)
    dy = torch.randn(ref.shape, generator=g, device=dev, dtype=torch.float64).bfloat16().double()
    ref.backward(dy)
    x_d = _nhwc(x).requires_grad_(True)
    y = ops.group_norm(x_d, None, None, c, act=_acts()[act])
    close("y", _nchw(y), ref.detach(), 1e-2)
    y.backward(_nhwc(dy))
    close("dx", _nchw(x_d.grad), xr.grad, 1e-2)

    # per-(image, channel) sums: the stand-alone pass, and the norm fed by them
    xh = x_d.detach()
    want = torch.stack([x.sum(dim=(2, 3)), (x * x).sum(dim=(2, 3))], dim=-1)
    cs = K.chan_stats(xh)
    close("chan_stats", cs, want, 1e-4)
    y2, _, _ = K.groupnorm_fwd(xh, None, None, c, act=_acts()[act], chan_stats=cs)
    close("y from chan_stats", _nchw(y2), ref.detach(), 1e-2)

    # the conv epilogue's sums of its own output, whose channel means the bias shifts by `offset` stds
    k = 3
    w = (torch.randn(c, c, k, k, generator=g, device=dev, dtype=torch.float64) / math.sqrt(c * k * k)).float()
    wf, _ = K.pack_conv_weight(w, want_dgrad=False)
    bias = (offset * torch.where(torch.rand(c, generator=g, device=dev) < 0.5, -1.0, 1.0)).float().contiguous()
    stats = torch.zeros(n, c, 2, device=dev)
    yc = K.conv2d_fwd(xh, wf, bias, c, k, k, pad=1, stats=stats)
    assert torch.equal(yc, K.conv2d_fwd(xh, wf, bias, c, k, k, pad=1))  # the fused sums leave the output alone
    yc64 = _nchw(yc)
    want = torch.stack([yc64.sum(dim=(2, 3)), (yc64 * yc64).sum(dim=(2, 3))], dim=-1)
    close("conv epilogue stats", stats, want, 1e-4)
    y3, _, _ = K.groupnorm_fwd(yc, None, None, c, act=_acts()[act], chan_stats=stats)
    close("y from epilogue stats", _nchw(y3), _act64(F.instance_norm(yc64, eps=1e-5), act), 1e-2)


@pytest.mark.gpu
@pytest.mark.parametrize("case", PAD_CASES, ids=lambda c: "c%d_%d_pad%d" % c)
def test_reflection_pad_cut_production_shape(K, case):
    """pad2d / pad2d_bwd bit-exact: the gradient holds small multiples of 1/8, so every sum of up to four reflected
    contributions is exact in any precision"""
    c, size, pad = case
    n, dev = BATCH, "cuda"
    g = torch.Generator(device=dev).manual_seed(c + size + pad)
    x = torch.randn(n, c, size, size, generator=g, device=dev, dtype=torch.float64).bfloat16()
    y = K.pad2d(_nhwc(x), pad, 0)
    assert torch.equal(y, _nhwc(F.pad(x.double(), (pad,) * 4, mode="reflect")))
    dpad = (torch.randint(-64, 64, (n, c, size + 2 * pad, size + 2 * pad), generator=g, device=dev) / 8.0).double()
    xr = torch.zeros(n, c, size, size, device=dev, dtype=torch.float64, requires_grad=True)
    F.pad(xr, (pad,) * 4, mode="reflect").backward(dpad)
    assert torch.equal(K.pad2d_bwd(_nhwc(dpad), pad, 0), _nhwc(xr.grad))


# (act, NHWC shape): the G output's tanh, D's first LeakyReLU, the ReLU between PatchSampleF's two Linears (its token
# grid of batch 4 x 256 patches)
ACT_CASES = [("tanh", (BATCH, SIZE, SIZE, 8)), ("lrelu", (BATCH, SIZE // 2, SIZE // 2, NDF)),
             ("relu", (1, BATCH * NUM_PATCHES // 16, 16, NC))]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ACT_CASES, ids=lambda c: c[0])
def test_act_bwd_cut_production_shape(K, case):
    act, shape = case
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(len(act) + shape[-1])
    u = 2.0 * torch.randn(shape, generator=g, device=dev, dtype=torch.float64)
    y = _act64(u, act).bfloat16()
    dy = torch.randn(shape, generator=g, device=dev, dtype=torch.float64).bfloat16()
    dx = K.act_bwd(y, dy, _acts()[act])
    close("dx", dx, dy.double() * _act_grad64(y.double(), act), 1e-2)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [BATCH, 2 * BATCH])
def test_resnet_block_add_cut_production_shape(K, n):
    """ops.add (x + conv_block(x)): copy_channels(accumulate=True) rounds the fp32 sum once, bit-exact"""
    from joligen_b200 import ops
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(n)
    a = torch.randn(n, SIZE // 4, SIZE // 4, 4 * NGF, generator=g, device=dev).bfloat16()
    b = torch.randn(n, SIZE // 4, SIZE // 4, 4 * NGF, generator=g, device=dev).bfloat16()
    out = ops.add(a, b)
    assert torch.equal(out, (a.float() + b.float()).bfloat16())
    assert torch.equal(a, a.clone())  # (the operands stay as they were)


# (kernel mode, target, sign, gan_oracle.gan_loss arguments): lsgan real / fake (config 3), the projected-D hinge real /
# fake, the generator's linear loss and wgangp's fake term
GAN_CASES = [("lsgan_real", 0, 1.0, 1.0, (True, "lsgan", True)), ("lsgan_fake", 0, 0.0, 1.0, (False, "lsgan", True)),
             ("hinge_real", 1, 0.0, 1.0, (True, "projected", True)),
             ("hinge_fake", 1, 0.0, -1.0, (False, "projected", True)),
             ("linear_G", 2, 0.0, 1.0, (True, "projected", False)), ("linear_fake", 2, 0.0, -1.0, (False, "wgangp", True))]


@pytest.mark.gpu
@pytest.mark.parametrize("case", GAN_CASES, ids=lambda c: c[0])
def test_gan_loss_cut_production_shape(K, case):
    """gan_loss_fwd / _bwd on D's logit map [4, 30, 30, 1] stored with ld 8"""
    from oracle import gan_oracle as G
    _, mode, target, sign, (is_real, gan_mode, relu) = case
    dev = "cuda"
    hw = SIZE // 8 - 2
    g = torch.Generator(device=dev).manual_seed(mode * 10 + int(sign))
    pred = (0.5 + torch.randn(BATCH, 1, hw, hw, generator=g, device=dev, dtype=torch.float64)).bfloat16().double()
    pr = pred.clone().requires_grad_(True)
    ref = G.gan_loss(pr, is_real, gan_mode, relu)
    grad_out = torch.tensor(0.75, device=dev)
    ref.backward(grad_out.double())
    pred_d = _nhwc(pred, 8)
    loss = K.gan_loss_fwd(pred_d, 1, mode, target, sign)
    close("loss", loss, ref.detach(), 1e-5)
    d = K.gan_loss_bwd(pred_d, 1, mode, target, sign, grad_out)
    close("dpred", _nchw(d, 1), pr.grad, 1e-2)
    assert float(d[..., 1:].float().abs().max()) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("layer", range(len(NCE_LAYERS)), ids=lambda i: "layer%d" % NCE_LAYERS[i])
def test_cut_sampling_cut_production_shape(K, layer):
    """PatchSampleF + MoNCE on one NCE layer's feature maps (keys from the source image, queries from the generated
    one, the same 256 positions): gather_rows (bit-exact), the MLP's two 1x1 convolutions, l2norm, monce_fwd / _bwd
    against cut_oracle in float64 — each stage on the stored output of the one before"""
    from oracle import cut_oracle as C
    from joligen_b200.nets_cut import PatchSampleF
    c, c8, size = NCE_FEATS[layer]
    n, dev, T = BATCH, "cuda", 0.07
    g = torch.Generator(device=dev).manual_seed(layer)
    feats = [_nhwc(torch.randn(n, c, size, size, generator=g, device=dev), c8) for _ in range(2)]  # (k, q)
    ids = torch.randperm(size * size, generator=g, device=dev)[:NUM_PATCHES]
    netF = PatchSampleF(use_mlp=True, nc=NC, init_gain=0.2)
    netF.set_device(torch.device(dev))
    netF.data_dependent_initialize([torch.empty(1, c, 1, 1)])
    mlp = netF.mlp_0
    with torch.no_grad():  # (the kernels read bf16 copies of the weights)
        for lin in (mlp[0], mlp[2]):
            lin.weight.copy_(lin.weight.bfloat16())
    rows = []
    w1, b1, w2, b2 = (t.detach().double() for t in (mlp[0].weight, mlp[0].bias, mlp[2].weight, mlp[2].bias))
    for f in feats:
        x = K.gather_rows(f, ids)
        assert torch.equal(x, f.reshape(n, size * size, c8)[:, ids].reshape(n * NUM_PATCHES, c8))
        x.requires_grad_(True)
        h = netF._mlp(mlp, x)
        ref = F.linear(F.relu(F.linear(x[:, :c].double(), w1, b1)), w2, b2)
        close("mlp", h, ref.detach(), 1e-2)
        y, norms = K.l2norm_fwd(h.detach(), 1e-7)
        close("l2norm", y, F.normalize(h.detach().double(), eps=1e-7), 1e-5)
        rows.append((h, y, norms, x))
    (hk, k, nk, _), (hq, q, nq, _) = rows
    qr, kr = q.double().cpu().requires_grad_(True), k.double().cpu().requires_grad_(True)
    ref = C.patch_nce_loss(qr, kr, n, T=T, kind="monce", num_patches_opt=NUM_PATCHES)
    gout = torch.full((n * NUM_PATCHES,), 1.0 / (n * NUM_PATCHES), dtype=torch.float64)
    ref.backward(gout)
    loss, lse, ws = K.monce_fwd(q, k, n, T, NUM_PATCHES)
    close("monce loss per patch", loss, ref.detach(), 1e-4)
    close("monce loss", loss.double().mean(), ref.detach().mean(), 1e-5)
    dq, dk = K.monce_bwd(q, k, lse, gout.float().to(dev), ws, n, T, NUM_PATCHES)
    close("monce dq", dq, qr.grad, 2e-3)
    close("monce dk", dk, kr.grad, 2e-3)
    # l2norm backward of the queries' gradient, back onto the MLP output
    dh = K.l2norm_bwd(q, dq, nq, 1e-7)
    hr = hq.detach().double().requires_grad_(True)
    F.normalize(hr, eps=1e-7).backward(dq.double())
    close("l2norm dx", dh, hr.grad, 1e-2)
    # the MLP's backward (two 1x1 convolutions on the token grid) from that gradient; the weight-gradient reference reads
    # the bf16 tensors the kernels store: the hidden activation and its gradient
    xq = rows[1][3]
    hq.backward(dh)
    x64, dh64 = xq.detach()[:, :c].double(), dh.double()
    t1 = F.relu(F.linear(x64, w1, b1)).bfloat16().double()
    dt1 = ((dh64 @ w2).bfloat16().double() * (t1 > 0)).bfloat16().double()
    close("mlp dx", xq.grad[:, :c], dt1 @ w1, 1e-2)
    close("mlp dW2", mlp[2].weight.grad, dh64.t() @ t1, 1e-3)
    close("mlp db2", mlp[2].bias.grad, dh64.sum(0), 1e-3)
    close("mlp dW1", mlp[0].weight.grad, dt1.t() @ x64, 1e-3)
    close("mlp db1", mlp[0].bias.grad, dt1.sum(0), 1e-3)
    # the gather's adjoint: the rows land on their positions, everything else is zero
    d_rows = torch.randn(n * NUM_PATCHES, c8, generator=g, device=dev).bfloat16()
    d_feat = K.gather_rows_bwd(d_rows, ids, (n, size, size, c8))
    want = torch.zeros(n, size * size, c8, dtype=torch.bfloat16, device=dev)
    want[:, ids] = d_rows.reshape(n, NUM_PATCHES, c8)
    assert torch.equal(d_feat.reshape(n, size * size, c8), want)


# ---------------------------------------------------------------------------------------------------------------------
# the case lists against the benchmark step, on the kernel double (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _conv_key(x_shape, cout, r, s, stride, pad, out_hw):
    _, h, w, cin = x_shape
    return ("conv", h, w, cin, cout, r, s, stride, pad) + tuple(out_hw)


class _Recorder:
    """Wraps kernels.conv2d_fwd / conv2d_cropped / conv2d_wgrad / groupnorm_fwd / pad2d of the installed kernel double:
    records the geometry of each call; the convolutions return zeros of the right shape instead of computing."""

    def __init__(self, K):
        self.K, self.keys = K, set()
        self.saved = {}

    def __enter__(self):
        K = self.K
        for name in ("conv2d_fwd", "conv2d_cropped", "conv2d_wgrad", "groupnorm_fwd", "pad2d"):
            self.saved[name] = getattr(K, name)
        keys = self.keys

        def conv2d_fwd(x, w_packed, bias, cout, r, s, stride=1, pad=None, act=0, residual=None, res_scale=1.0,
                       out=None, stats=None, gn=None):
            pad = (r - 1) // 2 if pad is None else pad
            n, h, w, _ = x.shape
            ho, wo = K.conv_out_size(h, w, r, s, stride, pad)
            # PatchSampleF's 1x1 "convolutions" run on a token grid whose height is the number of patch rows
            keys.add(("fwd",) + (_conv_key(x.shape, cout, r, s, stride, pad, (ho, wo)) if r * s > 1 else
                                 ("linear", x.shape[-1], cout)) + (act,))
            y = torch.zeros((n, ho, wo, cout), dtype=torch.bfloat16)
            if out is None:
                return y
            with torch.autograd._unsafe_preserve_version_counter(out):
                out.copy_(y)
            return out

        def conv2d_cropped(x, w_packed, bias, cout, r, s, pad, out_hw, act=0):
            keys.add(("cropped",) + _conv_key(x.shape, cout, r, s, 1, pad, out_hw) + (act,))
            return torch.zeros((x.shape[0],) + tuple(out_hw) + (cout,), dtype=torch.bfloat16)

        def conv2d_wgrad(x, dy, cout, r, s, stride=1, pad=None, out=None, beta=0.0):
            pad = (r - 1) // 2 if pad is None else pad
            if r * s > 1:
                keys.add(("wgrad",) + _conv_key(x.shape, cout, r, s, stride, pad, dy.shape[1:3]))
            return torch.zeros((cout, x.shape[-1], r, s))

        def groupnorm_fwd(x, gamma, beta, groups, film=None, act=0, eps=1e-5, out=None, chan_stats=None):
            keys.add(("norm", x.shape[-1], x.shape[1], groups, gamma is None, act))
            return self.saved["groupnorm_fwd"](x, gamma, beta, groups, film, act, eps, out, chan_stats)

        def pad2d(x, pad, mode=0):
            keys.add(("pad", x.shape[-1], x.shape[1], pad, mode))
            return self.saved["pad2d"](x, pad, mode)

        for name, fn in (("conv2d_fwd", conv2d_fwd), ("conv2d_cropped", conv2d_cropped),
                         ("conv2d_wgrad", conv2d_wgrad), ("groupnorm_fwd", groupnorm_fwd), ("pad2d", pad2d)):
            setattr(K, name, fn)
        return self

    def __exit__(self, *exc):
        for name, fn in self.saved.items():
            setattr(self.K, name, fn)


def _expected_keys():
    """the kernel calls the GPU cases above make, derived from ConvActFn / ConvTranspose2dFn"""
    A = _acts()
    keys = set()
    for _, kind, cin, cout, k, stride, pad, reflect, act, size in CONV_LAYERS:
        cin8, cout8 = _c8(cin), _c8(cout)
        if reflect:
            keys.add(("pad", cin8, size, reflect, 0))
        hin = size + 2 * reflect
        if kind == "convT":
            ho = 2 * size
            keys.add(("cropped", "conv", 2 * size, 2 * size, cin8, cout8, k, k, 1, k - 1 - pad, ho, ho, A["none"]))
            keys.add(("fwd", "conv", ho, ho, cout8, cin8, k, k, 2, pad, size, size, A["none"]))
            keys.add(("wgrad", "conv", ho, ho, cout8, cin8, k, k, 2, pad, size, size))
            continue
        ho = (hin + 2 * pad - k) // stride + 1
        keys.add(("fwd", "conv", hin, hin, cin8, cout8, k, k, stride, pad, ho, ho, A[act]))
        keys.add(("wgrad", "conv", hin, hin, cin8, cout8, k, k, stride, pad, ho, ho))
        if stride == 1:
            keys.add(("fwd", "conv", ho, ho, cout8, cin8, k, k, 1, k - 1 - pad, hin, hin, A["none"]))
        else:
            keys.add(("cropped", "conv", 2 * ho, 2 * ho, cout8, cin8, k, k, 1, k - 1 - pad, hin, hin, A["none"]))
    for c, size, act in NORM_SHAPES:
        keys.add(("norm", c, size, c, True, A[act]))
    for c, c8, _ in NCE_FEATS:
        keys.add(("fwd", "linear", c8, NC, A["relu"]))
        keys.add(("fwd", "linear", NC, NC, A["none"]))
        keys.add(("fwd", "linear", NC, c8, A["none"]))  # the first Linear's dgrad
    return keys


def test_cases_match_the_benchmark_step(monkeypatch):
    """One CutTrainer step of bench.py --config 3 (batch 1, 256x256) on the kernel double: the set of convolution,
    InstanceNorm and padding geometries it launches is exactly the set the GPU cases of this file exercise."""
    from unittest import mock
    sys.path.insert(0, os.path.dirname(__file__))
    import kernel_double as KD
    from joligen_b200 import kernels as K
    from joligen_b200 import nets_cut, nets_gan
    from joligen_b200 import synthetic
    from joligen_b200.trainer_cut import CutTrainer
    torch.manual_seed(0)
    with KD.installed(), _Recorder(K) as rec:
        netG = nets_gan.ResnetGenerator(3, 3, NGF, n_blocks=9)
        netD = nets_gan.NLayerDiscriminator(3, NDF, n_layers=3)
        synthetic.dezero_init_(netG, 11)
        synthetic.dezero_init_(netD, 12)
        netF = nets_cut.PatchSampleF(use_mlp=True, nc=NC)
        g = torch.Generator().manual_seed(1234)
        host = {"A": torch.rand(1, 3, SIZE, SIZE, generator=g) * 2 - 1,
                "B": torch.rand(1, 3, SIZE, SIZE, generator=g) * 2 - 1}
        netF.data_dependent_initialize(netG.get_feats(host["A"], NCE_LAYERS))
        synthetic.dezero_init_(netF, 13)
        with mock.patch("torch.cuda.is_available", return_value=True):
            tr = CutTrainer(netG, netF, netD, nce_layers=NCE_LAYERS, num_patches=NUM_PATCHES, nce_loss="monce",
                            gan_mode="lsgan", G_lr=2e-4, D_lr=1e-4, optim="adam", cuda_graph=False, device="cpu")
        tr.set_input(host)
        monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: False)
        tr.optimize_parameters()
    expected = _expected_keys()
    assert rec.keys == expected, sorted(map(str, rec.keys ^ expected))
    assert {k for k in expected if k[0] == "pad"} == {("pad", c, size, pad, 0) for c, size, pad in PAD_CASES}
