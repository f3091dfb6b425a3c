"""Drives the UNMODIFIED reference (oracle/_ref, staged by oracle/install_ref.py) through its own public control
path — options -> models.create_model -> model.setup -> model.set_input -> model.optimize_parameters()
(train.py:183-199, 268-282; models/base_model.py:1302-1377) — for bench.py's reference arm (CPU, all host threads) and
for the GPU incumbent (the same stock code on cuda:0: fp32, and TF32 as train.py --with_tf32 sets it, :536-538).

Nothing of joligen_b200 is imported here.  Optional third-party packages that the reference imports at module level
but never touches on this path (visdom, lpips, clip, timm, ...) are replaced by MagicMock modules when they are not
installed; torch / numpy are the real ones.
"""
import importlib.abc
import importlib.machinery
import json
import os
import sys
import tempfile
import time
from unittest import mock

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = os.path.join(os.path.dirname(HERE), "oracle", "_ref")

OPTIONAL = [
    "thop", "torchviz", "piq", "lpips", "positional_encodings", "clip", "timm", "bitsandbytes", "imgaug",
    "dominate", "visdom", "aim", "diffusers", "peft", "segment_anything", "mobile_sam", "torchinfo", "addict",
    "onnx", "DISTS_pytorch", "vision_aided_loss", "ouisdom", "tifffile", "wget", "xformers", "ftfy", "iopath",
    "pytorchvideo", "open_clip", "kornia", "onnxruntime", "cv2", "torchvision",
]


class _MockLoader(importlib.abc.Loader):
    def create_module(self, spec):
        m = mock.MagicMock(name=spec.name)
        m.__name__, m.__path__, m.__spec__, m.__loader__ = spec.name, [], spec, self
        return m

    def exec_module(self, module):
        pass


class _StubFinder(importlib.abc.MetaPathFinder):
    def __init__(self, names):
        self.names = set(names)

    def find_spec(self, fullname, path, target=None):
        if fullname.split(".")[0] in self.names:
            return importlib.machinery.ModuleSpec(fullname, _MockLoader(), is_package=True)
        return None


def available():
    return os.path.exists(os.path.join(REF_ROOT, "models", "base_model.py"))


def _install_import_path():
    sys.dont_write_bytecode = True
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)

    def importable(name):
        try:
            __import__(name)
            return True
        except Exception:
            return False

    sys.meta_path.insert(0, _StubFinder([m for m in OPTIONAL if not importable(m)]))


def _flatten(d, prefix=""):
    flat = {}
    for k, v in d.items():
        if isinstance(v, dict):
            flat.update(_flatten(v, prefix + k + "_"))
        else:
            flat[prefix + k] = v
    return flat


def build_palette_model(size=256, batch=32, device="cpu", with_tf32=False):
    """BASELINE.json config 2 (SURVEY.md section 8d) through the reference's option parser and model factory."""
    import torch
    _install_import_path()
    import train as ref_train
    from models import create_model
    from options.train_options import TrainOptions

    with open(os.path.join(REF_ROOT, "examples", "example_ddpm_mario.json")) as f:
        flat = _flatten(json.load(f))
    tmp = tempfile.mkdtemp(prefix="jg_ref_")
    use_cuda = device != "cpu"
    flat.update({
        "gpu_ids": "0" if use_cuda else "-1", "data_crop_size": size, "data_load_size": size,
        "train_batch_size": batch, "dataroot": tmp, "checkpoints_dir": tmp, "name": "bench",
        "model_type": "palette", "G_netG": "unet_mha", "G_ngf": 64, "G_unet_mha_channel_mults": [1, 2, 4, 8],
        "G_unet_mha_res_blocks": [2, 2, 2, 2], "G_unet_mha_attn_res": [16], "G_unet_mha_num_head_channels": 32,
        "G_unet_mha_group_norm_size": 32, "alg_diffusion_cond_embed": "", "alg_diffusion_cond_embed_dim": 32,
        "alg_diffusion_task": "inpainting", "alg_diffusion_cond_image_creation": "y_t", "alg_palette_loss": "MSE",
        "train_optim": "adamw", "train_G_lr": 1e-4, "train_G_ema": True, "train_G_ema_beta": 0.999,
        "train_iter_size": 1, "G_diff_n_timestep_train": 2000, "output_no_html": True, "with_tf32": bool(with_tf32),
    })
    opt = TrainOptions().parse_json(flat, save_config=False)
    opt.use_cuda = use_cuda
    opt.optim = ref_train.optim
    opt.jg_dir = REF_ROOT
    opt.total_iters = 0
    opt.num_test_images = 0
    if use_cuda:
        # what launch_training does for --with_tf32 (train.py:536-538); the default is strict fp32
        torch.backends.cuda.matmul.allow_tf32 = bool(with_tf32)
        torch.backends.cudnn.allow_tf32 = bool(with_tf32)
    torch.manual_seed(1234)
    model = create_model(opt, 0)
    model.setup(opt)
    model.use_temporal = False
    if use_cuda:
        model.single_gpu()
    return model, opt


def synthetic_batch(batch, size, seed):
    """The bench's config-2 inputs (SURVEY.md section 8d), generated with torch only."""
    import math
    import torch
    g = torch.Generator().manual_seed(seed)
    gt = (0.5 * torch.randn(batch, 3, size, size, generator=g)).clamp(-1, 1)
    mask = torch.zeros(batch, 1, size, size, dtype=torch.int64)
    for i in range(batch):
        frac = 0.1 + 0.3 * float(torch.rand((), generator=g))
        side = max(1, int(round(size * math.sqrt(frac))))
        y0 = int(torch.randint(0, size - side + 1, (), generator=g))
        x0 = int(torch.randint(0, size - side + 1, (), generator=g))
        mask[i, 0, y0:y0 + side, x0:x0 + side] = 1
    cond = gt * (1 - mask) + torch.randn(batch, 3, size, size, generator=g) * mask
    return {"A": cond, "B": gt, "B_label_mask": mask, "B_label_cls": torch.zeros(batch, dtype=torch.long),
            "A_img_paths": ["synthetic"] * batch}


def time_steps(model, batch, size, steps, warmup, device="cpu", budget_s=None):
    """-> (seconds per step, steps timed, last loss).  CPU: perf_counter; GPU: CUDA events + synchronize."""
    import torch
    data = synthetic_batch(batch, size, 1234)
    for _ in range(warmup):
        model.set_input(data)
        model.optimize_parameters()
    times = []
    if device == "cpu":
        for _ in range(steps):
            t0 = time.perf_counter()
            model.set_input(data)
            model.optimize_parameters()
            times.append(time.perf_counter() - t0)
            if budget_s is not None and sum(times) > budget_s:
                break
        sec = sum(times) / len(times)
        n = len(times)
    else:
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            model.set_input(data)
            model.optimize_parameters()
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) / 1000.0 / steps
        n = steps
    return sec, n, float(model.loss_G_tot)


def main():
    """python baseline/ref_runner.py --device cuda --batch 8 --steps 3 --warmup 2 [--tf32]  -> one JSON line."""
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--device", default="cpu")
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--tf32", action="store_true")
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--budget", type=float, default=0.0)
    a = ap.parse_args()
    import torch
    if a.threads:
        torch.set_num_threads(a.threads)
    model, _ = build_palette_model(a.size, a.batch, a.device, a.tf32)
    sec, n, loss = time_steps(model, a.batch, a.size, a.steps, a.warmup, a.device, a.budget or None)
    out = {"images_per_s": a.batch / sec, "s_per_step": sec, "steps_timed": n, "warmup": a.warmup, "batch": a.batch,
           "size": a.size, "device": a.device, "tf32": bool(a.tf32), "loss_last": loss,
           "threads": torch.get_num_threads(), "torch": str(torch.__version__)}
    if a.device != "cpu":
        out["max_mem_gb"] = torch.cuda.max_memory_allocated() / 2 ** 30
        out["gpu"] = torch.cuda.get_device_name(0)
    print("REF_RESULT " + json.dumps(out))


if __name__ == "__main__":
    main()
