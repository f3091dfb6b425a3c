"""bench.py — training-step throughput of the B200 path on BASELINE.json's configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5]
                    [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL); rank 0 prints ONE JSON line.

--config 2 (default, the headline): Palette UNet ngf 64, mults 1-2-4-8, 2 ResBlocks / level, attention at 32x32,
256x256, per-GPU batch 32, bf16 activations / fp32 accumulate, synthetic self-supervised box masks, random-init
de-zeroed weights.  A "step" = set_input + optimize_parameters() = noising prologue + UNet forward + eps-loss +
backward (dgrad + wgrad) + gradient all-reduce + fused AdamW + EMA.
--config 3 / 4 / 5: cut_model resnet_9blocks + NLayerD (b=4/GPU), palette UNet-ref (128^2 b=16 or --size 512x384 b=2),
UNetVid 8 x 128^2 (1 clip/GPU): same step definition through their trainers.

  value   : images/s with the batch already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e     : images/s through the public API with HOST (pinned) batches: H2D copy of the inputs and a D2H read of the
            loss inside every timed step
  roofline: bound "tensor".  `frac` is STEP-LEVEL (BASELINE.md section 2): algorithmic FLOPs of the whole step / step
            time / measured sustained cuBLAS bf16 peak.  `conv` carries the implicit-GEMM family alone: FLOPs actually
            issued by the conv launches (de-padded) / their summed CUDA-event duration in an instrumented eager pass.
            `traffic` = DRAM read + write bytes of the implicit-GEMM launches of ONE step from the committed ncu launch
            list of the same step (profiles/r02_conv_traffic.json, config 2 only; null otherwise): DRAM bytes cannot be
            measured inside a timed run.
  cpu_baseline / --impl reference: the UNMODIFIED reference (oracle/_ref, staged by oracle/install_ref.py) driven
            through options -> create_model -> optimize_parameters() on the host cores (kind "reference"); the oracle
            port only if the staged reference is missing (kind "port").
  incumbent_gpu: the same unmodified reference on cuda:0 (cuDNN, fp32 and TF32), CUDA-event timed, reduced batch.

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step handed its caller — DIR/loss.npy (the
step's loss value(s), float64), DIR/params_<net>.npy (every trained network's updated weights, flattened in parameter
order, float32) and DIR/ema.npy (the EMA copy, when the trainer keeps one) — 64 MB at most in all: an array over its
share holds a fixed, seeded sample of its elements.  Weights and inputs are seeded, so two builds of the project can be
compared output for output on the same arguments.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FWD_GMAC_PER_IMG_256 = 206.63  # SURVEY.md §8(d): Palette UNet 256^2 forward; train step = 3x
METRIC = "train-step images/sec Palette UNet 256^2 bf16"
# SURVEY.md §8(d) forward GMAC per image (per clip for cfg 5); the train step is 3x (fwd + dgrad + wgrad)
CONFIG_INFO = {
    2: dict(metric=METRIC, batch=32, size=(256, 256)),
    3: dict(metric="train-step images/sec CUT resnet_9blocks G + NLayerD 256^2 bf16", batch=4, size=(256, 256)),
    4: dict(metric="train-step images/sec Palette UNet-ref (ref attention) bf16", batch=16, size=(128, 128)),
    5: dict(metric="train-step frames/sec UNetVid 8-frame 128^2 bf16", batch=1, size=(128, 128)),
    6: dict(metric="train-step frames/sec b2b JiTVid-B/16 8-frame 128^2 bf16", batch=1, size=(128, 128)),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5, 6])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the configuration's)")
    ap.add_argument("--size", default="", help="H or HxW (default: the configuration's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-incumbent", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of CUDA-graph replay")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the last timed step's outputs to DIR/<name>.npy (64 MB at most)")
    a = ap.parse_args()
    info = CONFIG_INFO[a.config]
    a.batch = a.batch or info["batch"]
    if a.size:
        parts = [int(v) for v in a.size.lower().split("x")]
        a.size = (parts[0], parts[-1])
    else:
        a.size = info["size"]
    return a


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "hbm_gbs": d.get("hbm_gbs"),
                "source": "MEASURED_PEAKS.json (sustained cuBLAS bf16; the step is seconds long)"}
    return {"bf16_tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower() == "active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def usable_cpu_threads():
    """Host threads this process can really run on: scheduler affinity capped by the cgroup CPU quota (a container
    that sees 128 logical CPUs but is throttled to a few cores makes a 128-thread torch run pathologically slow).
    torchrun exports OMP_NUM_THREADS=1 to its workers: the reference arm sets its thread count explicitly from here."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // period))
            break
        except Exception:
            continue
    return n


def cpu_threads():
    return int(os.environ.get("JG_CPU_THREADS", "0")) or usable_cpu_threads()


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline / GPU incumbent: the unmodified reference from oracle/_ref, in a child process
# ---------------------------------------------------------------------------------------------------------------------
def _run_ref_runner(extra, timeout):
    env = dict(os.environ)
    env.pop("OMP_NUM_THREADS", None)  # torchrun's OMP_NUM_THREADS=1 must not throttle the CPU arm
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "GROUP_RANK", "LOCAL_WORLD_SIZE"):
        env.pop(k, None)
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "ref_runner.py")] + [str(x) for x in extra]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    except subprocess.TimeoutExpired:
        return None, "timeout after %d s" % timeout
    for line in r.stdout.splitlines():
        if line.startswith("REF_RESULT "):
            return json.loads(line[len("REF_RESULT "):]), None
    return None, (r.stderr.strip().splitlines() or ["no output"])[-1][:300]


def reference_available():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "models", "base_model.py"))


def cpu_reference_throughput(size, steps, warmup=1, threads=None, budget_s=120.0):
    """The reference's CPU training step on the host cores, bounded sample: batch 1 at the full resolution."""
    threads = threads or cpu_threads()
    b = 1
    if reference_available():
        res, err = _run_ref_runner(["--device", "cpu", "--batch", b, "--size", size, "--steps", steps, "--warmup",
                                    warmup, "--threads", threads, "--budget", budget_s], timeout=int(budget_s * 3 + 180))
        if res is not None:
            return {"value": res["images_per_s"], "unit": "images/s", "cores": res["threads"], "kind": "reference",
                    "steps_timed": res["steps_timed"], "batch": b,
                    "sample": "%d optimize_parameters() of batch %d at %dx%d by the unmodified reference (fp32 torch-CPU, "
                              "create_model -> PaletteModel, AdamW + EMA), %d threads of %d logical CPUs, %.2f s/step"
                              % (res["steps_timed"], b, size, size, res["threads"], os.cpu_count() or 0,
                                 res["s_per_step"])}
        note = "reference run failed (%s); oracle port instead" % err
    else:
        note = "oracle/_ref missing; oracle port instead"
    out = cpu_port_throughput(size, steps, threads, budget_s)
    out["note"] = note
    return out


def cpu_port_throughput(size, steps, threads, budget_s):
    """Fallback: the oracle's restatement of the same step (used only when oracle/_ref did not travel)."""
    from oracle import palette_oracle as O
    torch.set_num_threads(threads)
    oc = O.OptimCfg(lr=1e-4)
    b = 1

    def one_step(state, cfg, sz, seed):
        data = O.synthetic_batch(b, sz, 77 + seed)
        torch.manual_seed(seed)
        t, u = O.sample_t_gamma(cfg, b)
        noise = torch.randn_like(data["gt"])
        t0 = time.perf_counter()
        O.train_step(state, cfg, oc, data["gt"], data["cond"], data["mask"], noise, t, u)
        return time.perf_counter() - t0

    cfg = O.UNetCfg(image_size=size)
    state = O.TrainState(params=O.init_params(cfg, 1234))
    one_step(state, O.UNetCfg(image_size=64), 64, 0)
    times = []
    for s in range(steps):
        times.append(one_step(state, cfg, size, 1 + s))
        if sum(times) > budget_s:
            break
    sec = sum(times) / len(times)
    return {"value": b / sec, "unit": "images/s", "cores": threads, "kind": "port", "steps_timed": len(times),
            "batch": b,
            "sample": "%d step(s) of batch %d at %dx%d (fwd+loss+bwd+AdamW+EMA), fp32 torch-CPU oracle port, "
                      "%d threads of %d logical CPUs, %.1f s/step" % (len(times), b, size, size, threads,
                                                                      os.cpu_count() or 0, sec)}


def gpu_incumbent(size, batch=8, steps=3, warmup=3):
    """The unmodified reference on cuda:0 (its stock cuDNN path): strict fp32 and --with_tf32."""
    if not reference_available():
        return {"unavailable": "oracle/_ref missing"}
    out = {"batch": batch, "steps": steps, "warmup": warmup,
           "what": "unmodified reference (create_model -> optimize_parameters), cuDNN NCHW, cudnn.benchmark, "
                   "CUDA-event timed; batch %d (fp32 activations of batch 32 do not leave room beside this process)"
                   % batch}
    for key, flag in (("fp32", []), ("tf32", ["--tf32"])):
        res, err = _run_ref_runner(["--device", "cuda", "--batch", batch, "--size", size, "--steps", steps,
                                    "--warmup", warmup] + flag, timeout=240)
        out[key] = ({"images_per_s": res["images_per_s"], "ms_per_step": 1000.0 * res["s_per_step"],
                     "max_mem_gb": res.get("max_mem_gb")} if res is not None else {"unavailable": err})
    return out


def run_reference(args):
    """--impl reference: rank 0 times the reference's CPU path; every step is a bounded sample (one image at the full
    resolution) of the GPU arm's workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.config != 2:
        print(json.dumps({"impl": "reference", "unavailable": "the CPU reference arm is wired for --config 2 only"}))
        return
    size = args.size[0]
    cb = cpu_reference_throughput(size, max(1, args.steps), warmup=max(1, min(args.warmup, 2)), budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "images/s", "n_gpus": args.gpus,
        "steps": cb["steps_timed"], "warmup": max(1, min(args.warmup, 2)), "ms_per_step": 1000.0 * cb["batch"] / cb["value"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "palette_model Palette UNet %dx%d bf16 batch=%d/GPU, synthetic self-supervised masks"
                               % (size, size, args.batch),
                   "sample": "each step = ONE image (batch %d, fp32) of that workload on the host CPU: %s"
                             % (cb["batch"], cb["sample"]),
                   "steps_requested": args.steps},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------------
def build_workload(args, rank, world):
    """-> (trainer, host batch dict, images per step per GPU, workload string, algorithmic step FLOPs or None)"""
    from joligen_b200 import nets, synthetic
    from joligen_b200.trainer import PaletteTrainer
    torch.manual_seed(1234)   # default initialisations and the in-step draws (noise, t): the same on every run
    h, w = args.size
    B = args.batch
    common = dict(in_channel=6, inner_channel=64, out_channel=3, tanh=False, n_timestep_train=2000,
                  n_timestep_test=1000, norm="groupnorm", group_norm_size=32, cond_embed_dim=32,
                  channel_mults=(1, 2, 4, 8), num_heads=1, num_head_channels=32)
    graph = not args.no_graph
    if args.config == 2:
        assert h == w
        net = nets.build_palette_generator(image_size=h)
        synthetic.dezero_init_(net, 1234)
        tr = PaletteTrainer(net, lr=1e-4, optim="adamw", ema=True, ema_beta=0.999, device="cuda", cuda_graph=graph,
                            graph_warmup=2)
        tr.broadcast_parameters()
        host = synthetic.synthetic_batch(B, h, 1234 + rank)
        alg = 3 * 2 * FWD_GMAC_PER_IMG_256 * 1e9 * B * (h / 256.0) ** 2
        name = "palette_model Palette UNet %dx%d bf16 batch=%d/GPU, synthetic self-supervised masks" % (h, w, B)
        return tr, host, B, name, alg
    if args.config == 4:
        from joligen_b200 import nets_ref
        unet = nets_ref.UNetGeneratorRefAttn(image_size=max(h, w), res_blocks=[2, 4, 4, 2], attn_res=[4, 8], **common)
        g = nets.DiffusionGenerator(nets.PaletteDenoiseFn(unet, 32), image_size=max(h, w), G_ngf=64)
        synthetic.dezero_init_(g, 3)
        tr = PaletteTrainer(g, lr=1e-4, optim="adamw", ema=True, device="cuda", cuda_graph=graph, graph_warmup=2)
        tr.broadcast_parameters()
        host = synthetic.synthetic_rect_batch(B, h, w, 1234 + rank)
        host["ref_A"] = 0.5 * torch.randn(B, 3, h, w, generator=torch.Generator().manual_seed(99 + rank))
        gmac = {(128, 128): 130.53, (512, 384): 3568.3}.get((h, w))
        name = "palette_model UNet-ref VITON (unet_mha_ref_attn, res_blocks 2-4-4-2, attention at ds 4, 8) %dx%d bf16 " \
               "batch=%d/GPU" % (h, w, B)
        return tr, host, B, name, (3 * 2 * gmac * 1e9 * B if gmac else None)
    if args.config == 5:
        from joligen_b200 import nets_vid
        frames = 8
        unet = nets_vid.UNetVid(image_size=h, res_blocks=[2, 2, 2, 2], attn_res=[16], **common)
        g = nets.DiffusionGenerator(nets.PaletteDenoiseFn(unet, 32), image_size=h, G_ngf=64)
        synthetic.dezero_init_(g, 3)
        tr = PaletteTrainer(g, lr=1e-4, optim="adamw", ema=True, device="cuda", cuda_graph=graph, graph_warmup=2)
        tr.broadcast_parameters()
        clips = [synthetic.synthetic_batch(frames, h, 1234 + rank * 64 + i) for i in range(B)]
        host = {k: torch.stack([c[k] for c in clips]) for k in clips[0]}
        gmac = 862.63 * (h / 128.0) ** 2
        name = "palette_model video UNet (unet_vid, MotionModule) %d-frame %dx%d bf16, %d clip(s)/GPU" % (frames, h, w, B)
        return tr, host, B * frames, name, 3 * 2 * gmac * 1e9 * B
    if args.config == 6:
        # BASELINE.json config 5 as written: b2b_model + vit_vid (example_b2b_vid_mario.json): JiTVid-B/16, 8 frames
        from joligen_b200 import nets_jit
        from joligen_b200.trainer_b2b import B2BTrainer
        frames = 8
        net = nets_jit.B2BGenerator(nets_jit.JiTViD(input_size=h, patch_size=16, in_channels=3, hidden_size=768, depth=12,
                                                    num_heads=12, in_context_len=32, in_context_start=4, max_frames=8,
                                                    motion_num_heads=8, motion_num_layers=2))
        synthetic.dezero_init_(net, 5)
        tr = B2BTrainer(net, lr=1e-4, beta1=0.9, beta2=0.95, ema=True, ema_beta=0.999, cuda_graph=graph, graph_warmup=2)
        tr.broadcast_parameters()
        g = torch.Generator().manual_seed(1234 + rank)
        gt = (0.5 * torch.randn(B, frames, 3, h, w, generator=g)).clamp(-1, 1)
        mask = (torch.rand(B, frames, 1, h, w, generator=g) > 0.6).float()
        host = {"A": gt * (1 - mask) + torch.randn(gt.shape, generator=g) * mask, "B": gt, "B_label_mask": mask}
        name = "b2b_model JiTVid-B/16 (vit_vid, 156 M parameters) %d-frame %dx%d bf16, %d clip(s)/GPU" % (
            frames, h, w, B)
        return tr, host, B * frames, name, None
    # config 3: CUT
    from joligen_b200 import nets_cut, nets_gan
    from joligen_b200.trainer_cut import CutTrainer
    netG = nets_gan.ResnetGenerator(3, 3, 64, n_blocks=9)
    netD = nets_gan.NLayerDiscriminator(3, 64, n_layers=3)
    synthetic.dezero_init_(netG, 11)
    synthetic.dezero_init_(netD, 12)
    netG, netD = netG.cuda(), netD.cuda()
    netF = nets_cut.PatchSampleF(use_mlp=True, nc=256)
    netF.set_device(torch.device("cuda"))
    g = torch.Generator().manual_seed(1234 + rank)
    host = {"A": torch.rand(B, 3, h, w, generator=g) * 2 - 1, "B": torch.rand(B, 3, h, w, generator=g) * 2 - 1}
    nce_layers = [0, 4, 8, 12, 16]
    netF.data_dependent_initialize(netG.get_feats(host["A"][:1].cuda(), nce_layers))
    synthetic.dezero_init_(netF, 13)
    tr = CutTrainer(netG, netF, netD, nce_layers=nce_layers, num_patches=256, nce_loss="monce", gan_mode="lsgan",
                    G_lr=2e-4, D_lr=1e-4, optim="adam", cuda_graph=False)
    name = "cut_model resnet_9blocks G + NLayerDiscriminator (basic) %dx%d bf16 batch=%d/GPU, MoNCE + identity NCE, " \
           "lsgan (projected-D backbone out of scope)" % (h, w, B)
    return tr, host, B, name, None


DUMP_BYTES = 64 << 20


def step_outputs(tr, out):
    """What one training step hands its caller, on the host: the loss value(s) optimize_parameters() returned, the
    updated weights of every network the trainer owns and its EMA copy.  An array over its share of DUMP_BYTES keeps a
    fixed, seeded sample of its elements (the same positions for the same shapes)."""
    losses = out if isinstance(out, (tuple, list)) else (out,)
    arrays = {"loss": torch.stack([l.detach().double().reshape(()) for l in losses]).cpu()}
    for name, m in sorted(vars(tr).items()):
        if isinstance(m, torch.nn.Module) and any(True for _ in m.parameters()):
            arrays["params_" + name] = torch.cat([p.detach().float().reshape(-1) for p in m.parameters()])
    if isinstance(getattr(tr, "ema", None), torch.Tensor):
        arrays["ema"] = tr.ema.detach().float().reshape(-1)
    share = (DUMP_BYTES - 4096) // 4 // max(1, len(arrays) - 1)
    for name, v in arrays.items():
        if name != "loss" and v.numel() > share:
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            v = v[idx.to(v.device)]
        arrays[name] = v.cpu()
    return arrays


def dump_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(path, name + ".npy"), v.numpy())


def ncu_conv_traffic(args):
    """DRAM bytes per step of the implicit-GEMM launches (ncu launch list committed under profiles/), config 2 at the
    default size only; None when there is no capture for the workload."""
    if args.config != 2 or tuple(args.size) != tuple(CONFIG_INFO[2]["size"]):
        return None
    path = os.path.join(ROOT, "profiles", "r02_conv_traffic.json")
    try:
        with open(path) as f:
            return float(json.load(f)["dram_bytes_total"])
    except (OSError, KeyError, ValueError):
        return None


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from joligen_b200 import lib as L

    L.load()
    assert L.load().jg_check_device() == 0, L.load().jg_last_error()
    tr, host, imgs_per_gpu, workload, alg_flops_step = build_workload(args, rank, world)
    host = {k: v.pin_memory() for k, v in host.items()}
    dev = {k: v.cuda() for k, v in host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_loss(out):
        return out[0] if isinstance(out, tuple) else out

    def run(steps, from_host):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        last = out = None
        for _ in range(steps):
            tr.set_input(host if from_host else dev)
            out = tr.optimize_parameters()
            if from_host:
                last = float(step_loss(out))  # D2H read of the step's loss
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms / steps, last, out

    run(max(args.warmup, 3), False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    L.launch_count[0] = 0
    ms, _, out = run(args.steps, False)
    launches = L.launch_count[0]
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        outputs = step_outputs(tr, out)   # before the passes below train on
    run(1, True)
    ms_e2e, last_loss, _ = run(args.steps, True)

    # instrumented pass: CUDA events around every C-ABI call; conv launches carry the FLOPs they issue
    recs = []
    allrecs = []

    @contextlib.contextmanager
    def hook(name, cargs):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        yield
        e1.record()
        if name in ("jg_conv2d_fwd", "jg_conv2d_fwd_ex", "jg_conv2d_wgrad", "jg_conv2d_wgrad_acc"):
            d = cargs[0]._obj
            flops = 2.0 * d.N * d.Ho * d.Wo * d.Cout * d.Cin * d.R * d.S
            recs.append((name, flops, e0, e1))
            tag = name
            if name == "jg_conv2d_fwd_ex":  # which GroupNorm reduction rides in the epilogue
                e = cargs[1]._obj
                tag = "jg_conv2d_fwd+" + ("stats" if e.stats else "") + ("gnsums" if e.gn_sums else "")
            allrecs.append((tag, (d.N, d.H, d.W, d.Cin, d.Cout, d.R, d.stride), flops, e0, e1))
        elif name == "jg_groupnorm_fwd":
            allrecs.append((name, tuple(int(v) for v in cargs[4:8]), 0.0, e0, e1))
        elif name == "jg_groupnorm_bwd":
            allrecs.append((name, tuple(int(v) for v in cargs[7:11]), 0.0, e0, e1))
        else:
            allrecs.append((name, None, 0.0, e0, e1))

    L.call_hook[0] = hook
    tr.set_input(dev)
    ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev_a.record()
    if hasattr(tr, "eager_step"):
        tr.eager_step()  # eager launches (the timed region above replays the same kernels from CUDA graphs)
    else:
        tr.optimize_parameters()
    ev_b.record()
    torch.cuda.synchronize()
    L.call_hook[0] = None
    if rank == 0 and os.environ.get("JG_BREAKDOWN"):
        agg = {}
        for name, shape, flops, e0, e1 in allrecs:
            key = name if shape is None else "%s %s" % (name, list(shape))
            a = agg.setdefault(key, {"calls": 0, "ms": 0.0, "flops": 0.0})
            a["calls"] += 1
            a["ms"] += e0.elapsed_time(e1)
            a["flops"] += flops
        rows = sorted(agg.items(), key=lambda kv: -kv[1]["ms"])
        with open(os.environ["JG_BREAKDOWN"], "w") as f:
            json.dump({"instrumented_step_ms": ev_a.elapsed_time(ev_b),
                       "sum_call_ms": sum(v["ms"] for _, v in rows),
                       "rows": [dict(key=k, tflops=(v["flops"] / v["ms"] / 1e9 if v["ms"] > 0 else 0), **v)
                                for k, v in rows]}, f, indent=1)
    conv_ms = sum(e0.elapsed_time(e1) for _, _, e0, e1 in recs)
    conv_flops_issued = sum(f for _, f, _, _ in recs)
    peaks = measured_peaks()

    if rank == 0:
        imgs = imgs_per_gpu * world
        value = imgs / (ms / 1000.0)
        step_flops = alg_flops_step if alg_flops_step is not None else conv_flops_issued
        achieved = step_flops / (ms / 1000.0) / 1e12
        conv_tf = conv_flops_issued / (conv_ms / 1000.0) / 1e12 if conv_ms > 0 else 0.0
        info = CONFIG_INFO[args.config]
        unit = "frames/s" if args.config in (5, 6) else "images/s"   # (video configurations count frames)
        line = {
            "metric": info["metric"], "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload, "baseline_config": args.config,
                       "global_batch": args.batch * world, "parallelism": "dp%d" % world,
                       "l2": "per-step activations (GBs) exceed the 126 MB L2; no explicit flush",
                       "optimizer": "fused Adam(W)+EMA", "loss_last": last_loss,
                       "launch": "CUDA graph replay (fwd+bwd graph incl. the bucketed gradient all-reduce, optimizer "
                                 "graph)" if getattr(tr, "_graph_fb", None) is not None else
                                 ("CUDA graph replay (one graph: forward, backward, optimizer)"
                                  if getattr(tr, "_graph", None) is not None else "eager")},
            "e2e": {"value": imgs / (ms_e2e / 1000.0), "unit": unit, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": achieved / peaks["bf16_tflops"], "traffic": ncu_conv_traffic(args),
                         "what": "STEP-LEVEL: %s FLOPs of one step (%.2f TFLOP) / device time of the whole step"
                                 % ("algorithmic (SURVEY.md 8d, 3 x forward)" if alg_flops_step is not None
                                    else "issued implicit-GEMM", step_flops / 1e12),
                         "kernel": "conv_halo(2) / conv_fwd / wgrad_halo(2) / conv_wgrad kernels (%d implicit-GEMM calls per "
                                   "step)" % len(recs),
                         "conv": {"achieved": conv_tf, "frac_conv": conv_tf / peaks["bf16_tflops"],
                                  "flops_issued_per_step": conv_flops_issued, "ms_per_step": conv_ms,
                                  "share_of_step": conv_ms / ms,
                                  "what": "FLOPs issued by the implicit-GEMM launches (de-padded shapes) / their summed "
                                          "CUDA-event time in an instrumented eager pass"},
                         "traffic_note": "DRAM read+write bytes of the implicit-GEMM launches of one step, from the "
                                         "committed ncu launch list profiles/r02_step_launches.csv (tools/ncu_traffic.py)"
                                         "; algorithmic operand bytes of the same launches: see DESIGN.md 3.1",
                         "peak_source": peaks["source"]},
        }
        if world > 1 and getattr(tr, "comm_stats", None):
            line["allreduce"] = tr.comm_stats()
        if world == 1 and args.config == 2:
            if not args.no_cpu_baseline:
                line["cpu_baseline"] = cpu_reference_throughput(args.size[0], args.cpu_steps)
            if not args.no_incumbent:
                line["incumbent_gpu"] = gpu_incumbent(args.size[0])
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
