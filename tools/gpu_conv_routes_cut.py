"""Which conv kernel each CUT production-shape case launches (tests/test_gpu_production_shapes_cut.py CONV_CASES):
one forward + backward per case under torch.profiler, printing the CUDA kernels of the conv launchers by name
(conv_fwd_kernel / conv_wgrad_kernel = generic implicit GEMM; *halo* = the halo-reuse kernels, *halo2* = CTA pairs).
JG_NO_HALO / JG_CONV_2CTA / JG_WGRAD_2CTA change the routes as they do for the tests.

    python tools/gpu_conv_routes_cut.py > routes.txt
"""
import os
import re
import sys

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import test_gpu_production_shapes_cut as T  # noqa: E402

SHOW = re.compile(r"conv|wgrad|halo|unpack|dilate|pad2d|act_bwd|bias_grad")


def short(name):
    name = re.sub(r"\(.*", "", name)          # drop the argument list
    return name.replace("void ", "").replace("jg::", "")


def main():
    for case in T.CONV_CASES:
        n, name, kind, cin, cout, k, stride, pad, reflect, act, size = case
        mod = T._make_module(kind, cin, cout, k, stride, pad, "cuda")
        x = T._nhwc(torch.randn(n, cin, size, size, device="cuda"), T._c8(cin)).requires_grad_(True)
        for _ in range(2):   # the second pass is the one recorded (module loads and TMA descriptors warmed up)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                y = T._run_layer(mod, kind, stride, pad, reflect, act, x)
                y.backward(torch.randn_like(y, dtype=torch.float32).bfloat16())
                torch.cuda.synchronize()
            mod.zero_grad()
            x.grad = None
        names = [short(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        print("n%d_%s: %s" % (n, name, " | ".join(s for s in names if SHOW.search(s))))


if __name__ == "__main__":
    main()
