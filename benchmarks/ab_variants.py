#!/usr/bin/env python
"""A/B timing of differently-compiled builds of the library on BASELINE config 2.

Build variants in the dev container (no GPU needed), e.g.
    GSB_VARIANT=E GSB_EXTRA_NVCC_FLAGS="-DBWD4_MINBLOCKS=8" python -m easygaussiansplatting_b200.build
then on the GPU box
    python benchmarks/ab_variants.py            # default build + every libgsplat_b200_*.so found
Each build runs in its own process (GSB_LIB selects the library): 30 timed fused fwd+bwd steps
(CUDA events) and 5 profiled ones (per-kernel CUDA events from the library).  Prints one line per
build; writes gpurun_out/ab_variants.json."""
import glob
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHILD = r"""
import ctypes as C, json, sys
import numpy as np, torch
sys.path.insert(0, %r)
from easygaussiansplatting_b200 import _lib
from easygaussiansplatting_b200.gsfunction import Camera, GSFunctionFused
from easygaussiansplatting_b200.scene import synthetic_scene, upstream_gradient
lib = _lib.load()
N, W, H = 1_000_000, 1920, 1080
dev = "cuda:0"
sc = synthetic_scene(N, W, H, sh_dim=48, seed=0)
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
cam = Camera(W, H, sc["fx"], sc["fy"], sc["cx"], sc["cy"], T(sc["Rcw"]), T(sc["tcw"]), T(sc["twc"]))
P = {k: T(sc[k]).requires_grad_() for k in ("pws", "shs", "scales", "rots")}
al = T(sc["alphas"][:, None]).requires_grad_()
us0 = torch.zeros((N, 2), device=dev, requires_grad=True)
dl = T(upstream_gradient(W, H, 0) * (3.0 * W * H))
def step():
    for p in list(P.values()) + [al]:
        p.grad = None
    image, _ = GSFunctionFused.apply(P["pws"], P["shs"], al, P["scales"], P["rots"], us0, cam)
    image.backward(dl)
for _ in range(5):
    step()
torch.cuda.synchronize()
best = 1e9
for rep in range(3):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        step()
    b.record(); torch.cuda.synchronize()
    best = min(best, a.elapsed_time(b) / 10)
lib.gsb_profile_enable(1)
for _ in range(5):
    step()
torch.cuda.synchronize()
lib.gsb_profile_enable(0)
kern = {}
for i in range(lib.gsb_profile_kernels()):
    ms, cnt = C.c_double(0), C.c_longlong(0)
    lib.gsb_profile_read(i, C.byref(ms), C.byref(cnt))
    if cnt.value:
        kern[lib.gsb_profile_kernel_name(i).decode()] = round(ms.value / 5, 4)
print("RESULT " + json.dumps({"ms_per_step": round(best, 4), "kernels": kern, "checksum": float(P["pws"].grad.abs().sum())}))
"""


def main():
    libs = [("default", "")] + sorted((os.path.basename(p)[len("libgsplat_b200_"):-3], p) for p in
                                      glob.glob(os.path.join(ROOT, "easygaussiansplatting_b200", "libgsplat_b200_*.so")))
    only = set(sys.argv[1:])
    out = {}
    for name, path in libs:
        if only and name not in only:
            continue
        env = dict(os.environ)
        if path:
            env["GSB_LIB"] = path
        r = subprocess.run([sys.executable, "-c", CHILD % ROOT], env=env, capture_output=True, text=True, timeout=600)
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
        if r.returncode != 0 or not line:
            out[name] = {"error": r.stderr[-800:]}
            print(name, "FAILED", r.stderr[-300:])
            continue
        out[name] = json.loads(line[0][7:])
        k = out[name]["kernels"]
        print("%-8s step %.4f ms  draw %.4f  draw_backward %.4f  pack %.4f  checksum %.6g" % (
            name, out[name]["ms_per_step"], k.get("draw", 0), k.get("draw_backward", 0), k.get("pack_records", 0),
            out[name]["checksum"]))
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "ab_variants.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
