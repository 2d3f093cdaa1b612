"""N2 (loss) and N3 (density) kernels on seeded inputs: per-kernel ms from the library's own
CUDA-event profile + SHA-1 prefixes of the outputs, one JSON line.  Two builds (GSB_LIB, see
ab_variants.py) compute the same thing exactly when their `grad_sha`, `cls_slots_sha` and `out_sha`
agree:  python benchmarks/ab_n2n3.py [--once] [--hw 1080x1920] [--n 1000000]"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from easygaussiansplatting_b200 import _lib, density as dn  # noqa: E402
from easygaussiansplatting_b200.loss import gau_loss_with_grad  # noqa: E402


def kernel_ms(lib, fn, reps):
    fn(); torch.cuda.synchronize()
    lib.gsb_profile_enable(1)
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    lib.gsb_profile_enable(0)
    out = {}
    for i in range(lib.gsb_profile_kernels()):
        ms, cnt = C.c_double(0), C.c_longlong(0)
        lib.gsb_profile_read(i, C.byref(ms), C.byref(cnt))
        if cnt.value:
            out[lib.gsb_profile_kernel_name(i).decode()] = ms.value / reps
    return out


def sha(*ts):
    h = hashlib.sha1()
    for t in ts:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--once", action="store_true", help="one call of each (for ncu)")
    ap.add_argument("--hw", default="1080x1920")
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--skip-density", action="store_true")
    a = ap.parse_args()
    H, W = (int(x) for x in a.hw.split("x"))
    dev = torch.device("cuda:0")
    lib = _lib.load()
    reps = 1 if a.once else 20
    g = torch.Generator(device=dev).manual_seed(7)
    yy, xx = torch.meshgrid(torch.arange(H, device=dev), torch.arange(W, device=dev), indexing="ij")
    base = torch.stack([0.5 + 0.4 * torch.sin(xx / 9.0 + c) * torch.cos(yy / 6.0 - c) for c in range(3)])
    img = (base + 0.08 * torch.randn(base.shape, device=dev, generator=g)).clamp(-0.2, 1.3).contiguous()
    gt = (base + 0.02 * torch.randn(base.shape, device=dev, generator=g)).clamp(0, 1).contiguous()
    res = {"env": {k: v for k, v in os.environ.items() if k.startswith("GSB_")}, "hw": [H, W]}
    loss, grad = gau_loss_with_grad(img, gt)
    res["loss"] = {"value": float(loss.item()), "grad_sha": sha(grad), "grad_abs_sum": float(grad.abs().sum().item())}
    res["loss"]["kernels_ms"] = kernel_ms(lib, lambda: gau_loss_with_grad(img, gt), reps)
    res["loss"]["total_ms"] = sum(res["loss"]["kernels_ms"].values())
    res["loss"]["hbm_GBps_on_132B_per_px"] = 132 * H * W / (res["loss"]["total_ms"] * 1e-3) / 1e9
    if not a.skip_density:
        N = a.n
        widths = dict(zip(dn.GAUSSIAN_TENSORS, dn.GAUSSIAN_WIDTHS))
        P = {k: torch.randn((N, w), device=dev, generator=g) for k, w in widths.items()}
        P["alphas_raw"] = torch.rand((N, 1), device=dev, generator=g) * 11.5 - 7.5
        P["scales_raw"] = torch.log(torch.exp(torch.rand((N, 1), device=dev, generator=g) * 4.1 - 4.6) *
                                    (torch.rand((N, 3), device=dev, generator=g) * 0.9 + 0.6))
        M = {k: torch.randn_like(v) * 1e-3 for k, v in P.items()}
        V = {k: torch.rand_like(v) * 1e-6 for k, v in P.items()}
        cnt = torch.randint(0, 6, (N,), device=dev, generator=g, dtype=torch.int32)
        acc = torch.randn((N, 1), device=dev, generator=g).abs() * 1.5e-6
        th = dn.raw_thresholds(5.0)
        cls, slots, counts = dn.plan(P["alphas_raw"], P["scales_raw"], acc, cnt, th)
        z = torch.randn((counts[2], 3), device=dev, generator=g)
        dst, dm, dv = dn.apply(cls, slots, counts, P, M, V, z)
        keys = sorted(dst)
        res["density"] = {"counts": list(counts), "cls_slots_sha": sha(cls, slots),
                          "out_sha": sha(*[dst[k] for k in keys], *[dm[k] for k in keys], *[dv[k] for k in keys])}

        def once():
            c2, s2, n2 = dn.plan(P["alphas_raw"], P["scales_raw"], acc, cnt, th)
            dn.apply(c2, s2, n2, P, M, V, z)
        res["density"]["kernels_ms"] = kernel_ms(lib, once, 1 if a.once else 5)
        K, Cn, S = counts
        by = 2 * 708 * K + 708 * (Cn + S) + 13 * N + 12 * S
        res["density"]["apply_GBps"] = by / (res["density"]["kernels_ms"]["density_apply"] * 1e-3) / 1e9
    print(json.dumps(res))


if __name__ == "__main__":
    main()
