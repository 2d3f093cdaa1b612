"""Golden fixture for the reference's own GPU parity script backward_gpu.py (:81-152): imports
the reference's backward_cpu.py and gsplat/gau_io.py on the CPU, builds the script's scene (the
4-Gaussian get_example_gs(), 45 rest-SH coefficients from np.random.rand after
np.random.seed(0), its camera at 32x16) and stores the inputs together with the 19 arrays the
script checks the GPU operators against.  Run with the reference checkout in GS_REFERENCE:

    GS_REFERENCE=<path to EasyGaussianSplatting> python tests/golden/make_golden_scripts.py
"""
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ["GS_REFERENCE"]
sys.path.insert(0, os.path.join(HERE, "..", "shims"))
sys.path.insert(0, REF)
sys.modules.setdefault("gsplatcu", types.ModuleType("gsplatcu"))  # gsplat/utils.py:2

import backward_cpu as bc  # noqa: E402
from gsplat.gau_io import get_example_gs  # noqa: E402


def main():
    np.random.seed(0)
    gs = get_example_gs()
    N, sh_rest_dim = gs.shape[0], 45
    sh_dim = 3 + sh_rest_dim
    shs = np.concatenate((gs["sh"], np.random.rand(N, sh_rest_dim)), axis=1).astype(np.float64)
    tcw = np.array([1.03796196, 0.42017467, 4.67804612])
    Rcw = np.array([[0.89699204, 0.06525223, 0.43720409],
                    [-0.04508268, 0.99739184, -0.05636552],
                    [-0.43974177, 0.03084909, 0.89759429]]).T
    twc = np.linalg.inv(Rcw) @ (-tcw)
    W, H, fx, fy = 32, 16, 16.0, 16.0
    cx, cy = W / 2.0, H / 2.0
    pws, alphas = gs["pw"].astype(np.float64), gs["alpha"].astype(np.float64)
    rots, scales = gs["rot"].astype(np.float64), gs["scale"].astype(np.float64)
    out = {k: [] for k in ("us", "pcs", "du_dpcs", "cov3ds", "dcov3d_drots", "dcov3d_dscales", "cov2ds",
                           "dcov2d_dcov3ds", "dcov2d_dpcs", "colors", "dcolor_dshs", "dcolor_dpws", "cinv2ds",
                           "dcinv2d_dcov2ds")}
    for i in range(N):
        pc, _ = bc.transform(pws[i], Rcw, tcw, True)
        u, du = bc.project(pc, fx, fy, cx, cy, True)
        c3, J3r, J3s = bc.compute_cov_3d(rots[i], scales[i], True)
        c2, J2c, J2p = bc.compute_cov_2d(c3, pc, Rcw, fx, fy, True)
        col, Jcs, Jcp = bc.sh2color(shs[i], pws[i], twc, True)
        ci, Jci = bc.calc_cinv2d(c2, True)
        for k, v in zip(out, (u, pc, du, c3, J3r, J3s, c2, J2c, J2p, col, Jcs, Jcp, ci, Jci)):
            out[k].append(v)
    out = {k: np.stack(v).astype(np.float64) for k, v in out.items()}
    out["dcolor_dshs"] = out["dcolor_dshs"].reshape(N, 1, sh_dim // 3)
    image_gt = np.zeros([H, W, 3])
    image = bc.get_image(alphas, out["cinv2ds"], out["colors"], out["us"], H, W)
    _, dl_dalphas, dl_dcinv2ds, dl_dcolors, dl_dus = bc.calc_loss(alphas, out["cinv2ds"], out["colors"], out["us"],
                                                                  image_gt, True)
    _, dloss_dgammas = bc.get_loss(image, image_gt)
    out.update(pws=pws, rots=rots, scales=scales, alphas=alphas, shs=shs, Rcw=Rcw, tcw=tcw, twc=twc,
               cam=np.array([fx, fy, cx, cy, W, H]), image=image, dloss_dgammas=dloss_dgammas,
               dloss_dus=dl_dus.reshape(N, 1, 2), dloss_dcinv2ds=dl_dcinv2ds.reshape(N, 1, 3),
               dloss_dalphas=dl_dalphas.reshape(N, 1, 1), dloss_dcolors=dl_dcolors.reshape(N, 1, 3))
    np.savez_compressed(os.path.join(HERE, "scripts.npz"), **out)
    print("scripts.npz", N, image.shape, float(image.max()))


if __name__ == "__main__":
    main()
