"""GPU parity: every operator of the `gsplatcu` surface (through the C ABI) against the CPU
oracle on the same seeded inputs, plus the reference-generated golden fixtures.

Tolerances (fp32 device arithmetic vs fp64 oracle on identical fp32 inputs):
  * integer / index outputs (areas, patch ranges, gsid_per_patch, culls, contrib): exact;
  * per-Gaussian values and Jacobians: elementwise |err| <= 2e-5 |ref| + 4e-6 max|ref|
    on random scenes, and the reference's own abs-1e-4 `check` (backward_cpu.py:61-65) on the
    reference-generated fixture;
  * image / final_tau: <= 5e-5 abs on pixels whose threshold decisions are unambiguous,
    <= 1e-2 on the (rare, counted) pixels the oracle flags as within 2e-5 of a threshold;
  * splatB gradients: max|err| / max|ref| <= 1e-4 (north_star) per tensor.
"""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from easygaussiansplatting_b200.scene import synthetic_scene, upstream_gradient

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
DEV = "cuda:0"


def gsc():
    import gsplatcu
    return gsplatcu


def t(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).to(DEV)


def n(x):
    return x.detach().cpu().numpy()


def check_vals(got, ref, name, rtol=2e-5, atol_scale=4e-6):
    """elementwise |got - ref| <= rtol |ref| + atol_scale * max|ref| (fp32 vs fp64)"""
    got = n(got).astype(np.float64).reshape(ref.shape)
    if not ref.size:
        return
    scale = max(np.max(np.abs(ref)), 1e-30)
    excess = np.abs(got - ref) - (rtol * np.abs(ref) + atol_scale * scale)
    i = np.argmax(excess)
    assert excess.flat[i] <= 0, "%s: got %r want %r (scale %.3g)" % (name, got.flat[i], ref.flat[i], scale)


def stage_pipeline(sc, calc_J=True):
    """runs the five per-Gaussian ops on the GPU; returns dict of torch tensors"""
    g = gsc()
    W, H = sc["width"], sc["height"]
    pws, rots, scales, shs = t(sc["pws"]), t(sc["rots"]), t(sc["scales"]), t(sc["shs"])
    Rcw, tcw, twc = t(sc["Rcw"]), t(sc["tcw"]), t(sc["twc"])
    o = {}
    r = g.project(pws, Rcw, tcw, sc["fx"], sc["fy"], sc["cx"], sc["cy"], calc_J)
    o["us"], o["pcs"], o["depths"] = r[:3]
    r3 = g.computeCov3D(rots, scales, o["depths"], calc_J)
    r2 = g.computeCov2D(r3[0], o["pcs"], Rcw, o["depths"], sc["fx"], sc["fy"], W, H, calc_J)
    rc = g.sh2Color(shs, pws, twc, calc_J)
    ri = g.inverseCov2D(r2[0], o["depths"], calc_J)
    o.update(cov3ds=r3[0], cov2ds=r2[0], colors=rc[0], cinv2ds=ri[0], areas=ri[1])
    if calc_J:
        o.update(du_dpcs=r[3], dcov3d_drots=r3[1], dcov3d_dscales=r3[2], dcov2d_dcov3ds=r2[1],
                 dcov2d_dpcs=r2[2], dcolor_dshs=rc[1], dcolor_dpws=rc[2], dcinv2d_dcov2ds=ri[2])
    return o


def scene_with_culls(N, W, H, sh_dim, seed):
    sc = synthetic_scene(N, W, H, sh_dim=sh_dim, seed=seed)
    rng = np.random.default_rng(seed + 17)
    idx = rng.choice(N, size=max(1, N // 50), replace=False)
    sc["pws"][idx, 2] = rng.uniform(-1.0, 0.19, len(idx)).astype(np.float32)  # behind / too close
    wide = rng.choice(N, size=max(1, N // 50), replace=False)
    sc["pws"][wide, 0] *= 6.0  # outside the 1.3*tan_fov cone -> clamp active
    if seed % 2 == 1:  # a general camera pose and un-normalised quaternions
        a, b = 0.15, -0.08
        Ry = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
        Rx = np.array([[1, 0, 0], [0, np.cos(b), -np.sin(b)], [0, np.sin(b), np.cos(b)]])
        sc["Rcw"] = (Ry @ Rx).astype(np.float32)
        sc["tcw"] = np.array([0.3, -0.2, 0.4], np.float32)
        sc["twc"] = (-(sc["Rcw"].astype(np.float64).T @ sc["tcw"].astype(np.float64))).astype(np.float32)
        sc["rots"] = (sc["rots"] * rng.uniform(0.8, 1.25, (N, 1))).astype(np.float32)
    return sc


# ---------------------------------------------------------------- per-Gaussian stages
@pytest.mark.parametrize("N,sh_dim", [(1, 48), (127, 3), (128, 12), (4999, 27), (20000, 48)])
def test_stages_vs_oracle(N, sh_dim):
    sc = scene_with_culls(N, 320, 240, sh_dim, seed=N)
    W, H = sc["width"], sc["height"]
    o = stage_pipeline(sc)
    us, pcs, depths, J = orc.project(sc["pws"], sc["Rcw"], sc["tcw"], sc["fx"], sc["fy"], sc["cx"], sc["cy"])
    d_gpu = n(o["depths"])
    culled = depths < 0
    z64 = sc["pws"].astype(np.float64) @ sc["Rcw"].astype(np.float64)[2] + float(sc["tcw"][2])
    amb = np.abs(z64 - 0.2) < 1e-5
    assert np.array_equal((d_gpu < 0)[~amb], culled[~amb])
    check_vals(o["us"], us, "us"); check_vals(o["pcs"], pcs, "pcs"); check_vals(o["du_dpcs"], J, "du_dpcs")
    check_vals(o["depths"], depths, "depths")
    # downstream ops are checked on the GPU's own fp32 inputs (what the op actually received)
    d32 = d_gpu.astype(np.float32).copy()
    cov3, J3r, J3s = orc.compute_cov3d(sc["rots"], sc["scales"], d32)
    check_vals(o["cov3ds"], cov3, "cov3ds"); check_vals(o["dcov3d_drots"], J3r, "dcov3d_drots")
    check_vals(o["dcov3d_dscales"], J3s, "dcov3d_dscales")
    cov2, J2c, J2p, cl = orc.compute_cov2d(n(o["cov3ds"]), n(o["pcs"]), sc["Rcw"], d32, sc["fx"], sc["fy"],
                                           W, H, return_clamped=True)
    if N >= 100:
        assert cl.any(), "scene should exercise the fov clamp"
    check_vals(o["cov2ds"], cov2, "cov2ds")
    check_vals(o["dcov2d_dcov3ds"], J2c, "dcov2d_dcov3ds")
    check_vals(o["dcov2d_dpcs"], J2p, "dcov2d_dpcs")
    col, Jcs, Jcp = orc.sh2color(sc["shs"], sc["pws"], sc["twc"])
    check_vals(o["colors"], col, "colors"); check_vals(o["dcolor_dshs"], Jcs, "dcolor_dshs")
    check_vals(o["dcolor_dpws"], Jcp, "dcolor_dpws")
    d_before = d32.copy()
    cinv, areas, Jci = orc.inverse_cov2d(n(o["cov2ds"]), d32)
    assert np.array_equal(d32, d_before)  # no NaN determinants in this scene
    check_vals(o["cinv2ds"], cinv, "cinv2ds"); check_vals(o["dcinv2d_dcov2ds"], Jci, "dcinv2d_dcov2ds")
    assert np.array_equal(n(o["areas"]), areas), "areas must be bit-exact"
    # culled rows are all-zero in every output (reference: torch::full zero fill)
    for k in ("us", "pcs", "cov3ds", "cov2ds", "cinv2ds", "du_dpcs", "dcov3d_drots", "dcov2d_dpcs",
              "dcinv2d_dcov2ds"):
        assert not n(o[k])[d_gpu < 0].any(), k
    assert not n(o["areas"])[d_gpu < 0].any()


def test_stages_no_jacobian_matches_with_jacobian():
    sc = scene_with_culls(3000, 320, 240, 48, seed=5)
    a, b = stage_pipeline(sc, True), stage_pipeline(sc, False)
    for k in ("us", "pcs", "depths", "cov3ds", "cov2ds", "colors", "cinv2ds", "areas"):
        assert torch.equal(a[k], b[k]), k


def test_stages_golden_reference_fixture():
    """values + Jacobians the reference's backward_cpu.py produced (tests/golden/stages.npz),
    with the reference's own abs-1e-4 criterion"""
    st = dict(np.load(os.path.join(G, "stages.npz")))
    fx, fy, cx, cy, W, H = st["cam"]
    g = gsc()
    us, pcs, depths, J = g.project(t(st["pws"]), t(st["Rcw"]), t(st["tcw"]), fx, fy, cx, cy, True)
    ok = lambda a, b: np.all(np.abs(n(a).astype(np.float64).reshape(b.shape) - b) < 1e-4)
    assert ok(us, st["us"]) and ok(pcs, st["pcs"]) and ok(J, st["du_dpcs"])
    c3, J3r, J3s = g.computeCov3D(t(st["rots"]), t(st["scales"]), depths, True)
    assert ok(c3, st["cov3ds"]) and ok(J3r, st["dcov3d_drots"]) and ok(J3s, st["dcov3d_dscales"])
    c2, J2c, J2p = g.computeCov2D(c3, pcs, t(st["Rcw"]), depths, fx, fy, W, H, True)
    assert ok(c2, st["cov2ds"]) and ok(J2c, st["dcov2d_dcov3ds"]) and ok(J2p, st["dcov2d_dpcs"])
    col, Jcs, Jcp = g.sh2Color(t(st["shs"]), t(st["pws"]), t(st["twc"]), True)
    assert ok(col, st["colors"]) and ok(Jcs, st["dcolor_dshs"]) and ok(Jcp, st["dcolor_dpws"])
    for k in (1, 4, 9):
        assert ok(g.sh2Color(t(st["shs"][:, :3 * k]), t(st["pws"]), t(st["twc"]), False)[0], st["colors_k%d" % k])
    ci, areas, Jci = g.inverseCov2D(c2, depths, True)
    assert ok(ci, st["cinv2ds"])
    # dcinv/dcov reaches ~1e2 here: compare relatively
    check_vals(Jci, st["dcinv2d_dcov2ds"], "dcinv2d_dcov2ds")


def test_inverse_cov2d_nan_cull():
    g = gsc()
    cov = t(np.array([[np.inf, np.inf, np.inf], [2, 0.5, 3], [np.nan, 0, 1]], dtype=np.float32))
    d = t(np.array([1, 2, 3], dtype=np.float32))
    cinv, areas, J = g.inverseCov2D(cov, d, True)
    assert n(d).tolist() == [-1.0, 2.0, -1.0]
    assert not n(cinv)[[0, 2]].any() and not n(areas)[[0, 2]].any() and not n(J)[[0, 2]].any()
    assert n(areas)[1].tolist() == [5, 6]


# ---------------------------------------------------------------- splat / splatB
def run_splat_case(N, W, H, sh_dim=3, seed=0, check_bwd=True, sc=None, tol_scale=1.0):
    # tol_scale > 1 only for adversarial scenes whose fp32 Mahalanobis terms cancel (see the
    # huge/needle test); every BASELINE-shaped case runs at 1.
    g = gsc()
    sc = sc or scene_with_culls(N, W, H, sh_dim, seed)
    o = stage_pipeline(sc, calc_J=False)
    alphas = t(sc["alphas"])
    us, cinv, col = n(o["us"]), n(o["cinv2ds"]), n(o["colors"])
    d_in, a_in = n(o["depths"]).copy(), n(o["areas"]).copy()
    image, contrib, ftau, ranges, gsid = g.splat(H, W, o["us"], o["cinv2ds"], alphas, o["depths"], o["colors"],
                                                 o["areas"])
    d_or, a_or = d_in.copy(), a_in.copy()
    ref = orc.splat(H, W, us, cinv, sc["alphas"], d_or, col, a_or, margin=2e-5 * tol_scale)
    # integer side: bit exact, including the in-place culls
    assert np.array_equal(n(o["depths"]), d_or), "in-place depth cull differs"
    assert np.array_equal(n(o["areas"]), a_or), "in-place areas cull differs"
    assert gsid.numel() == ref["P"]
    assert np.array_equal(n(ranges), ref["ranges"]), "patch_range_per_tile differs"
    assert np.array_equal(n(gsid), ref["gsid"]), "gsid_per_patch (sort order) differs"
    amb = ref["ambiguous"]
    frac = amb.mean()
    assert frac < 5e-3 * tol_scale, "too many ambiguous pixels: %g" % frac
    img = n(image).astype(np.float64)
    err = np.abs(img - ref["image"]).max(axis=0)
    assert err[~amb].max(initial=0) <= 5e-5 * tol_scale, "image err %.3e" % err[~amb].max()
    assert err.max(initial=0) <= 1e-2, "ambiguous-pixel image err %.3e" % err.max()
    assert np.array_equal(n(contrib)[~amb], ref["contrib"][~amb]), "contrib differs"
    terr = np.abs(n(ftau).astype(np.float64) - ref["final_tau"])
    assert terr[~amb].max(initial=0) <= 1e-5 * tol_scale, "final_tau err %.3e" % terr[~amb].max()
    if not check_bwd:
        return sc, o, (image, contrib, ftau, ranges, gsid), ref
    dl = upstream_gradient(W, H, seed) * (3.0 * W * H)  # O(1) upstream gradient
    grads = g.splatB(H, W, o["us"], o["cinv2ds"], alphas, o["depths"], o["colors"], contrib, ftau, ranges, gsid,
                     t(dl))
    *refg, amb_gs = orc.splat_backward(H, W, us, cinv, sc["alphas"], col, ref, dl, return_ambiguous=True,
                                         margin=2e-5 * tol_scale)
    # Gaussians with a replayed alpha' within 2e-5 of the 0.002 skip threshold may take the
    # other branch in fp32, which moves their own gradient by one whole pixel term (the conic
    # term carries dx^2): bounded separately and counted.
    assert amb_gs.mean() <= 0.01 * tol_scale, "too many threshold-ambiguous Gaussians: %g" % amb_gs.mean()
    for got, want, name in zip(grads, refg, ("dloss_dus", "dloss_dcinv2ds", "dloss_dalphas", "dloss_dcolors")):
        assert tuple(got.shape) == want.shape, name
        err = np.abs(n(got).astype(np.float64) - want).reshape(len(want), -1).max(axis=1)
        s = np.abs(want).max(initial=1e-30)
        assert err[~amb_gs].max(initial=0) / s <= 1e-4 * tol_scale, "%s: normalised max err %.3e" % (
            name, err[~amb_gs].max() / s)
        assert err.max(initial=0) / s <= 5e-3 * tol_scale, "%s: ambiguous-Gaussian err %.3e" % (name, err.max() / s)
    return sc, o, (image, contrib, ftau, ranges, gsid), ref


@pytest.mark.parametrize("N,W,H", [(10000, 256, 256),      # BASELINE config 1 shape
                                   (3000, 250, 130),       # ragged right / bottom tiles
                                   (50000, 512, 512),      # config 4 corner
                                   (4001, 320, 200),       # rotated camera, un-normalised quaternions
                                   (200, 64, 48)])
def test_splat_and_splatB_vs_oracle(N, W, H):
    run_splat_case(N, W, H, seed=N)


def test_splat_dense_early_termination():
    """many opaque layers: every pixel reaches tau < 1e-4 long before the list ends, and a
    tile's list spans several shared-memory batches"""
    W, H, N = 96, 64, 6000
    sc = synthetic_scene(N, W, H, sh_dim=3, seed=11)
    sc["alphas"][:] = np.random.default_rng(1).uniform(0.6, 0.99, N).astype(np.float32)
    sc["scales"] *= 3.0
    _, _, (image, contrib, ftau, ranges, gsid), ref = run_splat_case(N, W, H, sc=sc, seed=11)
    lens = ref["ranges"][:, 1] - ref["ranges"][:, 0]
    assert lens.max() > 300 and (ref["final_tau"] < 1e-4).mean() > 0.5
    assert ref["contrib"].max() < lens.max()


def test_splat_alpha_clamp_and_tiny_alpha():
    W, H, N = 80, 80, 400
    sc = synthetic_scene(N, W, H, sh_dim=3, seed=2)
    sc["alphas"][::3] = 1.0          # alpha' clamps at 0.99 near the centre (kernel.cu:245)
    sc["alphas"][1::7] = 0.001       # can never reach 0.002
    sc["alphas"][2::11] = 0.002
    run_splat_case(N, W, H, sc=sc, seed=2)


def test_splat_huge_and_needle_gaussians():
    """footprints covering hundreds of tiles, extreme anisotropy (needles at 45 degrees) and
    Gaussians centred far outside the frame whose 3-sigma box still reaches it"""
    W, H, N = 400, 304, 3000
    sc = synthetic_scene(N, W, H, sh_dim=3, seed=13)
    rng = np.random.default_rng(13)
    big = rng.choice(N, 40, replace=False)
    sc["scales"][big] *= rng.uniform(20, 60, (40, 1)).astype(np.float32)      # sigma up to ~200 px
    needle = rng.choice(N, 300, replace=False)
    sc["scales"][needle, 0] *= 40.0                                            # 100:1 anisotropy
    sc["scales"][needle, 1:] *= 0.4
    far = rng.choice(N, 100, replace=False)
    sc["pws"][far, 0] *= 1.6                                                   # centres off-screen
    sc["scales"][far] *= 15.0
    sc["alphas"][big] = rng.uniform(0.02, 0.3, 40).astype(np.float32)
    # Integer side (culls, ranges, patch order, contrib) stays bit-exact.  The float side gets
    # 20x the usual bound: along a 100:1 needle the terms a*dx^2, c*dy^2, 2b*dx*dy reach ~1e5
    # and cancel to O(10), so ANY fp32 evaluation (the reference's included) carries ~1e-2
    # absolute noise in the exponent of far pixels; the oracle evaluates it in fp64.
    _, _, out, ref = run_splat_case(N, W, H, sc=sc, seed=13, tol_scale=20.0)
    lens = ref["ranges"][:, 1] - ref["ranges"][:, 0]
    assert ref["P"] > 15 * N and lens.min() > 30      # every tile is covered by the big ones


def test_splat_golden_blend_fixture():
    """image + splatB grads the reference's backward_cpu.py produced (tests/golden/blend.npz)"""
    bl = dict(np.load(os.path.join(G, "blend.npz")))
    fx, fy, cx, cy, W, H = bl["cam"]
    W, H = int(W), int(H)
    g = gsc()
    cov2 = bl["cov2ds"].astype(np.float32)
    areas = t(np.ceil(3 * np.sqrt(cov2[:, [0, 2]])).astype(np.int32), torch.int32)
    depths = t(bl["pws"][:, 2])
    us, cinv, col, al = t(bl["us32"]), t(bl["cinv32"]), t(bl["colors32"]), t(bl["alphas"])
    image, contrib, ftau, ranges, gsid = g.splat(H, W, us, cinv, al, depths, col, areas)
    assert np.all(np.abs(n(image).transpose(1, 2, 0) - bl["image"]) < 1e-4)
    grads = g.splatB(H, W, us, cinv, al, depths, col, contrib, ftau, ranges, gsid, t(bl["dloss_dgammas"]))
    for got, name in zip(grads, ("dloss_dus", "dloss_dcinv2ds", "dloss_dalphas", "dloss_dcolors")):
        assert np.all(np.abs(n(got) - bl[name]) < 1e-4), name
        s = np.abs(bl[name]).max()
        assert np.abs(n(got) - bl[name]).max() / s < 1e-4, name


def test_full_chain_golden_fixture():
    """params -> image -> L1 loss -> parameter grads through the GSFunction mirror, against
    backward_cpu.backward() (tests/golden/blend.npz chain_*), <= 1e-4 normalised"""
    from easygaussiansplatting_b200.gsfunction import Camera, GSFunction
    bl = dict(np.load(os.path.join(G, "blend.npz")))
    fx, fy, cx, cy, W, H = bl["cam"]
    cam = Camera(int(W), int(H), fx, fy, cx, cy, t(bl["Rcw"]), t(bl["tcw"]), t(np.zeros(3, np.float32)))
    P = {k: t(bl[k]).requires_grad_() for k in ("pws", "shs", "scales", "rots")}
    alphas = t(bl["alphas"][:, None]).requires_grad_()
    us = torch.zeros((len(bl["pws"]), 2), device=DEV, requires_grad=True)
    image, mask = GSFunction.apply(P["pws"], P["shs"], alphas, P["scales"], P["rots"], us, cam)
    gt = t(bl["image_gt"].transpose(2, 0, 1))
    loss = torch.nn.functional.l1_loss(image, gt)
    loss.backward()
    assert abs(loss.item() - float(bl["chain_loss"][0])) < 1e-5
    assert mask.all()
    for name, ref in (("rots", "chain_drots"), ("scales", "chain_dscales"), ("shs", "chain_dshs"),
                      ("pws", "chain_dpws")):
        e = np.abs(n(P[name].grad) - bl[ref]).max() / np.abs(bl[ref]).max()
        assert e < 1e-4, (name, e)
    e = np.abs(n(alphas.grad) - bl["chain_dalphas"]).max() / np.abs(bl["chain_dalphas"]).max()
    assert e < 1e-4, ("alphas", e)


# ---------------------------------------------------------------- degenerate inputs
def test_empty_and_all_culled():
    g = gsc()
    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=DEV)
    out = g.splat(40, 50, z(0, 2), z(0, 3), z(0), z(0), z(0, 3), z(0, 2, dt=torch.int32))
    assert out[0].shape == (3, 40, 50) and not out[0].any() and out[4].numel() == 0 and not out[2].any()
    assert g.project(z(0, 3), torch.eye(3, device=DEV), z(3), 1, 1, 0, 0, True)[3].shape == (0, 2, 3)
    # all Gaussians culled by depth -> P == 0
    N = 10
    d = torch.full((N,), -1.0, device=DEV)
    out = g.splat(32, 32, z(N, 2), z(N, 3), z(N), d, z(N, 3), z(N, 2, dt=torch.int32))
    assert out[4].numel() == 0 and not out[0].any() and not out[1].any()
    gr = g.splatB(32, 32, z(N, 2), z(N, 3), z(N), d, z(N, 3), out[1], out[2], out[3], out[4], z(3, 32, 32))
    assert all(not x.any() for x in gr) and gr[0].shape == (N, 1, 2)


def test_single_patch():
    """P == 1: the reference never closes the range (kernel.cu:140-143); we render it"""
    g = gsc()
    us = t(np.array([[8.0, 8.0]], np.float32)); cinv = t(np.array([[0.5, 0.0, 0.5]], np.float32))
    al = t(np.array([0.8], np.float32)); d = t(np.array([1.5], np.float32))
    col = t(np.array([[1.0, 0.5, 0.25]], np.float32)); ar = t(np.array([[5, 5]], np.int32), torch.int32)
    image, contrib, ftau, ranges, gsid = g.splat(16, 16, us, cinv, al, d, col, ar)
    assert gsid.tolist() == [0] and ranges.tolist() == [[0, 1]]
    assert abs(image[0, 8, 8].item() - 0.8) < 1e-6 and contrib[8, 8].item() == 1


def test_input_validation_raises():
    g = gsc()
    with pytest.raises(ValueError):
        g.project(torch.zeros(4, 3), torch.eye(3), torch.zeros(3), 1, 1, 0, 0, True)  # CPU tensors
    with pytest.raises(TypeError):
        g.project(torch.zeros(4, 3, device=DEV, dtype=torch.float64), torch.eye(3, device=DEV),
                  torch.zeros(3, device=DEV), 1, 1, 0, 0, True)
    with pytest.raises(ValueError):
        g.sh2Color(torch.zeros(4, 15, device=DEV), torch.zeros(4, 3, device=DEV), torch.zeros(3, device=DEV), False)


def test_non_contiguous_inputs():
    g = gsc()
    sc = synthetic_scene(500, 64, 64, sh_dim=12, seed=9)
    big = t(np.concatenate([sc["pws"], sc["pws"]], axis=1))  # [N,6]; slice is non-contiguous
    pws_nc = big[:, :3]
    assert not pws_nc.is_contiguous()
    a = g.project(pws_nc, t(sc["Rcw"]), t(sc["tcw"]), sc["fx"], sc["fy"], sc["cx"], sc["cy"], False)
    b = g.project(t(sc["pws"]), t(sc["Rcw"]), t(sc["tcw"]), sc["fx"], sc["fy"], sc["cx"], sc["cy"], False)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    # unaligned (offset) views take the scalar path
    off = t(np.concatenate([np.zeros(1, np.float32), sc["pws"].reshape(-1)]))[1:].view(-1, 3)
    c = g.project(off, t(sc["Rcw"]), t(sc["tcw"]), sc["fx"], sc["fy"], sc["cx"], sc["cy"], False)
    assert all(torch.equal(x, y) for x, y in zip(c, b))


# ---------------------------------------------------------------- full size (BASELINE config 2)
def test_config2_full_size_properties_and_oracle():
    """1M Gaussians, 1920x1080, SH degree 3: forward + backward vs the oracle at full size
    (the C oracle takes seconds with OpenMP), plus size-independent properties."""
    N, W, H = 1_000_000, 1920, 1080
    sc = synthetic_scene(N, W, H, sh_dim=48, seed=0)
    sc, o, (image, contrib, ftau, ranges, gsid), ref = run_splat_case(N, W, H, sc=sc, seed=0)
    r = n(ranges)
    lens = r[:, 1] - r[:, 0]
    assert lens.sum() == gsid.numel() and 2_000_000 < gsid.numel() < 3_200_000
    # sortedness: within each tile depth keys are non-decreasing, ties by ascending id
    g_ids = n(gsid).astype(np.int64)
    dk = (n(o["depths"]).astype(np.float32) * np.float32(1000.0)).astype(np.uint32).astype(np.int64)
    key = dk[g_ids] * (1 << 21) + g_ids
    tile_of = np.repeat(np.arange(len(r)), lens)
    full = tile_of * (1 << 53) + key
    assert np.all(np.diff(full) > 0)
    # idempotence: rendering twice gives bit-identical forward outputs
    g = gsc()
    again = g.splat(H, W, o["us"], o["cinv2ds"], t(sc["alphas"]), o["depths"], o["colors"], o["areas"])
    assert torch.equal(again[0], image) and torch.equal(again[1], contrib) and torch.equal(again[4], gsid)
    # transmittance bound: 0 <= tau <= 1 and image finite
    assert torch.isfinite(image).all() and ftau.min() >= 0 and ftau.max() <= 1


def test_reference_backward_gpu_script_checks():
    """The 19 checks of the reference's parity script backward_gpu.py (81-152): its operator call
    sequence on its 4-Gaussian example scene at 32x16, every output and Jacobian, the image and
    splatB's four gradients against what its backward_cpu.py computed (tests/golden/scripts.npz,
    make_golden_scripts.py), each with the script's abs-1e-4 `check`.  Then the inference call
    sequence of forward_gpu.py (47-60) on the same Gaussians at 979x546."""
    d = dict(np.load(os.path.join(G, "scripts.npz")))
    g = gsc()
    fx, fy, cx, cy, W, H = d["cam"]
    W, H = int(W), int(H)
    pws, rots, scales, alphas, shs = (t(d[k]) for k in ("pws", "rots", "scales", "alphas", "shs"))
    Rcw, tcw, twc = t(d["Rcw"]), t(d["tcw"]), t(d["twc"])
    us, pcs, _, du_dpcs = g.project(pws, Rcw, tcw, fx, fy, cx, cy, True)
    depths = t(np.array([1, 2, 3, 4]))  # the script's fixed depths, not the projected ones
    c3, J3r, J3s = g.computeCov3D(rots, scales, depths, True)
    c2, J2c, J2p = g.computeCov2D(c3, pcs, Rcw, depths, fx, fy, W, H, True)
    col, Jcs, Jcp = g.sh2Color(shs, pws, twc, True)
    ci, areas, Jci = g.inverseCov2D(c2, depths, True)
    image, contrib, ftau, ranges, gsid = g.splat(H, W, us, ci, alphas, depths, col, areas)
    grads = g.splatB(H, W, us, ci, alphas, depths, col, contrib, ftau, ranges, gsid, t(d["dloss_dgammas"]))
    got = dict(us=us, pcs=pcs, du_dpcs=du_dpcs, cov3ds=c3, dcov3d_drots=J3r, dcov3d_dscales=J3s, cov2ds=c2,
               dcov2d_dcov3ds=J2c, dcov2d_dpcs=J2p, colors=col, dcolor_dshs=Jcs, dcolor_dpws=Jcp, cinv2ds=ci,
               dcinv2d_dcov2ds=Jci, image=image.permute(1, 2, 0))
    got.update(zip(("dloss_dus", "dloss_dcinv2ds", "dloss_dalphas", "dloss_dcolors"), grads))
    failed = [k for k, v in got.items() if not np.all(np.abs(n(v).astype(np.float64).reshape(d[k].shape) - d[k]) < 1e-4)]
    assert len(got) == 19 and not failed, failed
    # forward_gpu.py: deg-0 colours, its own camera; it passes (height, width) to computeCov2D in that order
    fx, fy, W, H = 581.6273640151177, 578.140202494143, 979, 546
    twc = torch.linalg.inv(Rcw) @ (-tcw)
    us, pcs, depths = g.project(pws, Rcw, tcw, fx, fy, W / 2, H / 2, False)
    c3 = g.computeCov3D(rots, scales, depths, False)[0]
    c2 = g.computeCov2D(c3, pcs, Rcw, depths, fx, fy, H, W, False)[0]
    col = g.sh2Color(shs[:, :3].contiguous(), pws, twc, False)[0]
    ci, areas = g.inverseCov2D(c2, depths, False)
    image = g.splat(H, W, us, ci, alphas, depths, col, areas)[0]
    assert list(image.shape) == [3, 546, 979] and float(image.max()) > 0.1


@pytest.mark.parametrize("N,W,H", [(2_000_000, 1920, 1080), (5_000_000, 3840, 2160)])
def test_large_configs_vs_oracle(N, W, H):
    """BASELINE config 5's scene size (2M Gaussians at 1080p) and config 4's largest corner
    (5M at 4K: 32 400 tiles, 15 tile bits + 14 depth bits = 8-bit digits, 4 sort passes) against the
    oracle at full size: culls, ranges and sort order bit-exact, image / gradients within the
    BASELINE-shaped tolerances of run_splat_case."""
    sc = synthetic_scene(N, W, H, sh_dim=12, seed=2)
    sc, o, (image, contrib, ftau, ranges, gsid), ref = run_splat_case(N, W, H, sc=sc, seed=2)
    assert 2.0 * N < gsid.numel() < 3.2 * N
