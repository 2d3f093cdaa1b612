#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: rendered Mpixels/s forward+backward @ 1M Gaussians, 1080p.

A "step" is one pass of the hot path over one synthetic view: parameters -> image ->
(given dL/dimage) -> gradients of every Gaussian parameter.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

ours, N == 1   config[1] of BASELINE.json: 1M synthetic Gaussians, 1920x1080, SH degree 3.
               `value`/`e2e` time the fused path (GSFunctionFused: gsb_preprocess_forward,
               splat, splatB, gsb_preprocess_backward -- every kernel ours).  The same step
               through the reference's seven-operator surface + its torch.bmm Jacobian chain
               (GSFunction mirror of gsplat/gsmodel.py:6-93) is reported beside it as
               `op_surface` (that is what the unmodified reference scripts exercise).
ours, N  > 1   multi-view data parallel (SURVEY 8e): the same shared Gaussians, one camera per
               rank per step, the parameter gradients summed over the ranks by the factorised
               exchange (parallel.MultiViewStep: all-reduce of 44 B/Gaussian + all-gather of the
               12 B/Gaussian dL/dcolor of every view, dL/dsh re-expanded locally); weak scaling
               in views, value = total pixels of all ranks / max-over-ranks time.  The flat
               236 B/Gaussian NCCL all-reduce and the peer-memory exchange are timed beside it.
               `config5`: BASELINE config 5 as written (2M shared Gaussians, 8 cameras per step
               split over the ranks, ONE exchange per step) at every N.
reference      the CPU restatement of the reference algorithm (oracle/, OpenMP pinned to every
               host core) on the SAME workload (whole 1920x1080 frame, all 1M Gaussians,
               forward + backward); rank 0 only.
Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rendered Mpixels/s fwd+bwd @1M Gaussians 1080p; grad max-rel-err vs CPU"
N_GAUSS, WIDTH, HEIGHT, SH_DIM = 1_000_000, 1920, 1080, 48
CROP_ROWS = HEIGHT  # CPU arm: the whole frame (a few seconds per pass with OpenMP on the host cores)
CROP_Y0 = 0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# ------------------------------------------------------------------ CPU arm (oracle port)
def cpu_sample(steps=1, warmup=0):
    """forward + backward of the reference algorithm on the host: per-Gaussian stages with
    Jacobians, tile binning + sort, per-pixel compositing, its backward and the Jacobian chain, on
    the whole 1080p view of the 1M-Gaussian scene, OpenMP threads = os.cpu_count() whatever the
    launcher exported.  Returns (Mpix/s, sec/step, threads, dict with the scene) over `steps` timed
    passes."""
    from oracle import oracle as orc
    from easygaussiansplatting_b200.scene import synthetic_scene, upstream_gradient
    orc.set_num_threads(os.cpu_count() or 1)
    sc = synthetic_scene(N_GAUSS, WIDTH, HEIGHT, sh_dim=SH_DIM, seed=0)
    W, H = WIDTH, CROP_ROWS
    cy = sc["cy"] - CROP_Y0
    dl = upstream_gradient(WIDTH, HEIGHT, 0)[:, CROP_Y0:CROP_Y0 + CROP_ROWS, :].copy() * (3.0 * WIDTH * HEIGHT)
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        us, pcs, depths, Ju = orc.project(sc["pws"], sc["Rcw"], sc["tcw"], sc["fx"], sc["fy"], sc["cx"], cy)
        d32 = f32(depths)
        c3, J3r, J3s = orc.compute_cov3d(sc["rots"], sc["scales"], d32)
        c2, J2c, J2p = orc.compute_cov2d(f32(c3), f32(pcs), sc["Rcw"], d32, sc["fx"], sc["fy"], W, H)
        col, Jcs, Jcp = orc.sh2color(sc["shs"], sc["pws"], sc["twc"])
        ci, areas, Jci = orc.inverse_cov2d(f32(c2), d32)
        fwd = orc.splat(H, W, f32(us), f32(ci), sc["alphas"], d32, f32(col), areas)
        g4 = orc.splat_backward(H, W, f32(us), f32(ci), sc["alphas"], f32(col), fwd, dl)
        orc.chain_backward(sc["Rcw"], *g4, Ju, J3r, J3s, J2c, J2p, Jcs, Jcp, Jci)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    sec = statistics.median(times)
    return W * H / sec / 1e6, sec, orc.num_threads(), dict(scene=sc, cy=cy, dl=dl, passes=len(times))


def sample_text(sec=None, passes=None):
    s = "the whole 1920x1080 view, all 1M Gaussians, SH deg 3, fwd+bwd (same config as the GPU arm)"
    if passes is not None:
        s += ", %d timed pass%s" % (passes, "" if passes == 1 else "es")
    return s + (", %.1f s per pass" % sec if sec is not None else "")


def config1_block():
    """BASELINE config 1 (forward_cpu.py on 10k Gaussians, 256x256, SH deg 0) on this host."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
        import config1_forward_cpu
        return config1_forward_cpu.run(repeats=3, gpu=True)
    except Exception as e:  # never let the side measurement take the bench line down
        return {"error": repr(e)[:200]}


def run_reference(args, rank):
    if rank != 0:
        return
    mpix, sec, threads, info = cpu_sample(steps=max(1, args.steps), warmup=min(1, args.warmup))
    line = {
        "impl": "reference", "metric": METRIC, "value": mpix, "unit": "Mpixels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "config2: 1M synthetic Gaussians, 1920x1080, SH deg 3, fwd+bwd",
                   "gaussians": N_GAUSS, "width": WIDTH, "height": HEIGHT, "sh_dim": SH_DIM},
        "steps_timed": info["passes"],
        "cpu_baseline": {"value": mpix, "unit": "Mpixels/s", "cores": threads, "kind": "port",
                         "sample": sample_text(sec, info["passes"])},
        "e2e": {"value": mpix, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            time.sleep(0.3)
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        sm, mx, reasons, pw = [], None, set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2]); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------ our arm
DUMP_ROWS = 65536  # Gaussians sampled for --dump-outputs: all of dL/dsh alone would be 192 MB


def dump_outputs(out_dir, image, per_gaussian):
    """--dump-outputs: the last timed step's outputs as <out_dir>/<name>.npy, float32.  The image
    whole; every per-Gaussian array on the same fixed, seeded sample of DUMP_ROWS Gaussians (rows
    in ascending order), so that two builds run with the same arguments compare output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rows = torch.from_numpy(np.sort(np.random.default_rng(0).choice(N_GAUSS, DUMP_ROWS, replace=False)))
    np.save(os.path.join(out_dir, "image.npy"), image.detach().float().cpu().numpy())
    for name, a in per_gaussian.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.detach()[rows.to(a.device)].float().cpu().numpy())


def run_ours(args, rank, world):
    import torch
    import torch.distributed as dist
    from easygaussiansplatting_b200 import _lib
    from easygaussiansplatting_b200.gsfunction import Camera, GSFunction, GSFunctionFused
    from easygaussiansplatting_b200.parallel import allreduce_grads
    from easygaussiansplatting_b200.scene import ring_camera, synthetic_scene, upstream_gradient

    # NCCL writes its version banner / diagnostics to stdout; keep stdout to the one JSON line
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    sc = synthetic_scene(N_GAUSS, WIDTH, HEIGHT, sh_dim=SH_DIM, seed=0)  # shared by all ranks
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    if world > 1:
        Rcw, tcw, twc = ring_camera(rank, world)
    else:
        Rcw, tcw, twc = sc["Rcw"], sc["tcw"], sc["twc"]
    cam = Camera(WIDTH, HEIGHT, sc["fx"], sc["fy"], sc["cx"], sc["cy"], T(Rcw), T(tcw), T(twc))
    params = {k: T(sc[k]).requires_grad_() for k in ("pws", "shs", "scales", "rots")}
    alphas = T(sc["alphas"][:, None]).requires_grad_()
    us0 = torch.zeros((N_GAUSS, 2), device=dev, requires_grad=True)
    leaves = [params["pws"], params["shs"], alphas, params["scales"], params["rots"]]
    dl_host = torch.from_numpy(upstream_gradient(WIDTH, HEIGHT, rank) * (3.0 * WIDTH * HEIGHT)).pin_memory()
    dl_dev = dl_host.to(dev)
    cam_host = torch.from_numpy(np.concatenate([np.asarray(Rcw).reshape(-1), tcw, twc]).astype(np.float32)).pin_memory()
    cam_dev = torch.empty(15, device=dev)
    img_host = torch.empty((3, HEIGHT, WIDTH), dtype=torch.float32).pin_memory()
    chk_host = torch.empty(1, dtype=torch.float32).pin_memory()

    # multi-view DP: the parameter gradients are summed over the views, either by the fused
    # exchange (the backward kernel pushes its tiles into peer memory + one reduce/broadcast
    # kernel, parallel.GradExchange) or by an NCCL all-reduce of the flat bucket.  `value` uses
    # what parallel.prefer_fused_exchange(world) selects (measured: the exchange wins at 2 GPUs,
    # NCCL's in-switch reduction at 8); both are always timed and reported in `allreduce`.
    exchange, use_ex = None, False
    if world > 1:
        from easygaussiansplatting_b200.parallel import GradExchange, prefer_fused_exchange
        exchange = GradExchange.from_process_group(N_GAUSS, SH_DIM // 3, dev)
        use_ex = prefer_fused_exchange(world)

    def make_step(F, use_exchange):
        def step(dl):
            for p in leaves:
                p.grad = None
            cam.grad_exchange = exchange if use_exchange else None
            image, mask = F.apply(params["pws"], params["shs"], alphas, params["scales"], params["rots"], us0, cam)
            image.backward(dl)
            if world > 1 and not use_exchange:
                allreduce_grads([p.grad for p in leaves])
            return image, mask
        return step

    step_fused, step_ops = make_step(GSFunctionFused, use_ex), make_step(GSFunction, False)
    step_fused_other = make_step(GSFunctionFused, not use_ex)   # the gradient sum done the other way
    mv, mv_out = None, [None]
    if world > 1:  # the selected multi-GPU step: factorised gradient sum (no autograd involved)
        from easygaussiansplatting_b200.parallel import MultiViewStep
        mv = MultiViewStep(params["pws"].detach(), params["rots"].detach(), params["scales"].detach(),
                           params["shs"].detach(), alphas.detach())

        def step_sel(dl):
            image, ctx = mv.render(cam)
            mv.backward(ctx, dl, last=True)
            mv_out[0] = mv.reduce()
            return image, None
    else:
        step_sel = step_fused

    copy_stream = torch.cuda.Stream(device=dev)
    ev_fwd, ev_dl = torch.cuda.Event(), torch.cuda.Event()

    def step_e2e():
        # host -> device: this view's camera and dL/dimage; device -> host: image + a gradient
        # checksum.  The two 24.9 MB PCIe copies ride a side stream: dL/dimage arrives while the
        # forward runs, the image leaves while the backward runs; the step ends when both
        # streams are done.
        main = torch.cuda.current_stream()
        cam_dev.copy_(cam_host, non_blocking=True)
        cam.Rcw, cam.tcw, cam.twc = cam_dev[:9].view(3, 3), cam_dev[9:12], cam_dev[12:15]
        copy_stream.wait_stream(main)  # the previous backward has finished reading dl_dev
        with torch.cuda.stream(copy_stream):
            dl_dev.copy_(dl_host, non_blocking=True)
            ev_dl.record(copy_stream)
        ctx = None
        if world > 1:
            image, ctx = mv.render(cam)
        else:
            for p in leaves:
                p.grad = None
            cam.grad_exchange = None
            image, _ = GSFunctionFused.apply(params["pws"], params["shs"], alphas, params["scales"], params["rots"],
                                             us0, cam)
        ev_fwd.record(main)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_fwd)
            img = image.detach()
            img.record_stream(copy_stream)
            img_host.copy_(img, non_blocking=True)
        main.wait_event(ev_dl)
        if world > 1:
            mv.backward(ctx, dl_dev, last=True)
            gp = mv.reduce()["dpws"]
        else:
            image.backward(dl_dev)
            gp = params["pws"].grad
        chk_host.copy_(gp.abs().sum().reshape(1), non_blocking=True)
        main.wait_stream(copy_stream)

    def timed(fn, steps, warmup, collective=True):
        """device time of `steps` calls; collective=True (every rank calls it): barrier on both
        sides and the max over ranks.  The rank-0-only legs below pass collective=False."""
        multi = collective and world > 1
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if multi:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if multi:
            dist.barrier()
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = tt.item()
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_sel(dl_dev)
    torch.cuda.synchronize()
    last = {"calls": 0}

    def step_timed():
        # only the last step's outputs are kept: an image held into the next step would change
        # which blocks the caching allocator hands out, and with it the timing
        out = step_sel(dl_dev)
        last["calls"] += 1
        if last["calls"] == args.steps:
            last["out"] = out
    launches0 = lib.gsb_profile_launches(-1)
    ms_dev = timed(step_timed, args.steps, 0)
    launches = lib.gsb_profile_launches(-1) - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # before any later leg replaces the gradients
        # (us0.grad is left out: it is never reset, so it sums every step run so far)
        image, mask = last["out"]
        if world > 1:
            outs = {k: mv_out[0][k] for k in ("dpws", "dshs", "dalphas", "dscales", "drots")}
        else:
            outs = dict(zip(("dpws", "dshs", "dalphas", "dscales", "drots"), (p.grad for p in leaves)), mask=mask)
        dump_outputs(args.dump_outputs, image, outs)
    ms_e2e = timed(step_e2e, args.steps, max(3, args.warmup // 2))
    cam.Rcw, cam.tcw, cam.twc = T(Rcw), T(tcw), T(twc)
    ms_ops = timed(lambda: step_ops(dl_dev), max(3, args.steps // 2), 3)
    ops_steps = max(3, args.steps // 2)
    pix = WIDTH * HEIGHT * world
    value = pix * args.steps / (ms_dev * 1e-3) / 1e6
    e2e = pix * args.steps / (ms_e2e * 1e-3) / 1e6

    allreduce = None
    if world > 1:  # the three ways of summing the gradients, against each other
        nccl_step = step_fused_other if use_ex else step_fused
        ex_step = step_fused if use_ex else step_fused_other
        nccl_step(dl_dev)
        ref_grads = [p.grad.clone() for p in leaves]
        ms_ar = timed(lambda: allreduce_grads([p.grad for p in leaves]), 10, 3)   # grads = flat bucket views
        nbytes = allreduce_grads([p.grad for p in leaves])
        n_other = max(5, args.steps // 2)
        ms_nccl = timed(lambda: nccl_step(dl_dev), n_other, 2) / n_other
        ms_ex = timed(lambda: ex_step(dl_dev), n_other, 2) / n_other
        ex_step(dl_dev)
        torch.cuda.synchronize()
        diff = max(float((p.grad - g).abs().max() / g.abs().max().clamp_min(1e-30)) for p, g in zip(leaves, ref_grads))
        step_sel(dl_dev)
        torch.cuda.synchronize()
        g = mv_out[0]
        fact = [g["dpws"], g["dshs"], g["dalphas"].reshape(-1, 1), g["dscales"], g["drots"]]
        diff_f = max(float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)) for a, b in zip(fact, ref_grads))
        allreduce = {"selected": "factorised (all-reduce 44 B + all-gather 12 B/view per Gaussian, local dL/dsh "
                                 "expansion; parallel.MultiViewStep)",
                     "factorised_bytes_per_rank": g["bytes_per_rank"], "flat_bucket_bytes": int(nbytes),
                     "step_ms_factorised": ms_dev / args.steps,
                     "step_ms_with_nccl_allreduce": ms_nccl, "step_ms_with_fused_exchange": ms_ex,
                     "nccl_flat_allreduce_alone_ms": ms_ar / 10,
                     "nccl_flat_allreduce_algbw_GBps": nbytes / (ms_ar / 10 * 1e-3) / 1e9,
                     "factorised_vs_nccl_max_rel_diff": diff_f,
                     "exchange_vs_nccl_max_rel_diff": diff, "exchange_status": exchange.status()}

    # ---- per-kernel durations with CUDA events on the launch stream (roofline leg)
    prof_steps = 5
    lib.gsb_profile_enable(1)
    for _ in range(prof_steps):
        step_sel(dl_dev)
    torch.cuda.synchronize()
    lib.gsb_profile_enable(0)
    kern = {}
    for i in range(lib.gsb_profile_kernels()):
        ms_tot, cnt = C.c_double(0), C.c_longlong(0)
        lib.gsb_profile_read(i, C.byref(ms_tot), C.byref(cnt))
        if cnt.value:
            kern[lib.gsb_profile_kernel_name(i).decode()] = ms_tot.value / prof_steps
    # ---- the same single-view step replayed as two CUDA graphs (graphed.GraphedFusedStep)
    graphs = None
    if rank == 0:
        try:
            from easygaussiansplatting_b200.graphed import GraphedFusedStep
            gstep = GraphedFusedStep(params["pws"], params["shs"], alphas, params["scales"], params["rots"], cam)

            def graphed_step():
                gstep.forward()
                gstep.dloss_dimage.copy_(dl_dev)
                gstep.backward()
            ms_g = timed(graphed_step, args.steps, 3, collective=False) / args.steps
            graphs = {"what": "forward and backward of this rank's view replayed as CUDA graphs over static buffers "
                              "(capacity-based rasterizer, lazily validated status; dL/dimage copied in between); "
                              "the kernels are launched by the graph, so `gpu_launches` does not see them",
                      "ms_per_step": ms_g, "value": WIDTH * HEIGHT / (ms_g * 1e-3) / 1e6, "unit": "Mpixels/s"}
            del gstep
        except Exception as e:  # noqa: BLE001
            graphs = {"error": repr(e)[:200]}
    config5 = run_config5(torch, dist, dev, rank, world, timed)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- algorithmic bytes of the dominant kernel (SURVEY 8d / BASELINE.md 3)
    from easygaussiansplatting_b200 import ops
    with torch.no_grad():
        us, ci, col, depths, areas = ops.preprocess(params["pws"], params["rots"], params["scales"], params["shs"],
                                                    cam.Rcw, cam.tcw, cam.twc, cam.fx, cam.fy, cam.cx, cam.cy,
                                                    WIDTH, HEIGHT)
        img, contrib, ftau, ranges, gsid = ops.splat(HEIGHT, WIDTH, us, ci, alphas, depths, col, areas)
        P = gsid.numel()
        gy, gx = (HEIGHT + 15) // 16, (WIDTH + 15) // 16
        pad = torch.zeros((gy * 16, gx * 16), dtype=torch.int32, device=dev)
        pad[:HEIGHT, :WIDTH] = contrib
        p_eff = int(pad.view(gy, 16, gx, 16).amax(dim=(1, 3)).sum().item())
    Tn, WH = gx * gy, WIDTH * HEIGHT
    alg = {"draw_backward": 44 * p_eff + 8 * Tn + 20 * WH + 36 * N_GAUSS,
           "draw": 44 * p_eff + 8 * Tn + 20 * WH}
    top = max(kern, key=kern.get)
    roof_k = top if top in alg else "draw_backward"
    peak, peak_src = peaks()
    achieved = alg[roof_k] / (kern[roof_k] * 1e-3) / 1e9
    traffic, traffic_src = None, None   # dram__bytes_read + write per launch from the committed ncu capture
    tpath = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get(roof_k), tj.get("source")
    roofline = {"bound": "hbm", "kernel": roof_k, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg[roof_k], "kernel_ms": kern[roof_k],
                "note": "draw/draw_backward are issue-bound on dense scenes (SURVEY 8d: ~140 flop/B); "
                        "profiles/ holds the ncu pipe utilisation and dram__bytes"}

    # ---- training loss (row N2): fused gau_loss fwd+grad vs the torch chain it replaces
    from easygaussiansplatting_b200.loss import gau_loss_with_grad
    import torch.nn.functional as F
    gt_img = (img.detach() + 0.05 * torch.randn_like(img)).clamp(0, 1)

    def torch_loss():
        x = img.detach().clone().requires_grad_()
        g1 = torch.tensor([np.exp(-(k - 5) ** 2 / 4.5) for k in range(11)], dtype=torch.float32, device=dev)
        g1 = (g1 / g1.sum()).unsqueeze(1)
        win = g1.mm(g1.t()).unsqueeze(0).unsqueeze(0).expand(3, 1, 11, 11).contiguous()
        mu1 = F.conv2d(x, win, padding=5, groups=3); mu2 = F.conv2d(gt_img, win, padding=5, groups=3)
        s11 = F.conv2d(x * x, win, padding=5, groups=3) - mu1.pow(2)
        s22 = F.conv2d(gt_img * gt_img, win, padding=5, groups=3) - mu2.pow(2)
        s12 = F.conv2d(x * gt_img, win, padding=5, groups=3) - mu1 * mu2
        ssim = ((2 * mu1 * mu2 + 1e-4) * (2 * s12 + 9e-4)) / ((mu1.pow(2) + mu2.pow(2) + 1e-4) * (s11 + s22 + 9e-4))
        (0.8 * torch.abs(x - gt_img).mean() + 0.2 * (1 - ssim.mean())).backward()
    ms_loss_fused = timed(lambda: gau_loss_with_grad(img, gt_img), 10, 3, collective=False) / 10
    ms_loss_torch = timed(torch_loss, 5, 2, collective=False) / 5
    loss_bytes = 132 * WH
    loss_info = {"what": "gau_loss forward + dloss/dimage at 1920x1080 (pytorch_ssim.py:64-67 + autograd)",
                 "fused_ms": ms_loss_fused, "torch_chain_ms": ms_loss_torch,
                 "algorithmic_bytes": loss_bytes, "achieved_GBps": loss_bytes / (ms_loss_fused * 1e-3) / 1e9,
                 "hbm_frac": loss_bytes / (ms_loss_fused * 1e-3) / 1e9 / peak}

    # ---- density control (row N3): classify + scan + one-pass rebuild of the 6 parameter
    # tensors and both Adam moments, on the bench scene's N with a synthetic optimizer state
    from easygaussiansplatting_b200 import density as dn
    g = torch.Generator(device=dev).manual_seed(3)
    widths = dict(zip(dn.GAUSSIAN_TENSORS, dn.GAUSSIAN_WIDTHS))
    dP = {k: torch.randn((N_GAUSS, w), device=dev, generator=g) for k, w in widths.items()}
    dP["alphas_raw"] = torch.rand((N_GAUSS, 1), device=dev, generator=g) * 11.5 - 7.5
    dP["scales_raw"] = torch.log(torch.exp(torch.rand((N_GAUSS, 1), device=dev, generator=g) * 4.1 - 4.6) *
                                 (torch.rand((N_GAUSS, 3), device=dev, generator=g) * 0.9 + 0.6))
    dM = {k: torch.randn_like(v) * 1e-3 for k, v in dP.items()}
    dV = {k: torch.rand_like(v) * 1e-6 for k, v in dP.items()}
    d_cnt = torch.randint(0, 6, (N_GAUSS,), device=dev, generator=g, dtype=torch.int32)
    d_acc = torch.randn((N_GAUSS, 1), device=dev, generator=g).abs() * 1.5e-6
    th = dn.raw_thresholds(5.0)
    counts = [None]

    def densify_once():
        cls, slots, cnts = dn.plan(dP["alphas_raw"], dP["scales_raw"], d_acc, d_cnt, th)
        z = torch.empty((cnts[2], 3), device=dev).normal_()
        dn.apply(cls, slots, cnts, dP, dM, dV, z)
        counts[0] = cnts
    ms_dens = timed(densify_once, 5, 2, collective=False) / 5
    lib.gsb_profile_enable(1)
    for _ in range(3):
        densify_once()
    torch.cuda.synchronize()
    lib.gsb_profile_enable(0)
    dkern = {}
    for i in range(lib.gsb_profile_kernels()):
        ms_tot, cnt = C.c_double(0), C.c_longlong(0)
        lib.gsb_profile_read(i, C.byref(ms_tot), C.byref(cnt))
        if cnt.value:
            dkern[lib.gsb_profile_kernel_name(i).decode()] = ms_tot.value / 3
    Kk, Cc, Ss = counts[0]
    apply_bytes = 2 * 708 * Kk + 708 * (Cc + Ss) + 13 * N_GAUSS + 12 * Ss   # rows moved once + cls/slots + z
    dens_info = {"what": "update_gaussian_density on 1M Gaussians with Adam moments (gsmodel.py:132-166, 236-318): "
                         "gsb_density_plan + gsb_density_apply, incl. the count read-back and output allocation",
                 "ms": ms_dens, "kernels_ms": dkern, "survivors_clones_splits": [Kk, Cc, Ss],
                 "apply_algorithmic_bytes": apply_bytes,
                 "apply_achieved_GBps": apply_bytes / (dkern.get("density_apply", float("nan")) * 1e-3) / 1e9,
                 "apply_hbm_frac": apply_bytes / (dkern.get("density_apply", float("nan")) * 1e-3) / 1e9 / peak,
                 "vs_reference": "profiles/r1_compare_density_ref.json (same inputs through the reference's gsmodel.py)"}
    del dP, dM, dV

    # ---- the reference's own CUDA extension on the same GPU, same harness (when it was built
    # into baseline/_ref by baseline/build_ref_gpu.sh): its own process -- both modules are `gsplatcu`
    ref_gpu = reference_gpu_block(local)

    # ---- CPU baseline + gradient error vs the CPU oracle on the same frame
    cpu_mpix, cpu_sec, cpu_threads, cpu = cpu_sample(steps=1, warmup=0)
    err = gpu_vs_cpu_crop(torch, dev, cpu)
    line = {
        "metric": METRIC, "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "config2: 1M synthetic Gaussians, 1920x1080, SH deg 3, forward+backward to "
                               "parameter gradients (fused preprocess fwd/bwd + splat + splatB)",
                   "gaussians": N_GAUSS, "width": WIDTH, "height": HEIGHT, "sh_dim": SH_DIM, "patches": P,
                   "p_eff": p_eff, "views_per_step": world,
                   "parallelism": ("1 view/rank, shared Gaussians; parameter gradients summed by the factorised "
                                   "exchange (NCCL all-reduce of 11 floats + all-gather of every view's dL/dcolor, "
                                   "dL/dsh expanded locally)" if world > 1 else "single GPU"),
                   "l2": "per-step working set (params+grads 0.47 GB, records 0.12 GB, sort buffers) > 126 MB L2; "
                         "no explicit flush"},
        "gaussians_per_s": N_GAUSS * world * args.steps / (ms_dev * 1e-3),
        "op_surface": {"what": "same step through the reference's 7-op surface (calc_J=True) and its Jacobian "
                               "chain exactly as gsmodel.py:6-93 writes it (GSFunction mirror); the chain's `@` "
                               "products on our JacobianTensor outputs run on gsb_small_bmm",
                       "value": pix * ops_steps / (ms_ops * 1e-3) / 1e6, "unit": "Mpixels/s",
                       "ms_per_step": ms_ops / ops_steps},
        "grad_max_rel_err_vs_cpu": err["grad_max_rel_err"], "parity_vs_cpu": err,
        "roofline": roofline,
        "kernel_ms_per_step": kern,
        "loss_n2": loss_info,
        "density_n3": dens_info,
        "cpu_baseline": {"value": cpu_mpix, "unit": "Mpixels/s", "cores": cpu_threads, "kind": "port",
                         "sample": sample_text(cpu_sec, cpu["passes"]), "config1": config1_block()},
        "ref_gpu": ref_gpu,
        "e2e": {"value": e2e, "unit": "Mpixels/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(dl_host.numel() * 4 + cam_host.numel() * 4),
                "d2h_bytes_per_step": int(img_host.numel() * 4 + 4),
                "what": "camera + dL/dimage from pinned host memory each step; image + gradient checksum back"},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    line["config5"] = config5
    line["cuda_graphs"] = graphs
    if allreduce is not None:
        line["allreduce"] = allreduce
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_config5(torch, dist, dev, rank, world, timed):
    """BASELINE config 5 as written: 2M shared Gaussians, 8 cameras per step on a ring, split over
    the ranks (8 / world views each, gradients accumulated locally), ONE factorised exchange per
    step.  Strong scaling in the ranks: the work per step is fixed.  Every rank runs it; rank 0
    reports.  world = 1: the 8 views in sequence, no exchange."""
    from easygaussiansplatting_b200.gsfunction import Camera
    from easygaussiansplatting_b200.parallel import MultiViewStep
    from easygaussiansplatting_b200.scene import ring_camera, synthetic_scene, upstream_gradient
    N5, V5 = 2_000_000, 8
    if V5 % world != 0:
        return {"skipped": "8 cameras do not split over %d ranks" % world}
    sc = synthetic_scene(N5, WIDTH, HEIGHT, sh_dim=SH_DIM, seed=1)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    mv = MultiViewStep(T(sc["pws"]), T(sc["rots"]), T(sc["scales"]), T(sc["shs"]), T(sc["alphas"][:, None]))
    mine = [v for v in range(V5) if v % world == rank]
    cams = []
    for v in mine:
        Rcw, tcw, twc = ring_camera(v, V5)
        cams.append(Camera(WIDTH, HEIGHT, sc["fx"], sc["fy"], sc["cx"], sc["cy"], T(Rcw), T(tcw), T(twc)))
    dl = T(upstream_gradient(WIDTH, HEIGHT, rank) * (3.0 * WIDTH * HEIGHT))
    out = [None]

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

    def step():
        ev[0].record()
        for i, cam in enumerate(cams):
            image, ctx = mv.render(cam)
            mv.backward(ctx, dl, last=i == len(cams) - 1)
        ev[1].record()
        out[0] = mv.reduce()
        ev[2].record()
    n = 8  # (6 warm-up steps: the allocator and NCCL settle on the 2M-Gaussian buffer sizes over the first few)
    ms = timed(step, n, 6) / n
    torch.cuda.synchronize()
    ms_render, ms_reduce = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])  # last step, this rank
    res = {"what": "config 5: 2M shared Gaussians, 8 cameras/step at 1920x1080, %d view(s) per rank, one "
                   "factorised gradient exchange per step (strong scaling over the ranks)" % len(mine),
           "gaussians": N5, "views_per_step": V5, "n_gpus": world, "ms_per_step": ms,
           "value": V5 * WIDTH * HEIGHT / (ms * 1e-3) / 1e6, "unit": "Mpixels/s", "scaling": "strong",
           "last_step_ms": {"render_and_backward": ms_render, "reduce": ms_reduce},
           "capacity_path": dict(__import__("easygaussiansplatting_b200.ops", fromlist=["x"]).CAPACITY_STATS),
           "exchange_bytes_per_rank": out[0]["bytes_per_rank"] if world > 1 else 0}
    del mv, out
    torch.cuda.empty_cache()
    return res


def reference_gpu_block(gpu_index):
    """t_fwd / t_bwd of the UNMODIFIED reference `gsplatcu` (baseline/_ref/gsplatcu*.so) through the
    same autograd wrapper on config 2, with the same clock sampler (benchmarks/compare_ref_gpu.py
    --arm ref).  None when the extension is not installed."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not (os.path.isdir(ref_dir) and any(f.startswith("gsplatcu") and f.endswith(".so") for f in os.listdir(ref_dir))):
        return None
    sampler = ClockSampler(gpu_index)
    sampler.start()
    try:
        with tempfile.TemporaryDirectory() as tmp:  # the arm's JSON and raw tensors are scratch
            out = os.path.join(tmp, "bench_ref_gpu")
            r = subprocess.run([sys.executable, os.path.join(ROOT, "benchmarks", "compare_ref_gpu.py"), "--arm",
                                "ref", "--iters", "10", "--out", out, "--configs", "config2"],
                               capture_output=True, text=True, timeout=600)
            clocks = sampler.stop()
            if r.returncode != 0:
                return {"error": r.stderr[-300:]}
            res = json.load(open(out + ".ref.json"))["config2"]
        return {"what": "the reference's own gsplatcu (unmodified, built for sm_100a) on this GPU: GSFunction.apply "
                        "(6 ops, calc_J=True) + image.backward (splatB + torch Jacobian chain), config 2, CUDA "
                        "events, median of 10",
                "t_fwd_ms": res["t_fwd_ms"], "t_bwd_ms": res["t_bwd_ms"], "splat_ms": res["splat_ms"],
                "splatB_ms": res["splatB_ms"], "value": res["mpix_per_s"], "unit": "Mpixels/s", "clocks": clocks}
    except Exception as e:
        sampler.stop()
        return {"error": repr(e)[:300]}


def gpu_vs_cpu_crop(torch, dev, cpu):
    """GPU vs CPU oracle on the CPU arm's frame (the whole 1920x1080 view of the 1M scene).
    splat / splatB are compared on the GPU's own fp32 op inputs (what the operator actually
    received); Gaussians whose alpha' comes within 2e-5 of the 0.002 threshold at some pixel are
    reported separately (an fp32 kernel may take the other branch there).  The per-Gaussian
    backward is compared with the fp64 Jacobian chain on the same upstream gradients."""
    from oracle import oracle as orc
    from easygaussiansplatting_b200 import ops
    sc, cy, dl = cpu["scene"], cpu["cy"], cpu["dl"]
    W, H = WIDTH, CROP_ROWS
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    n = lambda x: x.detach().cpu().numpy()
    pws, rots, scales, shs = T(sc["pws"]), T(sc["rots"]), T(sc["scales"]), T(sc["shs"])
    Rcw, tcw, twc, al = T(sc["Rcw"]), T(sc["tcw"]), T(sc["twc"]), T(sc["alphas"])
    us, ci, col, depths, areas = ops.preprocess(pws, rots, scales, shs, Rcw, tcw, twc, sc["fx"], sc["fy"],
                                                sc["cx"], cy, W, H)
    d_in, a_in = n(depths).copy(), n(areas).copy()
    image, contrib, ftau, ranges, gsid = ops.splat(H, W, us, ci, al, depths, col, areas)
    grads = ops.splatB(H, W, us, ci, al, depths, col, contrib, ftau, ranges, gsid, T(dl))
    gp = ops.preprocessB(pws, rots, scales, shs, Rcw, tcw, twc, sc["fx"], sc["fy"], sc["cx"], cy, W, H,
                         grads[0], grads[1], grads[3])
    ref = orc.splat(H, W, n(us), n(ci), sc["alphas"], d_in, n(col), a_in)
    *rg, amb = orc.splat_backward(H, W, n(us), n(ci), sc["alphas"], n(col), ref, dl, return_ambiguous=True)
    okpix = ~ref["ambiguous"]
    out = {"image_max_abs_err": float(np.abs(n(image) - ref["image"]).max(axis=0)[okpix].max()),
           "ambiguous_pixels": int(ref["ambiguous"].sum()), "ambiguous_gaussians": int(amb.sum()),
           "sort_order_exact": bool(np.array_equal(n(gsid), ref["gsid"]))}
    worst, worst_amb = 0.0, 0.0
    for got, want, name in zip(grads, rg, ("dloss_dus", "dloss_dcinv2ds", "dloss_dalphas", "dloss_dcolors")):
        e = np.abs(n(got).astype(np.float64) - want).reshape(len(want), -1).max(axis=1) / np.abs(want).max()
        out[name] = float(e[~amb].max())
        worst, worst_amb = max(worst, out[name]), max(worst_amb, float(e.max()))
    # per-Gaussian backward: fp64 Jacobian chain on the GPU's own splatB gradients
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    u64, pcs, dep, Ju = orc.project(sc["pws"], sc["Rcw"], sc["tcw"], sc["fx"], sc["fy"], sc["cx"], cy)
    d32 = f32(dep)
    c3, J3r, J3s = orc.compute_cov3d(sc["rots"], sc["scales"], d32)
    c2, J2c, J2p = orc.compute_cov2d(f32(c3), f32(pcs), sc["Rcw"], d32, sc["fx"], sc["fy"], W, H)
    _, Jcs, Jcp = orc.sh2color(sc["shs"], sc["pws"], sc["twc"])
    _, _, Jci = orc.inverse_cov2d(f32(c2), d32)
    chain = orc.chain_backward(sc["Rcw"], n(grads[0]), n(grads[1]), n(grads[2]), n(grads[3]), Ju, J3r, J3s, J2c,
                               J2p, Jcs, Jcp, Jci)
    for got, name in zip(gp, ("pws", "shs", "scales", "rots")):
        out["d" + name] = float(np.abs(n(got).astype(np.float64) - chain[name]).max() / np.abs(chain[name]).max())
        worst = max(worst, out["d" + name])
    out["grad_max_rel_err"] = worst
    out["grad_max_rel_err_incl_ambiguous"] = max(worst, worst_amb)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the image and a fixed sample of the parameter gradients of the last timed "
                         "step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    # stdout carries exactly one JSON line: native libraries (NCCL's version banner) write to
    # fd 1 directly, so fd 1 is pointed at stderr and the line goes to a private copy of stdout
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
