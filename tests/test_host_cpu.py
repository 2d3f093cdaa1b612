"""CPU-only checks of the host side: the C-ABI library loads and exports exactly what
include/gsplat_b200.h declares, the operator surface refuses to run without CUDA (no silent
fallback), and the multi-view data-parallel gradient exchange works at world_size 2 (gloo)."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "gsplat_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gsb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from easygaussiansplatting_b200 import _lib, build
    build.build()
    lib = _lib.load()
    syms = header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(lib, s), "libgsplat_b200.so does not export %s" % s
    assert sorted(_lib.SIGNATURES) == syms, "ctypes signatures drifted from the header"
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(set(re.findall(r" T (gsb_[a-z0-9_]+)", out)))
    assert exported == syms
    assert lib.gsb_abi_version() == 1
    names = [lib.gsb_profile_kernel_name(i).decode() for i in range(lib.gsb_profile_kernels())]
    assert "draw" in names and "draw_backward" in names


def test_no_library_kernels_and_host_only_entry_points():
    """the binary holds no CUB / thrust kernel (round 1 sorted and scanned with them), and the
    host-only workspace queries answer without a GPU"""
    from easygaussiansplatting_b200 import _lib, build
    build.build()
    lib = _lib.load()
    r = subprocess.run(["cuobjdump", "-elf", "-symbols", _lib.LIB_PATH], capture_output=True, text=True)
    kernels = [ln for ln in r.stdout.splitlines() if "STT_FUNC" in ln]
    assert len(kernels) > 30
    assert not [ln for ln in kernels if "cub" in ln or "thrust" in ln], "a library kernel is linked in"
    for name in ("k_rects_scan", "k_radix_pass", "k_colscan", "k_density_slots", "k_density_apply_rows",
                 "k_ssim_fwd_rows", "k_ssim_bwd_rows", "k_draw3", "k_draw_bwd4"):
        assert any(name in ln for ln in kernels), name
    prev = 0
    for n in (0, 1, 1000, 1 << 20, 5 << 20):
        b = lib.gsb_density_workspace_bytes(n)
        assert b >= 256 + 12 * (n // 1024) and b >= prev
        prev = b
    assert lib.gsb_gau_loss_workspace_bytes(1080, 1920) >= 9 * 4 * 1080 * 1920
    assert lib.gsb_splat_bin_workspace_bytes(1000) < lib.gsb_splat_bin_workspace_bytes(1 << 20)
    assert lib.gsb_splat_workspace_bytes(1000, 64, 64, 10) <= lib.gsb_splat_workspace_bytes(1000, 64, 64, 100000)


def test_rasterizers_are_sm100a_with_cp_async_record_gather():
    """built for sm_100a; each rasterizer kernel gathers its records with 16-byte cp.async copies
    waited on per group (SASS LDGSTS + LDGDEPBAR) and uses packed fp32 math; the library reads no
    user-set kernel switch from the environment"""
    from easygaussiansplatting_b200 import _lib, build
    build.build()
    r = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True)
    assert "code for sm_100a" in r.stdout
    sass = {}
    for part in re.split(r"^\s+Function : ", r.stdout, flags=re.M)[1:]:
        name, body = part.split("\n", 1)
        sass[name.strip()] = body
    for kernel in ("k_draw3", "k_draw_bwd4"):
        found = [n for n in sass if re.search(r"\d%sE" % kernel, n)]
        assert len(found) == 1, (kernel, found)
        body = sass[found[0]]
        for ins in ("LDGSTS.E.BYPASS.128", "LDGDEPBAR", "FFMA2", "MUFU.EX2"):
            assert ins in body, "%s: %s missing" % (kernel, ins)
    strings = re.findall(rb"[\x20-\x7e]{4,}", open(_lib.LIB_PATH, "rb").read())
    assert sorted({s.decode() for s in strings if s.startswith(b"GSB_")}) == ["GSB_EXCHANGE_TIMEOUT_S"]


def test_ops_refuse_cpu_tensors():
    import gsplatcu
    with pytest.raises(ValueError, match="CUDA"):
        gsplatcu.project(torch.zeros(4, 3), torch.eye(3), torch.zeros(3), 1.0, 1.0, 0.0, 0.0, True)
    with pytest.raises(ValueError, match="CUDA"):
        gsplatcu.splat(16, 16, torch.zeros(1, 2), torch.zeros(1, 3), torch.zeros(1), torch.zeros(1),
                       torch.zeros(1, 3), torch.zeros(1, 2, dtype=torch.int32))


def test_product_never_imports_oracle():
    for pkg in ("easygaussiansplatting_b200", "gsplatcu"):
        for root, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    txt = open(os.path.join(root, f)).read()
                    assert "oracle" not in txt.replace("the oracle", "").replace("CPU oracle", "") or \
                        not re.search(r"^\s*(from|import)\s+oracle", txt, flags=re.M), f


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from easygaussiansplatting_b200.parallel import allreduce_grads, view_index
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
g = torch.Generator().manual_seed(100 + rank)
grads = [torch.randn(50, 3, generator=g), torch.randn(50, 48, generator=g), None, torch.randn(50, 1, generator=g)]
want = []
for r in range(world):
    gg = torch.Generator().manual_seed(100 + r)
    want.append([torch.randn(50, 3, generator=gg), torch.randn(50, 48, generator=gg), torch.randn(50, 1, generator=gg)])
nbytes = allreduce_grads(grads)
assert nbytes == 50 * 52 * 4
for i, t in enumerate([grads[0], grads[1], grads[3]]):
    s = sum(w[i] for w in want)
    assert torch.allclose(t, s, atol=1e-6), (rank, i)
assert [view_index(3, r, world) for r in range(world)] == [3 * world + r for r in range(world)]
# gradients that are views tiling one flat bucket (what ops.preprocessB returns) are reduced in place
bucket = torch.arange(50 * 10, dtype=torch.float32) * (rank + 1)
views = [bucket[:200].view(50, 4), bucket[200:350].view(50, 3), bucket[350:].view(50, 3)]
extra = torch.full((50, 1), float(rank + 1))
nb = allreduce_grads(views + [extra])
assert nb == 4 * (500 + 50)
tot = sum(range(1, world + 1))
assert torch.equal(bucket, torch.arange(500, dtype=torch.float32) * tot) and torch.all(extra == tot)
assert views[1].data_ptr() == bucket.data_ptr() + 800
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
"""


def test_multiview_grad_allreduce_gloo_world2(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_WORKER % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29531", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and ("ok %d" % r) in o, o


_WORKER_FACT = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r)
from easygaussiansplatting_b200.parallel import factorised_sum
from oracle import oracle as orc
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
N, K3, VL = 300, 16, 2                       # 2 local views per rank -> 4 views in total
rng = np.random.default_rng(7)               # same on every rank: positions, every view's data
pws = rng.normal(size=(N, 3)).astype(np.float32) * 3
twc_all = rng.normal(size=(world * VL, 3)).astype(np.float32) * 8
col_all = rng.normal(size=(world * VL, N, 3)).astype(np.float32)
small_all = rng.normal(size=(world, 11 * N)).astype(np.float32)
def basis(twc):                              # Y_l(dir) of every Gaussian for one camera centre: the oracle's dcolor/dsh
    return orc.sh2color(np.zeros((N, 3 * K3), np.float32), pws, twc)[1].reshape(N, K3)
def expand(tw, col):                         # CPU stand-in of ops.sh_grad_expand (same contract)
    out = np.zeros((N, K3, 3))
    for v in range(tw.shape[0]):
        out += basis(tw[v].numpy())[:, :, None] * col[v].numpy().astype(np.float64)[:, None, :]
    return torch.from_numpy(out.reshape(N, 3 * K3))
lo = rank * VL
small, dshs = factorised_sum(torch.from_numpy(small_all[rank].copy()), torch.from_numpy(col_all[lo:lo + VL].copy()),
                             torch.from_numpy(twc_all[lo:lo + VL].copy()), None, expand)
assert np.allclose(small.numpy(), small_all.sum(0), atol=1e-5)
want = expand(torch.from_numpy(twc_all), torch.from_numpy(col_all))    # every view, in rank order
assert torch.allclose(dshs, want, atol=1e-9), float((dshs - want).abs().max())
dist.barrier(); dist.destroy_process_group()
print("ok", rank)
"""


def test_factorised_multiview_sum_gloo_world2(tmp_path):
    """parallel.factorised_sum on 2 CPU ranks x 2 local views: the 11-float bucket is all-reduced,
    the per-view dL/dcolor and camera centres are gathered in rank order and the expansion
    sum_v Y(dir_v) (x) dL/dcolor_v sees all 4 views on every rank."""
    script = tmp_path / "wf.py"
    script.write_text(_WORKER_FACT % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and ("ok %d" % r) in o, o
