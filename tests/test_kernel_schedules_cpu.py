"""Lane-level models of two kernel schedules, checked against the CPU oracles (no GPU needed).

These are transliterations of the index logic of `k_ssim_fwd_rows` / `k_ssim_bwd_rows`
(csrc/loss.cu: 48-column line buffers filled by 16-byte or scalar loads, 12-slot register ring,
two rows in flight, strips with a 5-row halo) and of `rows_job` in csrc/density.cu (32-row groups,
the plan table, fixed lane -> (row, column) maps for the [*, 45] arrays, three rounds per row pair):
every lane of every warp is walked in Python, uninitialised storage is NaN and asserted never to be
read, every output element is asserted to be written exactly once, and the result must equal the
oracle's.  They were written before the kernels first ran on a GPU and caught the schedule errors a
parity test would only have reported as "wrong numbers"; they guard the same logic against edits.
They say nothing about synchronisation or memory spaces -- that is what the GPU tests are for."""
import numpy as np
import pytest

from oracle import density_oracle as do
from oracle import oracle as orc

f32 = np.float32

# ------------------------------------------------------------------ csrc/loss.cu, row streaming
LR, SWARPS, SLINE, SPAD = 5, 4, 48, 8

def win11():
    w = np.array([np.exp(-((x - 5) ** 2) / (2.0 * 1.5 * 1.5)) for x in range(11)], dtype=np.float32)
    s = f32(0)
    for x in range(11): s = f32(s + w[x])
    return (w / s).astype(np.float32)

RING=12
def ring_slot(i, k): return (i + 2 + k) % RING

class RowFetch:
    def __init__(self, NIMG, VEC, lane, x0, W, imgs, line):
        # imgs: list of flat arrays (plane row 0 base), line: np array [NIMG][2][SLINE]
        self.NIMG, self.VEC, self.W = NIMG, VEC, W
        self.imgs, self.line = imgs, line
        self.ent = []
        if VEC:
            ROUNDS = (12 * NIMG + 31) // 32
            for r in range(ROUNDS):
                per = []
                for l in lane:
                    q = l + 32 * r; im = q // 12; ch = q - 12 * im; col = x0 - SPAD + 4 * ch
                    ok = q < 12 * NIMG and col >= 0 and col < W
                    imc = im if im < NIMG else 0
                    per.append((ok, imc, col, 4 * ch, q < 12 * NIMG))
                self.ent.append(per)
        else:
            for m in range(NIMG):
                for h in range(2):
                    per = []
                    for l in lane:
                        j = l + 32 * h; col = x0 - SPAD + j
                        ok = j < SLINE and col >= 0 and col < W
                        per.append((ok, m, col, j if j < SLINE else 0, (h == 0) or (l + 32 < SLINE)))
                    self.ent.append(per)
        self.v = None
    def fetch(self, yy, W, H):
        yin = 0 <= yy < H
        o = yy * W
        vals = []
        for per in self.ent:
            pv = []
            for (ok, m, col, d, st) in per:
                if self.VEC:
                    v = np.zeros(4, np.float32)
                    if yin and ok:
                        assert (o + col) % 4 == 0
                        v = self.imgs[m][o + col:o + col + 4].copy(); assert len(v) == 4
                else:
                    v = np.zeros(1, np.float32)
                    if yin and ok: v = self.imgs[m][o + col:o + col + 1].copy()
                pv.append(v)
            vals.append(pv)
        self.v = vals
    def stage(self, buf):
        for per, pv in zip(self.ent, self.v):
            for (ok, m, col, d, st), v in zip(per, pv):
                if st:
                    self.line[m][buf][d:d + len(v)] = v

def strip_rows(H, W, sms=148):
    xblocks = (W + 32 * SWARPS - 1) // (32 * SWARPS)
    strips = max(1, (sms * 4) // (3 * xblocks))
    sh = (H + strips - 1) // strips
    return max(sh, 16)

def run_loss_rows(img, gt, lam=0.2, SH=None, VEC=None):
    _, H, W = img.shape
    HW = H * W
    win = win11()
    if SH is None: SH = strip_rows(H, W)
    if VEC is None: VEC = W % 4 == 0
    maps = np.full(9 * HW, np.nan, np.float32)
    acc = np.zeros(2, np.float64)
    imgf, gtf = img.reshape(-1), gt.reshape(-1)
    gx, gy = (W + 127) // 128, (H + SH - 1) // SH
    lane = np.arange(32)
    C1, C2 = f32(0.01 * 0.01), f32(0.03 * 0.03)
    for c in range(3):
      for by in range(gy):
        for bx in range(gx):
          red = np.zeros((2, SWARPS), np.float32)
          for wid in range(SWARPS):
            x0 = (bx * SWARPS + wid) * 32; x = x0 + lane
            yb = by * SH; ye = min(yb + SH, H)
            xin = x < W
            n = ye - yb + 2 * LR
            l1 = np.zeros(32, np.float32); ss = np.zeros(32, np.float32)
            if x0 < W:
                line = np.full((2, 2, SLINE), np.nan, np.float32)
                rf = RowFetch(2, VEC, lane, x0, W, [imgf[c * HW:(c + 1) * HW], gtf[c * HW:(c + 1) * HW]], line)
                r01 = np.full((RING, 2, 32), np.nan, np.float32); r23 = r01.copy(); r4 = np.full((RING, 32), np.nan, np.float32)
                rf.fetch(yb - LR, W, H); rf.stage(0); rows = [None, None]; rf.fetch(yb - LR + 1, W, H); rows[1] = rf.v; rf.fetch(yb - LR + 2, W, H); rows[0] = rf.v
                for t0 in range(0, n, RING):
                    for i in range(RING):
                        t = t0 + i
                        if t < n:
                            yy = yb - LR + t
                            rf.v = rows[(i + 1) & 1]; rf.stage((i + 1) & 1); rf.fetch(yy + 3, W, H); rows[(i + 1) & 1] = rf.v
                            base = lane + SPAD - LR
                            mm = np.zeros((2, 32), np.float32); ee = np.zeros((2, 32), np.float32); e12 = np.zeros(32, np.float32)
                            for k in range(11):
                                a = line[0][i & 1][base + k]; b = line[1][i & 1][base + k]
                                assert not np.isnan(a).any() and not np.isnan(b).any()
                                if k == LR and t >= LR and t < n - LR: l1 = l1 + np.abs(a - b)
                                mm[0] += win[k] * a; mm[1] += win[k] * b
                                ee[0] += win[k] * a * a; ee[1] += win[k] * b * b
                                e12 += win[k] * a * b
                            r01[i] = mm; r23[i] = ee; r4[i] = e12
                            if t >= 2 * LR:
                                v01 = np.zeros((2, 32), np.float32); v23 = np.zeros((2, 32), np.float32); v4 = np.zeros(32, np.float32)
                                for k in range(11):
                                    sl = ring_slot(i, k)
                                    assert not np.isnan(r4[sl]).any()
                                    v01 += win[k] * r01[sl]; v23 += win[k] * r23[sl]; v4 += win[k] * r4[sl]
                                mu1, mu2 = v01
                                s11 = v23[0] - mu1 * mu1; s22 = v23[1] - mu2 * mu2; s12 = v4 - mu1 * mu2
                                A1 = 2 * mu1 * mu2 + C1; A2 = 2 * s12 + C2
                                B1 = mu1 * mu1 + mu2 * mu2 + C1; B2 = s11 + s22 + C2
                                inv = 1 / (B1 * B2); ssim = A1 * A2 * inv
                                ss = ss + np.where(xin, ssim, 0)
                                o = (yy - LR) * W + x
                                m0 = (2 * mu2 * (A2 - A1)) * inv - ssim * (2 * mu1 * (B2 - B1)) * inv
                                for l in range(32):
                                    if xin[l]:
                                        assert 0 <= yy - LR < H
                                        assert np.isnan(maps[c * HW + o[l]])
                                        maps[c * HW + o[l]] = m0[l]
                                        maps[(3 + c) * HW + o[l]] = (-ssim / B2)[l]
                                        maps[(6 + c) * HW + o[l]] = (2 * A1 * inv)[l]
            red[0][wid] = l1.sum(); red[1][wid] = ss.sum()
          acc[0] += red[0].astype(np.float64).sum(); acc[1] += red[1].astype(np.float64).sum()
    assert not np.isnan(maps).any()
    npix = 3.0 * HW
    loss = (1 - lam) * acc[0] / npix + lam * (1 - acc[1] / npix)
    grad = np.full(3 * HW, np.nan, np.float32)
    inv_n = f32(1.0 / npix)
    for c in range(3):
      for by in range(gy):
        for bx in range(gx):
          for wid in range(SWARPS):
            x0 = (bx * SWARPS + wid) * 32; x = x0 + lane
            if x0 >= W: continue
            yb = by * SH; ye = min(yb + SH, H)
            xin = x < W; n = ye - yb + 2 * LR
            line = np.full((3, 2, SLINE), np.nan, np.float32)
            rf = RowFetch(3, VEC, lane, x0, W, [maps[c * HW:(c + 1) * HW], maps[(3 + c) * HW:(4 + c) * HW], maps[(6 + c) * HW:(7 + c) * HW]], line)
            r01 = np.full((RING, 2, 32), np.nan, np.float32); r2 = np.full((RING, 32), np.nan, np.float32)
            rf.fetch(yb - LR, W, H); rf.stage(0); rows = [None, None]; rf.fetch(yb - LR + 1, W, H); rows[1] = rf.v; rf.fetch(yb - LR + 2, W, H); rows[0] = rf.v
            pq = [np.zeros(32, np.float32), np.zeros(32, np.float32)]; gq = [np.zeros(32, np.float32), np.zeros(32, np.float32)]
            for t0 in range(0, n, RING):
                for i in range(RING):
                    t = t0 + i
                    if t < n:
                        yy = yb - LR + t
                        rf.v = rows[(i + 1) & 1]; rf.stage((i + 1) & 1); rf.fetch(yy + 3, W, H); rows[(i + 1) & 1] = rf.v
                        p_cur, g_cur = pq[i & 1].copy(), gq[i & 1].copy()
                        if t + 2 >= 2 * LR and t + 2 < n:
                            for l in range(32):
                                if xin[l]:
                                    o1 = (yy - LR) * W + x[l] + 2 * W
                                    assert 0 <= o1 < HW
                                    pq[i & 1][l] = imgf[c * HW + o1]; gq[i & 1][l] = gtf[c * HW + o1]
                        base = lane + SPAD - LR
                        h01 = np.zeros((2, 32), np.float32); h2 = np.zeros(32, np.float32)
                        for k in range(11):
                            q0 = line[0][i & 1][base + k]; q1 = line[1][i & 1][base + k]; q2 = line[2][i & 1][base + k]
                            assert not (np.isnan(q0).any() or np.isnan(q1).any() or np.isnan(q2).any())
                            h01[0] += win[k] * q0; h01[1] += win[k] * q1; h2 += win[k] * q2
                        r01[i] = h01; r2[i] = h2
                        if t >= 2 * LR:
                            v01 = np.zeros((2, 32), np.float32); v2 = np.zeros(32, np.float32)
                            for k in range(11):
                                sl = ring_slot(i, k)
                                v01 += win[k] * r01[sl]; v2 += win[k] * r2[sl]
                            for l in range(32):
                                if xin[l]:
                                    o = (yy - LR) * W + x[l]
                                    p = p_cur[l]; g = g_cur[l]
                                    assert p == imgf[c * HW + o] and g == gtf[c * HW + o]
                                    sgn = 1.0 if p > g else (-1.0 if p < g else 0.0)
                                    assert np.isnan(grad[c * HW + o])
                                    grad[c * HW + o] = (1 - lam) * sgn * inv_n - lam * inv_n * (v01[0][l] + 2 * p * v01[1][l] + g * v2[l])
    assert not np.isnan(grad).any()
    return loss, grad.reshape(3, H, W)



@pytest.mark.parametrize("H,W,SH", [(37, 53, None), (16, 16, None), (40, 36, 16), (23, 132, 7), (33, 128, 11)])
def test_loss_row_streaming_schedule(H, W, SH):
    rng = np.random.default_rng(H * 1000 + W)
    yy, xx = np.mgrid[0:H, 0:W]
    base = np.stack([0.5 + 0.4 * np.sin(xx / 9.0 + c) * np.cos(yy / 6.0 - c) for c in range(3)])
    img = np.clip(base + rng.normal(scale=0.08, size=base.shape), -0.2, 1.3).astype(np.float32)
    gt = np.clip(base + rng.normal(scale=0.02, size=base.shape), 0, 1).astype(np.float32)
    ref = orc.gau_loss(img, gt)
    for vec in ([True, False] if W % 4 == 0 else [False]):
        loss, grad = run_loss_rows(img, gt, SH=SH, VEC=vec)
        e = np.abs(grad - ref["dloss_dimage"]).max() / np.abs(ref["dloss_dimage"]).max()
        assert abs(loss - ref["loss"]) < 2e-6 and e < 3e-4, (vec, loss, e)


# ------------------------------------------------------------------ csrc/density.cu, row groups
KEEP, CLONE, SPLIT, PRUNE = 0, 1, 2, 3
NAMES = ("pws", "low_shs", "high_shs", "alphas_raw", "scales_raw", "rots_raw")
WID = (3, 3, 45, 1, 3, 4)

def random_state(N, seed, sense=5.0):
    rng = np.random.default_rng(seed)
    P = dict(pws=rng.uniform(-2, 2, (N, 3)), low_shs=rng.normal(size=(N, 3)), high_shs=rng.normal(size=(N, 45)) * 0.1,
             alphas_raw=rng.uniform(-7.5, 4, (N, 1)),
             scales_raw=np.log(np.exp(rng.uniform(np.log(0.002 * sense), np.log(0.12 * sense), (N, 1))) * rng.uniform(0.6, 1.5, (N, 3))),
             rots_raw=rng.normal(size=(N, 4)) * rng.uniform(0.3, 2, (N, 1)))
    P = {k: v.astype(np.float32) for k, v in P.items()}
    M = {k: (rng.normal(size=v.shape) * 1e-3).astype(np.float32) for k, v in P.items()}
    acc = (np.abs(rng.normal(size=(N, 1))) * 1.5e-6).astype(np.float32)
    cnt = rng.integers(0, 6, N).astype(np.int32); acc[cnt == 0] = 0
    return P, M, acc, cnt

def rows_job(w, src, dst, row0, tab, K, C, newval):
    gsrc = src[row0 * w:]
    def emit(r, col, info, val):
        cl = (info[0] & 0xffffffff) >> 30
        if cl == PRUNE: return
        d = (info[0] & 0x3fffffff) * w + col
        assert np.isnan(dst[d]); dst[d] = val
        if cl == KEEP: return
        d = info[1] * w + col
        assert np.isnan(dst[d]); dst[d] = newval(val, cl == SPLIT, row0 + r, info[1] - K - C, col)
    pruned = (PRUNE << 30, 0)
    # (table entries of rows past the end of the array are PRUNE: no row bound is checked)
    if w == 45:  # DG_PAIRS = 4 row pairs, i.e. 12 loads, in flight per lane
        for p0 in range(0, 16, 4):
            for lane in range(32):
                rsel = [0, 1 if lane >= 13 else 0, 1]
                col = [lane, 32 + lane if lane < 13 else lane - 13, 19 + lane]
                st = []
                for q in range(4):
                    for rd in range(3):
                        r = 2 * (p0 + q) + rsel[rd]
                        info = pruned if (rd == 2 and lane >= 26) else tab[r]
                        v = gsrc[r * w + col[rd]] if ((info[0] & 0xffffffff) >> 30) != PRUNE else None
                        st.append((r, col[rd], info, v))
                for (r, c_, info, v) in st: emit(r, c_, info, v)
    else:  # w = 1, 3, 4: the group is w rounds of 32 lanes
        for lane in range(32):
            st = []
            for u in range(w):
                e = 32 * u + lane; r = e // w
                info = tab[r]
                v = gsrc[e] if ((info[0] & 0xffffffff) >> 30) != PRUNE else None
                st.append((r, e - r * w, info, v))
            for (r, c_, info, v) in st: emit(r, c_, info, v)



@pytest.mark.parametrize("N,seed", [(1, 1), (257, 2), (300, 9), (2000, 4)])
def test_density_row_group_schedule(N, seed):
    P, M, acc, cnt = random_state(N, seed)
    cls = do.classify(P["alphas_raw"], P["scales_raw"], acc, cnt, do.thresholds(5.0))
    flags = np.stack([cls != PRUNE, cls == CLONE, cls == SPLIT], axis=1).astype(np.int64)
    slots = np.cumsum(flags, axis=0) - flags
    K, C, S = (int(x) for x in flags.sum(axis=0))
    z = np.zeros((S, 3), np.float32)
    oP, oM, oV, _ = do.densify(P, M, M, cls, z)
    for name, w in zip(NAMES, WID):
        for setname, srcd, ref, nv in (("p", P, oP, lambda val, sp, i, s, c: val), ("m", M, oM, lambda *a: 0.0)):
            src = srcd[name].reshape(-1)
            dst = np.full((K + C + S) * w, np.nan, np.float32)
            for g in range((N + 31) // 32):
                row0 = g * 32
                tab = []
                for lane in range(32):
                    row = row0 + lane
                    c, sl = PRUNE, (0, 0, 0)
                    if row < N: c, sl = int(cls[row]), tuple(int(x) for x in slots[row])
                    tab.append(((c << 30) | sl[0], K + C + sl[2] if c == SPLIT else K + sl[1]))
                rows_job(w, src, dst, row0, tab, K, C, nv)
            assert not np.isnan(dst).any(), (name, setname)
            got = dst.reshape(-1, w)
            if setname == "m":
                assert np.array_equal(got, ref[name]), (name, "m")
            else:
                assert np.array_equal(got[:K], ref[name][:K]), name
                if name in ("low_shs", "high_shs"): assert np.array_equal(got, ref[name]), name
                else: # untransformed copies of the sources land in the right rows
                    assert np.array_equal(got[K:K + C], P[name][cls == CLONE]) and np.array_equal(got[K + C:], P[name][cls == SPLIT]), name
