"""Multi-view data parallelism (SURVEY 8e; not present in the reference, which is single
process / single GPU).  One process per GPU, Gaussians replicated, one camera per rank per
step; the only exchange is the SUM of the parameter gradients (236 B/Gaussian) over ranks.

Two implementations of that exchange (prefer_fused_exchange(world) says which one wins where;
bench.py times both at every world size):
  GradExchange      the fused per-Gaussian backward pushes each gradient tile into the owning
                    GPU's peer memory while it computes (gsb_preprocess_backward_push) and one
                    kernel sums and broadcasts (gsb_grad_reduce_broadcast) -- csrc/comm.cu.
                    torch.distributed only carries the 64-byte IPC handles at start-up.
  allreduce_grads   NCCL (or gloo in the CPU tests) all-reduce of the flat gradient bucket after
                    the backward."""
import ctypes as C

import torch
import torch.distributed as dist


def view_index(step, rank, world):
    """camera index rendered by `rank` at `step` (8 cameras/step at world=8, config 5)"""
    return step * world + rank


def _coalesce(tensors):
    """Group tensors that are contiguous views tiling one storage range (the fused backward
    writes dL/dpws, dL/dshs, dL/dscales, dL/drots into one flat bucket) so the group can be
    reduced in place with a single collective and no staging copy."""
    groups, rest = {}, []
    for t in tensors:
        if t.is_contiguous() and t.numel() > 0:
            groups.setdefault((t.untyped_storage().data_ptr(), t.dtype), []).append(t)
        else:
            rest.append(t)
    flats = []
    for (_, dtype), ts in groups.items():
        ts.sort(key=lambda t: t.storage_offset())
        lo, hi = ts[0].storage_offset(), ts[0].storage_offset()
        ok = True
        for t in ts:
            if t.storage_offset() != hi:
                ok = False
                break
            hi += t.numel()
        if ok and len(ts) > 1:
            flats.append(torch.as_strided(ts[0], (hi - lo,), (1,), lo))
        else:
            rest.extend(ts)
    return flats, rest


def allreduce_grads(tensors, group=None, average=False):
    """In-place SUM (or mean) all-reduce of a list of gradient tensors.  Tensors that already
    share a flat bucket are reduced in place; the others go through one concatenated bucket.
    Returns the number of bytes reduced."""
    tensors = [t for t in tensors if t is not None]
    if not tensors:
        return 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    flats, rest = _coalesce(tensors)
    nbytes = 0
    for f in flats:
        if world > 1:
            dist.all_reduce(f, op=dist.ReduceOp.SUM, group=group)
            if average:
                f /= world
        nbytes += f.numel() * f.element_size()
    if rest:
        flat = torch.cat([t.reshape(-1) for t in rest])
        if world > 1:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
            if average:
                flat /= world
        off = 0
        for t in rest:
            n = t.numel()
            t.copy_(flat[off:off + n].view_as(t))
            off += n
        nbytes += flat.numel() * flat.element_size()
    return nbytes


# ----------------------------------------------------------------------------- fused exchange

def rows_per_rank(N, world, tile=128):
    """rows each rank owns in the exchange (csrc/comm.cu exchange_geom): ceil(ceil(N / 128) /
    world) tiles of 128 Gaussians, dealt round-robin (rank r owns tiles r, r + world, ...)"""
    tiles = (N + tile - 1) // tile
    return max(1, (tiles + world - 1) // world) * tile


class _DeviceSpan:
    """exposes raw device memory to torch.as_tensor through __cuda_array_interface__"""

    def __init__(self, ptr, n_floats):
        self.__cuda_array_interface__ = {"shape": (n_floats,), "typestr": "<f4", "data": (ptr, False), "version": 2}


class GradExchange:
    """Sum of the fused backward's parameter gradients over `world` ranks through peer memory.

        ex = GradExchange.from_process_group(N, sh_dim3, device)      # once; collective
        ...
        grads = ex.backward(pws, rots, scales, shs, cam, moments=moments, cinv2ds=cinv2ds)
                                                  # dict dpws dshs dscales drots dalphas, already summed

    The returned tensors are views of this rank's result region and are overwritten by the next
    call.  `regions` (low-level constructor): device pointers of every rank's region as seen
    from this process, own region included -- several "ranks" may also live in one process on
    one GPU (tests), each on its own stream."""

    def __init__(self, N, sh_dim3, world, rank, regions, device, own_region=None, peers=()):
        from . import _lib
        self.lib = _lib.load()
        self.N, self.k3, self.world, self.rank, self.device = int(N), int(sh_dim3), int(world), int(rank), device
        self.regions = (C.c_void_p * world)(*[C.c_void_p(int(r)) for r in regions])
        self._own, self._peers = own_region, list(peers)
        self.epoch = 0
        self.rows_total = rows_per_rank(self.N, self.world) * self.world
        base = int(regions[rank])
        ks = 3 * self.k3
        self._views = {}
        for seg, (name, k) in enumerate((("dshs", ks), ("drots", 4), ("dpws", 3), ("dscales", 3), ("dalphas", 1))):
            off = self.lib.gsb_exchange_result_offset(self.N, self.k3, self.world, seg)
            t = torch.as_tensor(_DeviceSpan(base + off, self.rows_total * k), device=device)
            self._views[name] = t.view(self.rows_total, k)[: self.N]

    @staticmethod
    def region_bytes(N, sh_dim3, world):
        from . import _lib
        return _lib.load().gsb_exchange_region_bytes(int(N), int(sh_dim3), int(world))

    @staticmethod
    def alloc_region(nbytes):
        """-> (device pointer, 64-byte IPC handle)"""
        from . import _lib
        lib = _lib.load()
        ptr, handle = C.c_void_p(0), (C.c_ubyte * 64)()
        _lib.check(lib.gsb_comm_alloc(nbytes, C.byref(ptr), handle), lib)
        return ptr.value, bytes(handle)

    @classmethod
    def from_process_group(cls, N, sh_dim3, device, group=None):
        """collective over the process group: every rank allocates its region and opens the
        others' through CUDA IPC"""
        from . import _lib
        lib = _lib.load()
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        with torch.cuda.device(device):
            own, handle = cls.alloc_region(cls.region_bytes(N, sh_dim3, world))
            handles = [None] * world
            dist.all_gather_object(handles, handle, group=group)
            regions, peers = [], []
            for r in range(world):
                if r == rank:
                    regions.append(own)
                    continue
                p = C.c_void_p(0)
                buf = (C.c_ubyte * 64).from_buffer_copy(handles[r])
                _lib.check(lib.gsb_comm_open(buf, C.byref(p)), lib)
                regions.append(p.value)
                peers.append(p.value)
            dist.barrier(group=group)
        return cls(N, sh_dim3, world, rank, regions, device, own_region=own, peers=peers)

    def push(self, pws, rots, scales, shs, cam, dloss_dus=None, dloss_dcinv2ds=None, dloss_dcolors=None,
             dloss_dalphas=None, moments=None, cinv2ds=None):
        """phase 1: the fused per-Gaussian backward, storing into the owners' staging slots.
        Upstream gradients: the four dloss_d* tensors of `splatB`, or moments[N,9] (from
        `splatB(..., moments_only=True)`) + the forward's cinv2ds -- then this view's own
        dloss_dus[N,2] is returned (it is not part of the exchange)."""
        from . import _lib
        from .ops import _chk, _ptr, _stream
        pws = _chk(pws, "pws", last=3, ndim=2); rots = _chk(rots, "rots", last=4, ndim=2)
        scales = _chk(scales, "scales", last=3, ndim=2); shs = _chk(shs, "shs", ndim=2)
        N = pws.shape[0]
        if N != self.N or shs.shape[1] != 3 * self.k3:
            raise ValueError("GradExchange was built for N=%d, sh_dim3=%d" % (self.N, self.k3))
        gu = gc = gcol = ga = dus = None
        if moments is not None:
            moments = _chk(moments, "moments", last=9, ndim=2); cinv2ds = _chk(cinv2ds, "cinv2ds", last=3, ndim=2)
            if moments.shape[0] != N or cinv2ds.shape[0] != N:
                raise ValueError("moments / cinv2ds must have N rows")
            dus = torch.empty((N, 2), dtype=torch.float32, device=pws.device)
        else:
            gu = _chk(dloss_dus, "dloss_dus", last=2); gc = _chk(dloss_dcinv2ds, "dloss_dcinv2ds", last=3)
            gcol = _chk(dloss_dcolors, "dloss_dcolors", last=3); ga = _chk(dloss_dalphas, "dloss_dalphas")
            if ga.numel() != N or gu.numel() != 2 * N:
                raise ValueError("upstream gradients disagree on N")
        self.epoch += 1
        with torch.cuda.device(pws.device):
            _lib.check(self.lib.gsb_preprocess_backward_push(
                N, self.k3, _ptr(pws), _ptr(rots), _ptr(scales), _ptr(shs), _ptr(_chk(cam.Rcw, "Rcw")),
                _ptr(_chk(cam.tcw, "tcw")), _ptr(_chk(cam.twc, "twc")), float(cam.fx), float(cam.fy), float(cam.cx),
                float(cam.cy), float(cam.width), float(cam.height), _ptr(gu), _ptr(gc), _ptr(gcol), _ptr(ga),
                _ptr(moments), _ptr(cinv2ds), _ptr(dus), self.world, self.rank, self.regions, self.epoch, _stream()),
                self.lib)
        return dus

    def reduce(self):
        """phase 2: sum the slots of the owned rows, broadcast, wait for the peers' slices"""
        from . import _lib
        from .ops import _stream
        with torch.cuda.device(self.device):
            _lib.check(self.lib.gsb_grad_reduce_broadcast(self.N, self.k3, self.world, self.rank, self.regions,
                                                          self.epoch, _stream()), self.lib)
        return self._views

    def backward(self, pws, rots, scales, shs, cam, dloss_dus=None, dloss_dcinv2ds=None, dloss_dcolors=None,
                 dloss_dalphas=None, moments=None, cinv2ds=None):
        """push + reduce; -> dict dpws dshs dscales drots dalphas (summed over ranks) and, with
        moments, `dus` (this view's own dL/du)"""
        dus = self.push(pws, rots, scales, shs, cam, dloss_dus, dloss_dcinv2ds, dloss_dcolors, dloss_dalphas,
                        moments=moments, cinv2ds=cinv2ds)
        out = dict(self.reduce())
        if dus is not None:
            out["dus"] = dus
        return out

    def status(self):
        """0 = fine; 1 = a flag wait timed out (a peer never arrived) -- results invalid"""
        from . import _lib
        s = C.c_int(0)
        _lib.check(self.lib.gsb_exchange_status(C.c_void_p(int(self.regions[self.rank])), C.byref(s)), self.lib)
        return s.value

    def close(self):
        for p in self._peers:
            self.lib.gsb_comm_close(C.c_void_p(p))
        self._peers = []
        if self._own is not None:
            self.lib.gsb_comm_free(C.c_void_p(self._own))
            self._own = None


class MultiViewStep:
    """One data-parallel training step over the views of all ranks with the FACTORISED gradient sum.

    Of the 236 B/Gaussian a view's parameter gradient occupies (SH degree 3), 192 B are dL/dsh =
    Y(dir_v) (x) dL/dcolor_v: an outer product of a basis every rank can evaluate itself and 3
    floats.  So the ranks exchange, per view, the 12-byte dL/dcolor (all-gather) and sum the
    other 11 floats (all-reduce, 44 B), and every rank re-expands dL/dsh = sum_v Y(dir_v) (x)
    dL/dcolor_v locally (gsb_sh_grad_expand): 44 + 12 V bytes per Gaussian instead of 236.

        mv = MultiViewStep(pws, rots, scales, shs, alphas, group=None)
        for cam, dl_fn in this rank's views of the step:          # 1 .. 8 / world views
            image, ctx = mv.render(cam)
            mv.backward(ctx, dloss_dimage)                        # accumulates locally
        g = mv.reduce()   # ONE exchange: dict dpws dshs dalphas dscales drots, summed over every view
                          # of every rank; g["dus"][i] is view i's own dL/du (densification statistic)

    The collectives go through torch.distributed (NCCL on GPUs); the all-gather of the colours
    is started before the expansion of the local result needs it and the all-reduce of the small
    bucket overlaps that expansion.  world == 1 (or no process group) degenerates to local sums."""

    def __init__(self, pws, rots, scales, shs, alphas, group=None):
        self.pws, self.rots, self.scales, self.shs, self.alphas = pws, rots, scales, shs, alphas
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.k3 = shs.shape[1] // 3
        self._small, self._colors, self._twcs, self._dus = None, [], [], []
        self._early = None

    def render(self, cam):
        from . import ops
        us, cinv2ds, colors, depths, areas, records = ops.preprocess(
            self.pws, self.rots, self.scales, self.shs, cam.Rcw, cam.tcw, cam.twc, cam.fx, cam.fy, cam.cx, cam.cy,
            cam.width, cam.height, alphas=self.alphas)
        image, contrib, final_tau, ranges, gsid = ops.splat(cam.height, cam.width, us, cinv2ds, self.alphas, depths,
                                                            colors, areas, records=records, capacity=True)
        return image, (cam, us, cinv2ds, depths, colors, contrib, final_tau, ranges, gsid)

    def backward(self, ctx, dloss_dimage, last=False):
        """last=True (the rank's final view of the step): the all-gather of the views' dL/dcolor
        starts here, right after the rasterizer backward, and runs under the per-Gaussian backward."""
        from . import ops
        cam, us, cinv2ds, depths, colors, contrib, final_tau, ranges, gsid = ctx
        moments = ops.splatB(cam.height, cam.width, us, cinv2ds, self.alphas, depths, colors, contrib, final_tau,
                             ranges, gsid, dloss_dimage, moments_only=True)
        self._colors.append(moments[:, 6:9])          # dL/dcolor of this view
        self._twcs.append(cam.twc.reshape(1, 3))
        if last and self.world > 1:
            self._early = _start_gathers(torch.stack(self._colors), torch.cat(self._twcs).contiguous(), self.group)
        gpw, _, gs, gq, dus, dal = ops.preprocessB(
            self.pws, self.rots, self.scales, self.shs, cam.Rcw, cam.tcw, cam.twc, cam.fx, cam.fy, cam.cx, cam.cy,
            cam.width, cam.height, None, None, None, moments=moments, cinv2ds=cinv2ds, compact=True)
        bucket = torch.as_strided(gpw, (gpw.shape[0] * 11,), (1,), gpw.storage_offset())  # [dpws|dscales|drots|dalphas]
        self._small = bucket if self._small is None else self._small.add_(bucket)
        self._dus.append(dus)

    def reduce(self):
        from . import ops
        N = self.pws.shape[0]
        expand = lambda tw, col: ops.sh_grad_expand(self.pws, tw, col, self.k3)
        if self._early is not None:
            colors = self._early[0]
            small, dshs = factorised_sum(self._small, None, None, self.group, expand, started=self._early)
        else:
            colors = torch.stack(self._colors)                   # [V_local, N, 3] (contiguous copy)
            twcs = torch.cat(self._twcs).contiguous()            # [V_local, 3]
            small, dshs = factorised_sum(self._small, colors, twcs, self.group, expand)
        out = {"dpws": small[:3 * N].view(N, 3), "dscales": small[3 * N:6 * N].view(N, 3),
               "drots": small[6 * N:10 * N].view(N, 4), "dalphas": small[10 * N:], "dshs": dshs, "dus": self._dus,
               "bytes_per_rank": int(small.numel() * 4 + colors.numel() * 4)}
        self._small, self._colors, self._twcs, self._dus = None, [], [], []
        self._early = None
        return out


def _start_gathers(colors, twcs, group):
    """-> (colors, all_colors, all_twcs, work handles): the two all-gathers of factorised_sum, started"""
    world = dist.get_world_size(group)
    N = colors.shape[1]
    all_colors = torch.empty((world * colors.shape[0], N, 3), dtype=colors.dtype, device=colors.device)
    all_twcs = torch.empty((world * twcs.shape[0], 3), dtype=twcs.dtype, device=twcs.device)
    w1 = dist.all_gather_into_tensor(all_twcs, twcs, group=group, async_op=True)
    w2 = dist.all_gather_into_tensor(all_colors, colors, group=group, async_op=True)
    return colors, all_colors, all_twcs, (w1, w2)


def factorised_sum(small, colors, twcs, group, expand, started=None):
    """The collective part of MultiViewStep.reduce: `small` (flat 11 N bucket) is summed over the
    ranks in place, `colors[V_local, N, 3]` / `twcs[V_local, 3]` are gathered from every rank (rank
    order, then local view order) and `expand(all_twcs, all_colors)` -> dL/dsh runs while the
    all-reduce is still in flight.  Works on any backend (gloo in the CPU tests)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return small, expand(twcs, colors)
    _, all_colors, all_twcs, (w1, w2) = started if started is not None else _start_gathers(colors, twcs, group)
    w3 = dist.all_reduce(small, op=dist.ReduceOp.SUM, group=group, async_op=True)
    w1.wait(); w2.wait()  # stream-ordered waits on NCCL; the all-reduce runs under the expansion
    dshs = expand(all_twcs, all_colors)
    w3.wait()
    return small, dshs


def prefer_fused_exchange(world):
    """Which gradient sum a training loop should use on `world` B200s of one NVSwitch node,
    from the measurements in profiles/ (bench.py times both at every world size):
    2 GPUs: GradExchange 1.876 ms/step vs 1.967 ms with NCCL (push hides under the backward,
    peer stores at ~500 GB/s); 8 GPUs: NCCL's in-switch (NVLS) reduction 2.075 ms vs 2.165 ms --
    with 7/8 of the bucket leaving every GPU in each phase the exchange is NVLink-bound and has
    only a 0.1 ms kernel to hide under.  4 GPUs is not measured; NCCL is assumed."""
    return world == 2
