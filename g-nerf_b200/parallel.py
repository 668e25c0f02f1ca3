"""Multi-GPU rendering: one process per GPU, rays are independent, one small exchange at the end.

Partition (SURVEY.md section 8(e)): by image first -- a GPU renders the images whose planes it holds, so
planes never move -- then by contiguous ray range inside an image when there are fewer images than GPUs.
The exchange is 136 bytes per ray (rgb [.,32] + depth [.,1] + weight_sum [.,1]) to every GPU, plus the one
cross-ray dependency: the global depth range MipRayMarcher2 clamps against
(training/volumetric_rendering/ray_marcher.py:50 reduces over the whole batch).  Two ways:
  * PeerGather (the GPU product path): the render kernel's epilogue stores each ray's outputs into this
    rank's slice of EVERY rank's gather buffers through peer-mapped NVLink pointers (tpr_render_peers), so the
    gather rides along with the render; one 2-float all-reduce carries the depth range and is also the barrier
    that completes the exchange.  No all-gather, no staging copy.
  * NCCL / gloo collectives (CPU tests, GPUs without peer access): every rank renders straight into its own
    slice of the gather buffers, then one all-reduce of the range and an in-place all-gather.
The host logic is backend-agnostic (NCCL on GPUs, gloo in the CPU tests); the per-shard render is the fused
CUDA renderer unless a test injects another callable.
"""
from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence

import torch
import torch.distributed as dist


@dataclass(frozen=True)
class Shard:
    image: int          # index into the global image batch
    ray_begin: int      # [ray_begin, ray_end) of that image
    ray_end: int

    @property
    def n_rays(self):
        return self.ray_end - self.ray_begin


def partition(n_img: int, n_rays: int, world: int) -> List[List[Shard]]:
    """Work list per rank.  n_img >= world: whole images, as evenly as possible (the first n_img % world
    ranks get one more).  n_img < world: ranks are dealt to images round-robin and each image's rays are cut
    into contiguous ranges over the ranks that share it."""
    if n_img <= 0 or n_rays <= 0 or world <= 0:
        raise ValueError('partition: n_img, n_rays and world must be positive')
    plan: List[List[Shard]] = [[] for _ in range(world)]
    if n_img >= world:
        base, extra = divmod(n_img, world)
        start = 0
        for r in range(world):
            cnt = base + (1 if r < extra else 0)
            plan[r] = [Shard(i, 0, n_rays) for i in range(start, start + cnt)]
            start += cnt
        return plan
    ranks_of = [[r for r in range(world) if r % n_img == i] for i in range(n_img)]
    for i, ranks in enumerate(ranks_of):
        k = len(ranks)
        base, extra = divmod(n_rays, k)
        begin = 0
        for j, r in enumerate(ranks):
            cnt = base + (1 if j < extra else 0)
            if cnt > 0:
                plan[r].append(Shard(i, begin, begin + cnt))
            begin += cnt
    return plan


def shard_ray_counts(plan: Sequence[Sequence[Shard]]) -> List[int]:
    return [sum(s.n_rays for s in shards) for shards in plan]


class _DeviceBlock:
    """A raw device allocation as a __cuda_array_interface__ object, so torch can wrap it without copying."""

    def __init__(self, ptr: int, n_floats: int):
        self.__cuda_array_interface__ = {'shape': (n_floats,), 'typestr': '<f4', 'data': (ptr, False), 'version': 2,
                                         'strides': None}


class PeerGather:
    """Gather buffers of one rank, mapped into every other rank of the node (NVLink / NVSwitch peer access).

    Holds ``sets`` (default 3, used round-robin) groups of three buffers -- rgb [world,n,m,32], depth [world,n,m,1],
    weight_sum [world,n,m,1] -- in ONE peer-mappable allocation (tpr_peer_alloc), exchanges the 64-byte IPC handles
    with ``all_gather_object`` and maps every peer's allocation (tpr_peer_open).  ``sinks(k)`` is the TprPeerSinks
    the render kernel needs to store this rank's slice into every peer; ``views(k)`` are this rank's own buffers.

    Lifetime of what ``render_sharded`` returns (the tensors ARE the gather buffers, no copy).  Rank A's render of step
    s+k (k = ``sets``) stores into the set that holds rank B's step-s outputs.  A can only launch that render after its
    all-reduce of step s+k-1 has completed, which needs B's all-reduce of step s+k-1 to be running on B's stream, i.e.
    everything B enqueued on that stream BEFORE its call s+k-1 has finished.  So: the outputs of call s may be read by
    work enqueued (on the stream the calls are made on) before this rank's call s+k-1 -- with the default three sets
    "until the call after the next one", with two sets only until the next call.  Reads enqueued later race with the
    peers' NVLink stores and see torn data; ``render_sharded`` therefore refuses fewer than two sets, and callers that
    keep results longer must clone them.
    """

    def __init__(self, n_local: int, n_rays: int, *, group=None, device=None, sets: int = 3):
        import ctypes
        from . import _lib
        if not dist.is_initialized():
            raise RuntimeError('PeerGather needs an initialised torch.distributed process group')
        self.group, self.world, self.rank = group, dist.get_world_size(group), dist.get_rank(group)
        if self.world - 1 > _lib.MAX_PEERS:
            raise RuntimeError(f'PeerGather supports at most {_lib.MAX_PEERS + 1} ranks')
        self.n, self.m, self.sets = int(n_local), int(n_rays), int(sets)
        if self.sets < 2:
            raise ValueError('PeerGather needs at least two buffer sets (a peer renders step s+1 into this rank while step s is read)')
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self._step = 0
        self._lib, self._ctypes = _lib, ctypes
        rays = self.world * self.n * self.m
        self._set_floats = rays * 34
        self._off = {'rgb': 0, 'depth': rays * 32, 'wsum': rays * 33}            # float offsets inside a set
        n_floats = self._set_floats * self.sets
        L = _lib.lib()
        ptr, handle = ctypes.c_void_p(), ctypes.create_string_buffer(_lib.PEER_HANDLE_BYTES)
        self._own, self._peer_base, self.flat = None, {}, None
        # Every step that can fail on ONE rank (allocation, IPC mapping) is followed by an exchange of the outcome, so that
        # all ranks raise together instead of one raising while the others wait in the next collective.
        with torch.cuda.device(self.device):
            err = None
            try:
                _lib.check(L.tpr_peer_alloc(n_floats * 4, ctypes.byref(ptr), handle), 'tpr_peer_alloc')
                self._own = ptr.value
                self.flat = torch.as_tensor(_DeviceBlock(self._own, n_floats), device=self.device)
                self.flat.zero_()
            except Exception as e:          # noqa: BLE001
                err = f'rank {self.rank}: {e}'
            handles = [None] * self.world
            dist.all_gather_object(handles, err if err is not None else handle.raw, group=group)
            failed = [h for h in handles if isinstance(h, str)]
            if not failed:
                try:
                    for r, h in enumerate(handles):
                        if r == self.rank:
                            continue
                        p = ctypes.c_void_p()
                        _lib.check(L.tpr_peer_open(h, ctypes.byref(p)), f'tpr_peer_open(rank {r})')
                        self._peer_base[r] = p.value
                except Exception as e:      # noqa: BLE001
                    err = f'rank {self.rank}: {e}'
                status = [None] * self.world
                dist.all_gather_object(status, err, group=group)
                failed = [s for s in status if s is not None]
            if failed:
                self._release()
                raise RuntimeError('PeerGather: ' + '; '.join(failed))
        dist.barrier(group=group)            # nobody renders into a peer before every rank has zeroed and mapped

    def _release(self):
        L = self._lib.lib()
        with torch.cuda.device(self.device):
            for p in self._peer_base.values():
                L.tpr_peer_close(self._ctypes.c_void_p(p))
            self.flat = None
            if self._own is not None:
                L.tpr_peer_free(self._ctypes.c_void_p(self._own))
        self._own, self._peer_base = None, {}

    def next_set(self) -> int:
        k = self._step % self.sets
        self._step += 1
        return k

    def views(self, k: int):
        """(rgb [world,n,m,32], depth [world,n,m,1], weight_sum [world,n,m,1]) of set k in this rank's memory."""
        base = k * self._set_floats
        rays = self.world * self.n * self.m
        mk = lambda off, c: self.flat[base + off: base + off + rays * c].view(self.world, self.n, self.m, c)   # noqa: E731
        return mk(self._off['rgb'], 32), mk(self._off['depth'], 1), mk(self._off['wsum'], 1)

    def sinks(self, k: int):
        """TprPeerSinks: where THIS rank's slice of set k lives in every peer's allocation."""
        s = self._lib.TprPeerSinks()
        s.n_peers = self.world - 1
        slice_rays = self.rank * self.n * self.m
        for i, (r, pb) in enumerate(sorted(self._peer_base.items())):
            b = pb + 4 * k * self._set_floats
            s.rgb[i] = b + 4 * (self._off['rgb'] + slice_rays * 32)
            s.depth[i] = b + 4 * (self._off['depth'] + slice_rays)
            s.weight_sum[i] = b + 4 * (self._off['wsum'] + slice_rays)
        return s

    def close(self):
        """Unmap the peers and free the allocation (collective: every rank must call it)."""
        if self._own is None:
            return
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        L = self._lib.lib()
        with torch.cuda.device(self.device):
            for p in self._peer_base.values():
                self._lib.check(L.tpr_peer_close(self._ctypes.c_void_p(p)), 'tpr_peer_close')
            dist.barrier(group=self.group)   # every mapping is gone before anybody frees
            self.flat = None
            self._lib.check(L.tpr_peer_free(self._ctypes.c_void_p(self._own)), 'tpr_peer_free')
        self._own, self._peer_base = None, {}


def _all_reduce_range(lo, hi, world, group):
    """(min over ranks of lo, max over ranks of hi) with ONE all-reduce: MAX of (-lo, hi)."""
    t = torch.cat([-lo, hi])
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return -t[0:1], t[1:2]


def _render_peer_gather(renderer, planes, decoder, ray_origins, ray_directions, rendering_options, noise, peer: 'PeerGather'):
    """render + gather in one kernel: see PeerGather."""
    n, m, _ = ray_origins.shape
    if (n, m) != (peer.n, peer.m):
        raise RuntimeError(f'PeerGather was built for {peer.n} images x {peer.m} rays per rank, got {n} x {m}')
    k = peer.next_set()
    bufs = peer.views(k)
    out = tuple(b[peer.rank] for b in bufs)
    renderer(planes, decoder, ray_origins, ray_directions, rendering_options, noise=noise, out=out, peer_sinks=peer.sinks(k))
    rng = renderer.last_depth_range
    # the depth range of the whole batch; on every rank this all-reduce completes only after every peer's render
    # kernel (and with it the peer's stores into this rank's buffers) has finished: it is the exchange's barrier
    lo, hi = _all_reduce_range(rng[0:1], rng[1:2], peer.world, peer.group)
    _clamp_cuda(bufs[1], lo, hi)             # nan_to_num + clamp of ALL gathered depths (4 bytes per ray)
    return tuple(b.view(peer.world * n, m, -1) for b in bufs)


def _default_local_render(renderer, planes, decoder, origins, dirs, options, noise, out):
    """Render one rank's rays with the fused CUDA renderer, leaving the global depth clamp to the caller."""
    renderer.defer_depth_clamp = True
    try:
        rgb, depth, wsum = renderer(planes, decoder, origins, dirs, options, noise=noise, out=out)
    finally:
        renderer.defer_depth_clamp = False
    return rgb, depth, wsum, renderer.last_depth_range


def render_sharded(renderer, planes, decoder, ray_origins, ray_directions, rendering_options, *,
                   group=None, noise=None, local_render: Optional[Callable] = None, gather: bool = True,
                   peer: Optional[PeerGather] = None):
    """Render THIS rank's images and return the whole job's outputs.  With ``peer`` (a PeerGather built once for
    this shape) the gather happens inside the render kernel over NVLink; without it, through collectives.

    planes [n_local,3,32,H,W], ray_origins / ray_directions [n_local,M,3]: this rank's share (image-sharded:
    every rank holds the same number of images).  Returns (rgb [world*n_local,M,32], depth [...,1],
    weight_sum [...,1]) in rank order when ``gather`` is true, else this rank's slice after the global clamp.
    """
    if peer is not None:
        return _render_peer_gather(renderer, planes, decoder, ray_origins, ray_directions, rendering_options, noise, peer)
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    n, m, _ = ray_origins.shape
    dev = ray_origins.device
    local_render = local_render or _default_local_render
    # gather buffers; this rank renders directly into its slice
    bufs = [torch.empty((world, n, m, c), device=dev, dtype=torch.float32) for c in (32, 1, 1)]
    out = tuple(b[rank] for b in bufs)
    rgb, depth, wsum, rng = local_render(renderer, planes, decoder, ray_origins, ray_directions, rendering_options, noise, out)
    for dst, src in zip(out, (rgb, depth, wsum)):
        if dst.data_ptr() != src.data_ptr():          # a local_render that ignored `out`
            dst.copy_(src)
    # the one cross-ray dependency: clamp(depth, min(all depths), max(all depths))
    lo, hi = _all_reduce_range(rng[0:1], rng[1:2], world, group)
    d = out[1]
    if d.is_cuda:
        _clamp_cuda(d, lo, hi)
    else:                                             # gloo / CPU tests
        d.copy_(torch.clamp(torch.nan_to_num(d, nan=float('inf')), lo, hi))
    if world == 1 or not gather:
        return out
    for b in bufs:
        dist.all_gather_into_tensor(b.view(-1), b[rank].reshape(-1), group=group)      # in place
    return tuple(b.view(world * n, m, -1) for b in bufs)


def _clamp_cuda(depth, lo, hi):
    import ctypes
    from . import _lib
    rr = torch.cat([lo, hi]).contiguous()
    with torch.cuda.device(depth.device):
        _lib.check(_lib.lib().tpr_clamp_depth(ctypes.c_void_p(depth.data_ptr()), depth.numel(),
                                              ctypes.c_void_p(rr.data_ptr()),
                                              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), 'tpr_clamp_depth')
    return depth


def render_ray_sharded(renderer, planes, decoder, ray_origins, ray_directions, rendering_options, *,
                       group=None, noise=None, local_render: Optional[Callable] = None):
    """Fewer images than GPUs: every rank holds ALL images (planes are 25 MB each) and renders the contiguous
    ray ranges `partition` assigns to it; the full [N,M,.] outputs are assembled on every rank with an
    all-gather of padded per-rank buffers."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    n, m, _ = ray_origins.shape
    dev = ray_origins.device
    plan = partition(n, m, world)
    local_render = local_render or _default_local_render
    cap = max(max((s.n_rays for s in shards), default=0) for shards in plan)
    per_rank = max(len(shards) for shards in plan)
    buf = torch.zeros((world, per_rank, cap, 34), device=dev, dtype=torch.float32)
    lo = torch.full((1,), float('inf'), device=dev)
    hi = torch.full((1,), float('-inf'), device=dev)
    for k, s in enumerate(plan[rank]):
        sl = slice(s.ray_begin, s.ray_end)
        nz = None
        if noise is not None:
            jit, u = noise
            df = u.shape[-1]
            nz = (jit[s.image:s.image + 1, sl], u.reshape(n, m, df)[s.image, sl].reshape(-1, df))
        rgb, depth, wsum, rng = local_render(renderer, planes[s.image:s.image + 1], decoder, ray_origins[s.image:s.image + 1, sl],
                                             ray_directions[s.image:s.image + 1, sl], rendering_options, nz, None)
        buf[rank, k, :s.n_rays, :32] = rgb[0]
        buf[rank, k, :s.n_rays, 32:33] = depth[0]
        buf[rank, k, :s.n_rays, 33:34] = wsum[0]
        lo = torch.minimum(lo, rng[0:1]); hi = torch.maximum(hi, rng[1:2])
    if world > 1:
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
        dist.all_gather_into_tensor(buf.view(-1), buf[rank].reshape(-1), group=group)
    rgb = torch.empty((n, m, 32), device=dev); depth = torch.empty((n, m, 1), device=dev); wsum = torch.empty((n, m, 1), device=dev)
    for r, shards in enumerate(plan):
        for k, s in enumerate(shards):
            sl = slice(s.ray_begin, s.ray_end)
            rgb[s.image, sl] = buf[r, k, :s.n_rays, :32]
            depth[s.image, sl] = buf[r, k, :s.n_rays, 32:33]
            wsum[s.image, sl] = buf[r, k, :s.n_rays, 33:34]
    depth = torch.clamp(torch.nan_to_num(depth, nan=float('inf')), lo, hi)
    return rgb, depth, wsum


# ----------------------------------------------------------------------------------------------------------------
# run_model (density grids, TriPlaneGenerator.sample / sample_mixed) sharded over point slabs
# ----------------------------------------------------------------------------------------------------------------
def point_slabs(n_pts: int, world: int) -> List[range]:
    """Contiguous slabs of the flattened point index, one per rank, as even as possible (the first n_pts % world ranks
    get one more).  For the density grid of gen_videos.py:33-55 the flattened index runs z-slowest, so a slab is a z-slab
    of the cube (SURVEY.md section 8(e))."""
    if n_pts <= 0 or world <= 0:
        raise ValueError('point_slabs: n_pts and world must be positive')
    base, extra = divmod(n_pts, world)
    out, begin = [], 0
    for r in range(world):
        cnt = base + (1 if r < extra else 0)
        out.append(range(begin, begin + cnt))
        begin += cnt
    return out


def run_model_sharded(renderer, planes, decoder, sample_coordinates, sample_directions, options, *, group=None,
                      want_rgb: bool = False, local_query: Optional[Callable] = None, gather: bool = True):
    """``ImportanceRenderer.run_model`` (VR/renderer.py:142-148) for one identity's planes held by EVERY rank (25 MB: each
    rank ran the backbone on the same ws with noise_mode='const', or received a broadcast) and the full coordinate tensor
    [N,P,3]: rank r queries the r-th contiguous slab of the P points and sigma (4 bytes per point; plus rgb, 128 bytes,
    only when asked for) is all-gathered in place, so every rank returns the complete {'rgb', 'sigma'} of the reference.
    ``gather=False`` returns this rank's slab only (a caller that writes its own z-slab of an .mrc volume).
    No collective touches the planes or the coordinates; density_noise is drawn per slab (each rank from its own generator).
    Inference only: the in-place all-gather would drop the other ranks' share of any gradient, so autograd raises."""
    if torch.is_grad_enabled():
        tensors = [planes, sample_coordinates] + (list(decoder.parameters()) if isinstance(decoder, torch.nn.Module) else [])
        if any(isinstance(t, torch.Tensor) and t.requires_grad for t in tensors):
            raise NotImplementedError('run_model_sharded is inference-only (its all-gather carries no gradient): call it under '
                                      'torch.no_grad() or use ImportanceRenderer.run_model for a differentiable query')
    world =dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    n, p, _ = sample_coordinates.shape
    slabs = point_slabs(p, world)
    mine = slabs[rank]
    query = local_query or (lambda xyz: renderer.run_model(planes, decoder, xyz, None, options, want_rgb=want_rgb))
    dev = sample_coordinates.device
    even = p % world == 0
    if not gather or world == 1:
        out = query(sample_coordinates[:, mine.start:mine.stop].contiguous()) if len(mine) else \
            {'rgb': torch.empty((n, 0, 32), device=dev) if want_rgb else None, 'sigma': torch.empty((n, 0, 1), device=dev)}
        return out
    cap = len(slabs[0])                                   # the largest slab
    # gather buffers [world, N, cap, C]: with one image and equal slabs that IS the [N,P,C] result, no unpacking copy
    chans = [('sigma', 1)] + ([('rgb', 32)] if want_rgb else [])
    bufs = {k: torch.empty((world, n, cap, c), device=dev, dtype=torch.float32) for k, c in chans}
    if len(mine):
        res = query(sample_coordinates[:, mine.start:mine.stop].contiguous())
        for k, _ in chans:
            bufs[k][rank, :, :len(mine)] = res[k]
    for k, _ in chans:
        dist.all_gather_into_tensor(bufs[k].view(-1), bufs[k][rank].reshape(-1), group=group)        # in place
    out = {'rgb': None}
    for k, c in chans:
        if n == 1 and even:
            out[k] = bufs[k].view(1, p, c)
        else:
            full = torch.empty((n, p, c), device=dev, dtype=torch.float32)
            for r, sl in enumerate(slabs):
                full[:, sl.start:sl.stop] = bufs[k][r, :, :len(sl)]
            out[k] = full
    return out
