"""ImportanceRenderer with the reference's interface, backed by the fused sm_100a kernels.

Mirrors /root/reference/g_nerf/training/volumetric_rendering/renderer.py (VR/renderer.py below):
same class name, same ``forward(planes, decoder, ray_origins, ray_directions, rendering_options)``
(:88) returning ``(rgb [N,M,32], depth [N,M,1], weight_sum [N,M,1])`` (:140), same
``run_model(planes, decoder, sample_coordinates, sample_directions, options)`` (:142-148), same
``plane_axes`` attribute (:86).  What happens inside is one fused kernel (csrc/triplane_b200.cu)
instead of ~40 ATen launches; nothing here computes the result with torch ops and there is no
CPU path -- CPU tensors raise.
"""
import ctypes

import torch

from .. import _lib
from . import math_utils
from .ray_marcher import MipRayMarcher2


def generate_planes():
    """The three plane axis triples (VR/renderer.py:23-37).  Kept as the public attribute the
    reference exposes; the kernels hard-code the resulting projection
    (plane 0 <- (x,y), plane 1 <- (x,z), plane 2 <- (z,x))."""
    return torch.tensor([[[1, 0, 0], [0, 1, 0], [0, 0, 1]],
                         [[1, 0, 0], [0, 0, 1], [0, 1, 0]],
                         [[0, 0, 1], [1, 0, 0], [0, 1, 0]]], dtype=torch.float32)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def project_onto_planes(planes, coordinates):
    """plane axes [n_planes,3,3], coordinates [N,M,3] -> projections [N*n_planes,M,2] (VR/renderer.py:39-53): the first two
    components of the point in each plane's basis.  forward() never calls this (the kernels hard-code the three
    resulting index pairs); kept because it is a public name of the reference module.  A handful of floats per plane, so
    it is plain tensor algebra on whatever device the inputs live on."""
    n, m, _ = coordinates.shape
    n_planes = planes.shape[0]
    basis = torch.linalg.inv(planes.to(coordinates))                       # [n_planes,3,3]
    return torch.einsum('nmc,pcd->npmd', coordinates, basis)[..., :2].reshape(n * n_planes, m, 2)


def sample_from_planes(plane_axes, plane_features, coordinates, mode='bilinear', padding_mode='zeros', box_warp=None):
    """plane_features [N,3,32,H,W] (or PackedPlanes), coordinates [N,M,3] -> [N,3,M,32]: the bilinear lookups on the three
    planes, not summed (VR/renderer.py:55-65) -- the tensor OSGDecoder.forward takes.  ``plane_axes`` must be the
    reference's three planes (generate_planes()): the kernel hard-codes their projection."""
    assert padding_mode == 'zeros'                                          # VR/renderer.py:56
    if mode != 'bilinear':
        raise NotImplementedError("sample_from_planes: only mode='bilinear' (what the reference's renderer uses)")
    if plane_axes is not None and not torch.equal(torch.as_tensor(plane_axes).detach().float().cpu(), generate_planes()):
        raise NotImplementedError('sample_from_planes: the B200 gather is specialised for the plane axes of generate_planes()')
    xyz = _require_cuda_f32(coordinates, 'coordinates', (3,))
    _forbid_autograd(plane_features if isinstance(plane_features, torch.Tensor) else None, xyz)
    pp = pack_planes(plane_features)
    n, m, _ = xyz.shape
    if pp.n_img != n:
        raise RuntimeError(f'batch mismatch: planes N={pp.n_img}, coordinates N={n}')
    with torch.cuda.device(xyz.device):
        out = torch.empty((n, 3, m, 32), device=xyz.device, dtype=torch.float32)
        _lib.check(_lib.lib().tpr_sample_planes(_ptr(pp.data), n, pp.height, pp.width, _ptr(xyz), m, float(box_warp), _ptr(out),
                                                _stream()), 'tpr_sample_planes')
    return out


def sample_from_3dgrid(grid, coordinates):
    """grid [1 or N,C,D,H,W], coordinates [N,P,3] in [-1,1] -> [N,P,C], trilinear with zero padding (VR/renderer.py:67-80;
    the reference never calls it)."""
    grid = _require_cuda_f32(grid, 'grid')
    xyz = _require_cuda_f32(coordinates, 'coordinates', (3,))
    _forbid_autograd(grid, xyz)
    if grid.dim() != 5:
        raise RuntimeError(f'grid must be [1 or N,C,D,H,W], got {tuple(grid.shape)}')
    n, p, _ = xyz.shape
    g, c, d, h, w = grid.shape
    with torch.cuda.device(xyz.device):
        out = torch.empty((n, p, c), device=xyz.device, dtype=torch.float32)
        _lib.check(_lib.lib().tpr_sample_3dgrid(_ptr(grid), g, c, d, h, w, _ptr(xyz), n, p, _ptr(out), _stream()),
                   'tpr_sample_3dgrid')
    return out


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_cuda_f32(t, name, shape_tail=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f'{name} must be a torch.Tensor')
    if not t.is_cuda:
        raise RuntimeError(f'{name} is on {t.device}: the B200 tri-plane renderer has no CPU path '
                           f'(use the reference renderer for CPU tensors)')
    if t.dtype != torch.float32:
        raise RuntimeError(f'{name} must be float32, got {t.dtype}')
    if shape_tail is not None and tuple(t.shape[-len(shape_tail):]) != tuple(shape_tail):
        raise RuntimeError(f'{name} has shape {tuple(t.shape)}, expected (..., {", ".join(map(str, shape_tail))})')
    return t.contiguous()


def _forbid_autograd(*tensors):
    if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in tensors):
        raise NotImplementedError(
            'this entry point of the B200 tri-plane renderer is forward-only: call it under torch.no_grad() or with '
            'requires_grad_(False) inputs (ImportanceRenderer.forward differentiates w.r.t. planes and the decoder only)')


def _wants_grad(planes, decoder):
    """Does the caller expect gradients for the planes or the decoder's parameters?"""
    if isinstance(planes, torch.Tensor) and planes.requires_grad:
        return True
    net = getattr(decoder, 'net', None)
    if net is None:
        return False
    return any(p.requires_grad for p in decoder.parameters())


class PackedPlanes:
    """Tri-planes repacked channels-last ([N,3,H,W,32]: one texel = one 128-byte line)."""

    def __init__(self, data, n_img, height, width):
        self.data, self.n_img, self.height, self.width = data, n_img, height, width

    @property
    def device(self):
        return self.data.device


def pack_planes(planes) -> PackedPlanes:
    """[N,3,32,H,W] (training/triplane.py:74) -> PackedPlanes.  Pass the result to forward/run_model
    in place of ``planes`` to reuse one packing across frames."""
    if isinstance(planes, PackedPlanes):
        return planes
    planes = _require_cuda_f32(planes, 'planes')
    if planes.dim() != 5 or planes.shape[1] != 3 or planes.shape[2] != 32:
        raise RuntimeError(f'planes must be [N,3,32,H,W], got {tuple(planes.shape)}')
    n, _, _, h, w = planes.shape
    out = torch.empty((n, 3, h, w, 32), dtype=torch.float32, device=planes.device)
    with torch.cuda.device(planes.device):
        _lib.check(_lib.lib().tpr_pack_planes(_ptr(planes), n, h, w, _ptr(out), _stream()), 'tpr_pack_planes')
    return PackedPlanes(out, n, h, w)


def pack_decoder(decoder, *, allow_grad=False) -> torch.Tensor:
    """Read an OSGDecoder-shaped module (training/triplane.py:113-122: net[0] = FC 32->64,
    net[1] = Softplus, net[2] = FC 64->33) and pack its parameters with the runtime gains
    (training/networks_stylegan2.py:118-119).  Anything else raises: there is no generic fallback."""
    net = getattr(decoder, 'net', None)
    if net is None or len(net) != 3:
        raise RuntimeError('decoder must be OSGDecoder-shaped: .net = [FullyConnectedLayer, Softplus, FullyConnectedLayer]')
    fc1, act, fc2 = net[0], net[1], net[2]
    if not isinstance(act, torch.nn.Softplus) or act.beta != 1 or act.threshold != 20:
        raise RuntimeError('decoder.net[1] must be torch.nn.Softplus(beta=1, threshold=20)')
    for fc, shape in ((fc1, (64, 32)), (fc2, (33, 64))):
        if tuple(fc.weight.shape) != shape or fc.bias is None or getattr(fc, 'activation', 'linear') != 'linear':
            raise RuntimeError(f'decoder layer must be a linear FullyConnectedLayer with weight {shape} and a bias')
    if not allow_grad:
        _forbid_autograd(fc1.weight, fc1.bias, fc2.weight, fc2.bias)
    w1 = _require_cuda_f32(fc1.weight.detach(), 'decoder.net[0].weight')
    b1 = _require_cuda_f32(fc1.bias.detach(), 'decoder.net[0].bias')
    w2 = _require_cuda_f32(fc2.weight.detach(), 'decoder.net[2].weight')
    b2 = _require_cuda_f32(fc2.bias.detach(), 'decoder.net[2].bias')
    L = _lib.lib()
    out = torch.empty(L.tpr_packed_decoder_bytes() // 4, dtype=torch.float32, device=w1.device)
    with torch.cuda.device(w1.device):
        _lib.check(L.tpr_pack_decoder(_ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2),
                                      float(fc1.weight_gain), float(fc1.bias_gain),
                                      float(fc2.weight_gain), float(fc2.bias_gain), _ptr(out), _stream()),
                   'tpr_pack_decoder')
    return out


def _density_noise(options):
    dn = float(options.get('density_noise', 0) or 0)                      # options.get('density_noise', 0) > 0, VR/renderer.py:146
    return dn if dn > 0 else 0.0


def _draw_noise(noise, n, m, dc, df, dn, dev, per_ray_limits=False):
    """The forward's random draws, made with the reference's own torch calls in the reference's order so that the CUDA
    generator advances exactly as the reference advances it: rand_like [N,M,Dc,1] (VR/renderer.py:190), then -- only
    with density_noise > 0 -- randn_like [N,M*Dc,1] (:146, coarse run_model), rand [N*M,Df] (:237), randn_like
    [N,M*Df,1] (:146, fine run_model).  ``noise`` = (jitter, u[, coarse noise, fine noise]) overrides them (parity
    tests feed the oracle and the kernels the same numbers)."""
    if noise is None:
        if per_ray_limits:
            # the 'auto' branch builds its depths as math_utils.linspace(...) [D,N,M,1] .permute(1,2,0,3) and calls rand_like
            # on that VIEW (VR/renderer.py:184-186): rand_like keeps the strides and fills in memory order, i.e. the draw is
            # rand([D,N,M,1]) seen through the same permutation
            jitter = torch.rand((dc, n, m, 1), device=dev, dtype=torch.float32).permute(1, 2, 0, 3).contiguous()
        else:
            jitter = torch.rand((n, m, dc, 1), device=dev, dtype=torch.float32)
        nz_c = torch.randn((n, m * dc, 1), device=dev, dtype=torch.float32) if dn > 0 else None
        u = torch.rand(n * m, df, device=dev) if df > 0 else None
        nz_f = torch.randn((n, m * df, 1), device=dev, dtype=torch.float32) if dn > 0 and df > 0 else None
        return jitter, u, nz_c, nz_f
    jitter = _require_cuda_f32(noise[0], 'noise[0]').reshape(n, m, dc, 1)
    u = _require_cuda_f32(noise[1], 'noise[1]').reshape(n * m, df) if df > 0 else None
    nz_c = nz_f = None
    if dn > 0:
        if len(noise) < 4:
            raise RuntimeError('density_noise > 0: noise must be (jitter, u, coarse density noise, fine density noise)')
        nz_c = _require_cuda_f32(noise[2], 'noise[2]').reshape(n, m * dc, 1)
        nz_f = _require_cuda_f32(noise[3], 'noise[3]').reshape(n, m * df, 1) if df > 0 else None
    return jitter, u, nz_c, nz_f


def _layout_flag(options):
    mode = options.get('output_layout', 'channels_last')
    if mode == 'channels_last':
        return _lib.LAYOUT_CHANNELS_LAST
    if mode == 'channels_first':
        return _lib.LAYOUT_CHANNELS_FIRST
    raise RuntimeError(f"rendering_options['output_layout'] must be 'channels_last' or 'channels_first', got {mode!r}")


def _mlp_flag(options):
    mode = options.get('decoder_precision', 'fp32')
    if mode == 'fp32':
        return _lib.MLP_FP32
    if mode == 'bf16':
        return _lib.MLP_BF16
    if mode == 'fp32_ffma':
        return _lib.MLP_FFMA
    raise RuntimeError(f"rendering_options['decoder_precision'] must be 'fp32', 'bf16' or 'fp32_ffma', got {mode!r}")


class ImportanceRenderer(torch.nn.Module):
    _timing_events = None

    def __init__(self):
        super().__init__()
        self.ray_marcher = MipRayMarcher2()
        self.plane_axes = generate_planes()
        # set by forward(); lets callers that shard rays over GPUs finish the global depth clamp
        self.last_depth_range = None
        self.last_fine = None
        self.debug_outputs = False
        self.defer_depth_clamp = False
        # plane cache (SURVEY.md section 8(f) row 1): remember the last repacked planes and reuse them while the caller
        # keeps passing the same, unmodified tensor (gen_videos.py renders 120 frames of one identity)
        self.cache_packed_planes = False
        self._plane_cache = None
        # training: let the forward kernel keep every sample's colours / sigma for the backward (132 B per sample);
        # False = keep nothing per sample, the backward re-evaluates them (3 ms more at config 2)
        self.keep_samples = True
        self.keep_features = True          # ... and its 32 summed plane features (128 B more per sample): no second gather

    def _packed(self, planes):
        """pack_planes with a one-entry cache.  A hit needs the same storage address, shape and version counter; the
        cache holds a reference to the tensor it packed, so that address cannot have been recycled for other data."""
        if isinstance(planes, PackedPlanes) or not self.cache_packed_planes or not isinstance(planes, torch.Tensor):
            return pack_planes(planes)
        key = (planes.data_ptr(), tuple(planes.shape), planes._version, planes.device)
        hit = self._plane_cache
        if hit is not None and hit[0] == key:
            return hit[2]
        pp = pack_planes(planes)
        self._plane_cache = (key, planes, pp)
        return pp

    # ------------------------------------------------------------------ forward (VR/renderer.py:88-140)
    def forward(self, planes, decoder, ray_origins, ray_directions, rendering_options, *, noise=None, out=None,
                peer_sinks=None):
        """``noise=(jitter [N,M,Dc,1], u [N*M,Df])`` overrides the two uniform draws (used by parity
        tests, which must feed the oracle and the kernels the same numbers); by default they are drawn
        with the reference's own torch calls in the reference's order (VR/renderer.py:190,237).
        ``out=(rgb, depth, weight_sum)`` renders into caller-owned contiguous tensors (the multi-GPU path
        passes slices of its gather buffers).  ``peer_sinks`` (a ``_lib.TprPeerSinks``, built by
        ``parallel.PeerGather``): the kernel also stores every ray's outputs into the peer GPUs' gather buffers over
        NVLink and leaves the depth clamp to the caller (it needs the all-reduced range)."""
        if torch.is_grad_enabled() and _wants_grad(planes, decoder):
            # training / fine-tuning (training/training_loop.py:335,377): same kernels forward, CUDA backward w.r.t.
            # planes and decoder (volumetric_rendering/backward.py)
            from .backward import render_with_grad
            if out is not None or peer_sinks is not None:
                raise NotImplementedError('out= / peer_sinks= are inference-only (no autograd through them)')
            return render_with_grad(self, planes, decoder, ray_origins, ray_directions, rendering_options, noise)
        return self._forward_impl(planes, decoder, ray_origins, ray_directions, rendering_options, noise=noise, out=out,
                                  peer_sinks=peer_sinks)[:3]

    def _forward_impl(self, planes, decoder, ray_origins, ray_directions, rendering_options, *, noise=None, out=None,
                      peer_sinks=None, train=False):
        """The forward proper.  Returns (rgb, depth, weight_sum, aux); ``train=True`` (the autograd path) additionally
        keeps what the backward needs in ``aux``: packed planes / decoder, the coarse and importance depths, the range."""
        opts = rendering_options
        ray_origins = _require_cuda_f32(ray_origins, 'ray_origins', (3,))
        ray_directions = _require_cuda_f32(ray_directions, 'ray_directions', (3,))
        _forbid_autograd(None if train or not isinstance(planes, torch.Tensor) else planes, ray_origins, ray_directions)
        if opts.get('clamp_mode', None) != 'softplus':
            raise AssertionError('MipRayMarcher only supports `clamp_mode`=`softplus`!')      # VR/ray_marcher.py:35
        dn = _density_noise(opts)
        pp = self._packed(planes)
        n, m, _ = ray_origins.shape
        # N cameras over N plane sets (the reference's batch), or F*P cameras over P plane sets, camera n sampling
        # set n % P: F frames of an orbit, each a batch of P identities, as one call (SURVEY.md section 8(f) row 4)
        if n % pp.n_img != 0 or ray_directions.shape != ray_origins.shape:
            raise RuntimeError(f'batch mismatch: planes N={pp.n_img}, origins {tuple(ray_origins.shape)}, '
                               f'directions {tuple(ray_directions.shape)}')
        layout = _layout_flag(opts)
        clamp_group = int(opts.get('depth_clamp_group', 0))
        dev = ray_origins.device
        dec = pack_decoder(decoder, allow_grad=train)
        dc = int(opts['depth_resolution'])
        df = int(opts['depth_resolution_importance'])
        L = _lib.lib()

        rs_t = re_t = None
        if opts['ray_start'] == opts['ray_end'] == 'auto':                                # VR/renderer.py:91-97
            if opts.get('disparity_space_sampling', False):
                # the reference's disparity branch (VR/renderer.py:174-181) takes python floats; with the per-ray tensors of
                # the 'auto' branch it dies on a shape mismatch.  Fail as loudly instead of sampling NaN depths.
                raise RuntimeError("ray_start = ray_end = 'auto' cannot be combined with disparity_space_sampling")
            rs_t, re_t = math_utils.get_ray_limits_box(ray_origins, ray_directions, box_side_length=opts['box_warp'])
            valid = re_t > rs_t
            if torch.any(valid).item():
                lo, hi = rs_t[valid].min(), rs_t[valid].max()
                rs_t[~valid] = lo
                re_t[~valid] = hi
            rs_t, re_t = rs_t.reshape(-1).contiguous(), re_t.reshape(-1).contiguous()
            ray_start = ray_end = 0.0
        else:
            ray_start, ray_end = float(opts['ray_start']), float(opts['ray_end'])

        with torch.cuda.device(dev):
            jitter, u, nz_c, nz_f = _draw_noise(noise, n, m, dc, df, dn, dev, per_ray_limits=rs_t is not None)
            o = _lib.TprOptions(ray_start=ray_start, ray_end=ray_end, box_warp=float(opts['box_warp']),
                                depth_resolution=dc, depth_resolution_importance=df,
                                disparity_space_sampling=int(bool(opts.get('disparity_space_sampling', False))),
                                white_back=int(bool(opts.get('white_back', False))), flags=_mlp_flag(opts),
                                tile_width=0, plane_sets=pp.n_img, output_layout=layout, depth_clamp_group=clamp_group,
                                density_noise=dn, density_noise_coarse=nz_c.data_ptr() if nz_c is not None else None,
                                density_noise_fine=nz_f.data_ptr() if nz_f is not None else None)
            if out is None and layout == _lib.LAYOUT_CHANNELS_FIRST:
                # Memory is [N,32,M] -- the feature image of training/triplane.py:81 -- and the tensor returned is its
                # [N,M,32] view, so the caller's `permute(0, 2, 1).reshape(N, 32, H, W).contiguous()` is a no-op
                rgb = torch.empty((n, 32, m), device=dev, dtype=torch.float32).permute(0, 2, 1)
                depth = torch.empty((n, m, 1), device=dev, dtype=torch.float32)
                wsum = torch.empty((n, m, 1), device=dev, dtype=torch.float32)
            elif out is None:
                rgb = torch.empty((n, m, 32), device=dev, dtype=torch.float32)
                depth = torch.empty((n, m, 1), device=dev, dtype=torch.float32)
                wsum = torch.empty((n, m, 1), device=dev, dtype=torch.float32)
            else:
                rgb, depth, wsum = out
                for t, c in ((rgb, 32), (depth, 1), (wsum, 1)):
                    dense = t.permute(0, 2, 1).is_contiguous() if (c == 32 and layout == _lib.LAYOUT_CHANNELS_FIRST) else t.is_contiguous()
                    if tuple(t.shape) != (n, m, c) or t.dtype != torch.float32 or t.device != dev or not dense:
                        raise RuntimeError(f'out tensors must be dense float32 [{n},{m},{c}] on {dev} '
                                           f"(rgb: the [N,M,32] view of an [N,32,M] buffer when output_layout='channels_first')")
            rng = torch.empty(2, device=dev, dtype=torch.float32)
            nscratch = L.tpr_render_scratch_bytes(n, m, ctypes.byref(o))
            scratch = torch.empty(nscratch, device=dev, dtype=torch.uint8)
            fine_d = fine_i = None
            if (self.debug_outputs or train) and df > 0:
                fine_d = torch.empty((n * m, df), device=dev, dtype=torch.float32)
                fine_i = torch.empty((n * m, df), device=dev, dtype=torch.int32)
            ev = self._timing_events          # bench.py: CUDA events bracketing the render launch on this stream
            if ev is not None:
                ev[0].record()
            saved = None
            if train and getattr(self, 'keep_samples', True):
                # keep every sample's colours / sigma for the backward (tpr_render_train); `kept` says whether the kernel that
                # ran could (the warp-specialised one), otherwise the backward re-evaluates them
                s_tot = dc + df
                s_col = torch.empty((n * m * s_tot, 32), device=dev, dtype=torch.float32)
                s_sig = torch.empty((n * m * s_tot,), device=dev, dtype=torch.float32)
                s_feat = (torch.empty((n * m * s_tot, 32), device=dev, dtype=torch.float32)
                          if getattr(self, 'keep_features', True) else None)
                kept = ctypes.c_int32(0)
                _lib.check(L.tpr_render_train(_ptr(pp.data), n, pp.height, pp.width, _ptr(dec), _ptr(ray_origins),
                                              _ptr(ray_directions), m, _ptr(jitter), _ptr(u), _ptr(rs_t), _ptr(re_t),
                                              ctypes.byref(o), _ptr(rgb), _ptr(depth), _ptr(wsum), _ptr(fine_d), _ptr(rng),
                                              _ptr(s_col), _ptr(s_sig), _ptr(s_feat), ctypes.byref(kept), _ptr(scratch), nscratch,
                                              _stream()),
                           'tpr_render_train')
                saved = (s_col, s_sig, s_feat) if kept.value else None
                if dn > 0 and saved is None:
                    raise NotImplementedError('density_noise > 0 with autograd needs the forward to keep its samples '
                                              '(keep_samples = True and 48+48-class sample counts): the backward would '
                                              're-evaluate sigma without the noise')
            elif peer_sinks is not None:
                _lib.check(L.tpr_render_peers(_ptr(pp.data), n, pp.height, pp.width, _ptr(dec), _ptr(ray_origins),
                                              _ptr(ray_directions), m, _ptr(jitter), _ptr(u), _ptr(rs_t), _ptr(re_t),
                                              ctypes.byref(o), _ptr(rgb), _ptr(depth), _ptr(wsum), _ptr(rng), _ptr(scratch),
                                              nscratch, ctypes.byref(peer_sinks), _stream()), 'tpr_render_peers')
            else:
                _lib.check(L.tpr_render(_ptr(pp.data), n, pp.height, pp.width, _ptr(dec), _ptr(ray_origins),
                                        _ptr(ray_directions), m, _ptr(jitter), _ptr(u), _ptr(rs_t), _ptr(re_t),
                                        ctypes.byref(o), _ptr(rgb), _ptr(depth), _ptr(wsum), _ptr(fine_d), _ptr(fine_i),
                                        _ptr(rng), 0 if self.defer_depth_clamp else 1, _ptr(scratch), nscratch, _stream()),
                           'tpr_render')
            if ev is not None:
                ev[1].record()
            aux = None
            if train:
                # the coarse depths the kernel derived from `jitter` (same device function, VR/renderer.py:169-192)
                coarse_d = torch.empty((n * m, dc), device=dev, dtype=torch.float32)
                _lib.check(L.tpr_sample_stratified(_ptr(jitter), n * m, _ptr(rs_t), _ptr(re_t), ctypes.byref(o), _ptr(coarse_d),
                                                   _stream()), 'tpr_sample_stratified')
                o.density_noise, o.density_noise_coarse, o.density_noise_fine = 0.0, None, None   # (constants of the graph)
                aux = dict(packed=pp, dec=dec, coarse=coarse_d, fine=fine_d, range=rng, options=o, saved=saved)
        self.last_depth_range = rng
        self.last_scratch = scratch                    # TPR_PHASE_TIMING=1: int64 phase counters at byte 64
        self.last_fine = (fine_d, fine_i)
        self._noise_keepalive = (nz_c, nz_f)            # the kernel reads them asynchronously
        return rgb, depth, wsum, aux

    # ------------------------------------------------------------------ forward with host buffers
    def forward_host(self, planes, decoder, ray_origins, ray_directions, rendering_options, *, noise=None, out=None,
                     defer_depth=False):
        """``forward`` for a caller whose tensors live in (pinned) HOST memory: ``planes`` [N,3,32,H,W],
        ``ray_origins`` / ``ray_directions`` [N,M,3] are CPU tensors and the three outputs are returned as pinned CPU
        tensors (or written into ``out``).  The library pipelines H2D copy, repack + render and D2H copy image by
        image (tpr_render_host), so the call costs about max(PCIe time, render time) instead of their sum.  The
        result is complete once the current CUDA stream has been synchronised.  Scalar ray limits only.
        ``defer_depth=True`` (rays sharded over GPUs): depth is left unclamped on the device and ``last_depth_range`` holds
        this GPU's range; all-reduce it (MIN, MAX) and call ``finish_host_depth(range)`` to clamp and fetch ``out[1]``."""
        opts = rendering_options
        for t, name in ((planes, 'planes'), (ray_origins, 'ray_origins'), (ray_directions, 'ray_directions')):
            if not isinstance(t, torch.Tensor) or t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
                raise RuntimeError(f'forward_host: {name} must be a contiguous float32 CPU tensor (pinned for async copies)')
        if planes.dim() != 5 or planes.shape[1] != 3 or planes.shape[2] != 32:
            raise RuntimeError(f'planes must be [N,3,32,H,W], got {tuple(planes.shape)}')
        if opts.get('clamp_mode', None) != 'softplus':
            raise AssertionError('MipRayMarcher only supports `clamp_mode`=`softplus`!')      # VR/ray_marcher.py:35
        dn = _density_noise(opts)
        if isinstance(opts['ray_start'], str) or isinstance(opts['ray_end'], str):
            raise NotImplementedError("forward_host supports scalar ray limits only (use forward() for 'auto')")
        n, _, _, h, w = planes.shape
        m = ray_origins.shape[1]
        if tuple(ray_origins.shape) != (n, m, 3) or ray_directions.shape != ray_origins.shape:
            raise RuntimeError(f'batch mismatch: planes N={n}, origins {tuple(ray_origins.shape)}, '
                               f'directions {tuple(ray_directions.shape)}')
        dec = pack_decoder(decoder)                  # the decoder's parameters are device tensors
        dev = dec.device
        dc = int(opts['depth_resolution'])
        df = int(opts['depth_resolution_importance'])
        L = _lib.lib()
        with torch.cuda.device(dev):
            jitter, u, nz_c, nz_f = _draw_noise(noise, n, m, dc, df, dn, dev)
            o = _lib.TprOptions(ray_start=float(opts['ray_start']), ray_end=float(opts['ray_end']),
                                box_warp=float(opts['box_warp']), depth_resolution=dc, depth_resolution_importance=df,
                                disparity_space_sampling=int(bool(opts.get('disparity_space_sampling', False))),
                                white_back=int(bool(opts.get('white_back', False))), flags=_mlp_flag(opts), tile_width=0,
                                density_noise=dn, density_noise_coarse=nz_c.data_ptr() if nz_c is not None else None,
                                density_noise_fine=nz_f.data_ptr() if nz_f is not None else None)
            if out is None:
                out = tuple(torch.empty((n, m, c), dtype=torch.float32).pin_memory() for c in (32, 1, 1))
            for t, c in zip(out, (32, 1, 1)):
                if tuple(t.shape) != (n, m, c) or t.dtype != torch.float32 or t.is_cuda or not t.is_contiguous():
                    raise RuntimeError(f'out tensors must be contiguous float32 CPU tensors [{n},{m},{c}]')
            nws = L.tpr_render_host_workspace_bytes(n, h, w, m)
            ws = getattr(self, '_host_ws', None)
            if ws is None or ws.numel() < nws or ws.device != dev:
                # kept for the renderer's lifetime: the library's copy streams use it behind torch's allocator's back
                ws = self._host_ws = torch.empty(nws, device=dev, dtype=torch.uint8)
            rng = torch.empty(2, device=dev, dtype=torch.float32)
            _lib.check(L.tpr_render_host(_ptr(planes), n, h, w, _ptr(dec), _ptr(ray_origins), _ptr(ray_directions), m,
                                         _ptr(jitter), _ptr(u), ctypes.byref(o), _ptr(out[0]), None if defer_depth else _ptr(out[1]),
                                         _ptr(out[2]), _ptr(rng), _ptr(ws), ws.numel(), _stream()), 'tpr_render_host')
            self._host_keepalive = (dec, jitter, u, nz_c, nz_f, planes, ray_origins, ray_directions)    # until the next call
        self.last_depth_range = rng
        self._host_pending = (n, h, w, m, out) if defer_depth else None
        return out

    def finish_host_depth(self, depth_range):
        """Second half of ``forward_host(defer_depth=True)``: clamp the depth left on the device against ``depth_range``
        (a device tensor [2]: the all-reduced (min, max) of every rank's ``last_depth_range``) and copy it into ``out[1]``."""
        if getattr(self, '_host_pending', None) is None:
            raise RuntimeError('finish_host_depth: no forward_host(defer_depth=True) call is pending')
        n, h, w, m, out = self._host_pending
        rr = _require_cuda_f32(depth_range, 'depth_range').reshape(2)
        ws = self._host_ws
        with torch.cuda.device(ws.device):
            _lib.check(_lib.lib().tpr_render_host_depth(_ptr(ws), ws.numel(), n, h, w, m, _ptr(rr), _ptr(out[1]), _stream()),
                       'tpr_render_host_depth')
        self._host_pending = None
        self._host_keepalive = self._host_keepalive + (rr,)
        return out

    # ------------------------------------------------------------------ run_model (VR/renderer.py:142-148)
    def run_model(self, planes, decoder, sample_coordinates, sample_directions, options, *, want_rgb=True, sigma_noise=None):
        """``sample_directions`` is accepted and ignored, exactly like OSGDecoder ignores it
        (training/triplane.py:124-136).  ``options['density_noise'] > 0`` adds ``randn_like(sigma) * density_noise``
        (VR/renderer.py:146); ``sigma_noise`` [N,P,1] overrides the draw (tests).
        Under autograd (planes or decoder parameters that require grad) the result is attached to them: this is the body of
        TriPlaneGenerator.sample / sample_mixed (training/triplane.py:92-104), e.g. EG3D's density regulariser."""
        if torch.is_grad_enabled() and _wants_grad(planes, decoder):
            from .backward import run_model_with_grad
            return run_model_with_grad(self, planes, decoder, sample_coordinates, options, want_rgb, sigma_noise)
        return self._run_model_impl(planes, decoder, sample_coordinates, options, want_rgb=want_rgb, sigma_noise=sigma_noise)[0]

    def _run_model_impl(self, planes, decoder, sample_coordinates, options, *, want_rgb=True, sigma_noise=None, train=False):
        """The point query proper.  Returns ({'rgb', 'sigma'}, aux); ``train=True`` (the autograd path) lets the decoder
        require grad and returns in ``aux`` what the backward needs: the packed planes and decoder and the coordinates."""
        xyz = _require_cuda_f32(sample_coordinates, 'sample_coordinates', (3,))
        _forbid_autograd(None if train or not isinstance(planes, torch.Tensor) else planes, xyz)
        dn = _density_noise(options)
        pp = self._packed(planes)
        n, p, _ = xyz.shape
        if pp.n_img != n:
            raise RuntimeError(f'batch mismatch: planes N={pp.n_img}, coordinates N={n}')
        dec = pack_decoder(decoder, allow_grad=train)
        dev = xyz.device
        with torch.cuda.device(dev):
            rgb = torch.empty((n, p, 32), device=dev, dtype=torch.float32) if want_rgb else None
            sigma = torch.empty((n, p, 1), device=dev, dtype=torch.float32)
            _lib.check(_lib.lib().tpr_run_model(_ptr(pp.data), n, pp.height, pp.width, _ptr(dec), _ptr(xyz), p,
                                                float(options['box_warp']), _ptr(rgb), _ptr(sigma),
                                                _mlp_flag(options), _stream()), 'tpr_run_model')
            if dn > 0:
                nz = (torch.randn((n, p, 1), device=dev, dtype=torch.float32) if sigma_noise is None
                      else _require_cuda_f32(sigma_noise, 'sigma_noise').reshape(n, p, 1))
                _lib.check(_lib.lib().tpr_add_density_noise(_ptr(sigma), _ptr(nz), n * p, dn, _stream()), 'tpr_add_density_noise')
        aux = dict(packed=pp, dec=dec, xyz=xyz) if train else None
        return {'rgb': rgb, 'sigma': sigma}, aux

    # ------------------------------------------------------------------ sort_samples / unify_samples (VR/renderer.py:150-167)
    def sort_samples(self, all_depths, all_colors, all_densities):
        """[N,M,S,1], [N,M,S,C], [N,M,S,1] -> the same three tensors with every ray's samples ordered by depth.  forward()
        never calls this (the sort happens per ray inside the fused kernel); the reference has no caller for it either."""
        d = _require_cuda_f32(all_depths, 'all_depths')
        c = _require_cuda_f32(all_colors, 'all_colors')
        s = _require_cuda_f32(all_densities, 'all_densities')
        _forbid_autograd(d, c, s)
        n, m, ns, ch = c.shape
        if tuple(d.shape) != (n, m, ns, 1) or tuple(s.shape) != (n, m, ns, 1):
            raise RuntimeError(f'depths / densities must be [{n},{m},{ns},1], got {tuple(d.shape)} / {tuple(s.shape)}')
        with torch.cuda.device(d.device):
            ds, cs, ss = torch.empty_like(d), torch.empty_like(c), torch.empty_like(s)
            _lib.check(_lib.lib().tpr_sort_samples(_ptr(d), _ptr(c), _ptr(s), n * m, ns, ch, _ptr(ds), _ptr(cs), _ptr(ss),
                                                   _stream()), 'tpr_sort_samples')
        return ds, cs, ss

    def unify_samples(self, depths1, colors1, densities1, depths2, colors2, densities2):
        """Concatenate the coarse and the importance samples of every ray and order them by depth (VR/renderer.py:157-167)."""
        return self.sort_samples(torch.cat([depths1, depths2], dim=-2), torch.cat([colors1, colors2], dim=-2),
                                 torch.cat([densities1, densities2], dim=-2))

    # ------------------------------------------------------------------ the remaining public helpers
    def sample_stratified(self, ray_origins, ray_start, ray_end, depth_resolution, disparity_space_sampling=False, *,
                          jitter=None):
        """Coarse depths [N,M,D,1] (VR/renderer.py:169-192); ``ray_start`` / ``ray_end`` are python floats or per-ray
        tensors [N,M,1].  forward() never calls this (the depths are produced inside the fused kernel by the same
        device function); it exists because it is part of the reference class.  ``jitter`` [N,M,D,1] overrides the
        ``torch.rand`` draw."""
        ray_origins = _require_cuda_f32(ray_origins, 'ray_origins', (3,))
        n, m, _ = ray_origins.shape
        dev, d = ray_origins.device, int(depth_resolution)
        per_ray = isinstance(ray_start, torch.Tensor)
        if per_ray != isinstance(ray_end, torch.Tensor):
            raise RuntimeError('ray_start and ray_end must both be floats or both be tensors')
        if disparity_space_sampling and per_ray:
            raise RuntimeError('disparity_space_sampling takes scalar ray limits (VR/renderer.py:174-181)')
        with torch.cuda.device(dev):
            if jitter is None:
                # the reference's rand_like, which for the per-ray branch fills a permuted [D,N,M,1] view (see _draw_noise)
                jitter = (torch.rand((d, n, m, 1), device=dev, dtype=torch.float32).permute(1, 2, 0, 3) if per_ray
                          else torch.rand((n, m, d, 1), device=dev, dtype=torch.float32))
            jitter = _require_cuda_f32(jitter, 'jitter').reshape(n, m, d, 1)
            rs = _require_cuda_f32(ray_start, 'ray_start').reshape(-1) if per_ray else None
            re = _require_cuda_f32(ray_end, 'ray_end').reshape(-1) if per_ray else None
            if per_ray and (rs.numel() != n * m or re.numel() != n * m):
                raise RuntimeError(f'per-ray limits must have {n * m} elements')
            o = _lib.TprOptions(ray_start=0.0 if per_ray else float(ray_start), ray_end=0.0 if per_ray else float(ray_end),
                                box_warp=1.0, depth_resolution=d, depth_resolution_importance=0,
                                disparity_space_sampling=int(bool(disparity_space_sampling)))
            out = torch.empty((n, m, d, 1), device=dev, dtype=torch.float32)
            _lib.check(_lib.lib().tpr_sample_stratified(_ptr(jitter), n * m, _ptr(rs), _ptr(re), ctypes.byref(o), _ptr(out),
                                                        _stream()), 'tpr_sample_stratified')
        return out

    def sample_importance(self, z_vals, weights, N_importance, *, u=None, return_inds=False):
        """z_vals [N,M,S,1], weights [N,M,S-1,1] -> [N,M,N_importance,1] (VR/renderer.py:194-212)."""
        z = _require_cuda_f32(z_vals, 'z_vals')
        w = _require_cuda_f32(weights, 'weights')
        n, m, s, _ = z.shape
        dev = z.device
        with torch.cuda.device(dev):
            if u is None:
                u = torch.rand(n * m, N_importance, device=dev)
            u = _require_cuda_f32(u, 'u')
            out = torch.empty((n, m, N_importance, 1), device=dev, dtype=torch.float32)
            inds = torch.empty((n * m, N_importance), device=dev, dtype=torch.int32)
            _lib.check(_lib.lib().tpr_sample_importance(_ptr(z), _ptr(w), _ptr(u), n * m, s, N_importance,
                                                        _ptr(out), _ptr(inds), _stream()), 'tpr_sample_importance')
        return (out, inds) if return_inds else out

    def sample_pdf(self, bins, weights, N_importance, det=False, eps=1e-5, *, u=None, return_inds=False):
        """bins [R,B+2], weights [R,B] -> samples [R,N_importance] (VR/renderer.py:214-253)."""
        if eps != 1e-5:
            raise NotImplementedError('sample_pdf: only the reference default eps=1e-5 is supported')
        bins = _require_cuda_f32(bins, 'bins')
        w = _require_cuda_f32(weights, 'weights')
        r, nb = w.shape
        dev = w.device
        with torch.cuda.device(dev):
            if u is None:
                u = (torch.linspace(0, 1, N_importance, device=dev).expand(r, N_importance) if det
                     else torch.rand(r, N_importance, device=dev))
            u = _require_cuda_f32(u, 'u')
            out = torch.empty((r, N_importance), device=dev, dtype=torch.float32)
            inds = torch.empty((r, N_importance), device=dev, dtype=torch.int32)
            _lib.check(_lib.lib().tpr_sample_pdf(_ptr(bins), bins.shape[1], _ptr(w), _ptr(u), r, nb, N_importance,
                                                 _ptr(out), _ptr(inds), _stream()), 'tpr_sample_pdf')
        return (out, inds) if return_inds else out
