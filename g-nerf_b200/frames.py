"""Many frames of one set of tri-planes in ONE renderer call, and a backbone/plane cache for callers that re-render the
same latents -- SURVEY.md section 8(f) rows 1 and 4, the callers either side of ImportanceRenderer.forward.

The reference's video loop (gen_videos.py:153-171) calls ``G.synthesis(ws, c_d, noise_mode='const', ...)`` once per frame
with the SAME ``ws``: every frame re-runs the StyleGAN2 backbone, re-derives the same planes and renders a batch of
P identities x 64^2 rays -- 0.4 M ray-samples, far too little to fill a B200.  Here the planes are produced and repacked
once and F frames x P identities are rendered as one batch: camera n = f * P + p samples plane set n % P
(``TprOptions.plane_sets``) and clamps its depth against the range of its own frame (``TprOptions.depth_clamp_group``
= P, what VR/ray_marcher.py:50 computes inside one reference forward).  The two uniform draws are made frame by frame
with the reference's calls (VR/renderer.py:190,237), so the result is the one the frame loop would have produced from the
same generator state.
"""
import torch

from .volumetric_rendering import renderer as _r
from .volumetric_rendering.ray_sampler import RaySampler


def draw_frame_noise(n_frames, batch, n_rays, dc, df, device, density_noise=0.0):
    """jitter [F*P,M,Dc,1] and u [F*P*M,Df] drawn frame by frame in the reference's order: rand[P,M,Dc,1] then rand[P*M,Df]
    per forward (VR/renderer.py:190,237), straight into the frame's slice of the batch buffers.  With density_noise > 0 a
    forward also draws randn[P,M*Dc,1] after the jitter and randn[P,M*Df,1] after u (VR/renderer.py:146); the tuple then has
    those two tensors ([F*P,M*Dc,1], [F*P,M*Df,1]) as well."""
    jitter = torch.empty((n_frames * batch, n_rays, dc, 1), device=device, dtype=torch.float32)
    u = torch.empty((n_frames * batch * n_rays, df), device=device, dtype=torch.float32) if df > 0 else None
    dn = density_noise > 0
    nz_c = torch.empty((n_frames * batch, n_rays * dc, 1), device=device, dtype=torch.float32) if dn else None
    nz_f = torch.empty((n_frames * batch, n_rays * df, 1), device=device, dtype=torch.float32) if dn and df > 0 else None
    for f in range(n_frames):
        torch.rand((batch, n_rays, dc, 1), device=device, dtype=torch.float32, out=jitter[f * batch:(f + 1) * batch])
        if dn:
            torch.randn((batch, n_rays * dc, 1), device=device, dtype=torch.float32, out=nz_c[f * batch:(f + 1) * batch])
        if df > 0:
            torch.rand(batch * n_rays, df, device=device, out=u[f * batch * n_rays:(f + 1) * batch * n_rays])
            if dn:
                torch.randn((batch, n_rays * df, 1), device=device, dtype=torch.float32, out=nz_f[f * batch:(f + 1) * batch])
    return (jitter, u, nz_c, nz_f) if dn else (jitter, u)


def render_frames(renderer, planes, decoder, cam2world, intrinsics, resolution, rendering_options, *,
                  ray_sampler=None, frames_per_call=None, noise=None):
    """Render F frames of P identities.

    planes      [P,3,32,H,W] (or PackedPlanes): one plane set per identity, as the backbone emits them
    cam2world   [F,4,4] (the same camera for every identity, as in gen_videos.py:166) or [F,P,4,4]
    intrinsics  [3,3], [F,3,3] or [F,P,3,3]
    noise       optional (jitter [F*P,M,Dc,1], u [F*P*M,Df]); default: drawn per frame like the reference's frame loop

    Returns the neural-rendered images exactly as TriPlaneGenerator.synthesis shapes them (training/triplane.py:81-82):
    ``feature_image`` [F,P,32,res,res], ``depth_image`` [F,P,1,res,res], ``weights_image`` [F,P,1,res,res]; the feature
    image is written channels-first by the kernel (no permute + contiguous pass).

    Under autograd (``planes`` or the decoder's parameters require grad) the three images are attached to them: each chunk
    of ``frames_per_call`` frames is one differentiable forward over the planes tensor (one autograd node; the backward
    scatters every frame's gradient into the P plane sets at once), and the images are views of its outputs (one chunk) or
    their concatenation.  Same noise draws and outputs as without autograd.
    """
    grad = torch.is_grad_enabled() and _r._wants_grad(planes, decoder)
    if grad and isinstance(planes, torch.Tensor):
        # the forward repacks the tensor itself (render_with_grad); PackedPlanes keep the inference path, which refuses them
        src, P, dev = planes, planes.shape[0], planes.device
    else:
        src = renderer._packed(planes) if hasattr(renderer, '_packed') else _r.pack_planes(planes)
        P, dev = src.n_img, src.device
    cam2world = torch.as_tensor(cam2world, dtype=torch.float32, device=dev)
    intrinsics = torch.as_tensor(intrinsics, dtype=torch.float32, device=dev)
    if cam2world.dim() == 3:
        cam2world = cam2world[:, None].expand(-1, P, -1, -1)
    F = cam2world.shape[0]
    if tuple(cam2world.shape) != (F, P, 4, 4):
        raise RuntimeError(f'cam2world must be [F,4,4] or [F,{P},4,4], got {tuple(cam2world.shape)}')
    if intrinsics.dim() == 2:
        intrinsics = intrinsics[None, None].expand(F, P, -1, -1)
    elif intrinsics.dim() == 3:
        intrinsics = intrinsics[:, None].expand(-1, P, -1, -1)
    if tuple(intrinsics.shape) != (F, P, 3, 3):
        raise RuntimeError(f'intrinsics must be [3,3], [F,3,3] or [F,{P},3,3], got {tuple(intrinsics.shape)}')
    sampler = ray_sampler if ray_sampler is not None else RaySampler()
    res = int(resolution)
    m = res * res
    dc, df = int(rendering_options['depth_resolution']), int(rendering_options['depth_resolution_importance'])
    opts = dict(rendering_options, output_layout='channels_first', depth_clamp_group=P)
    if not grad:
        feat = torch.empty((F, P, 32, res, res), device=dev, dtype=torch.float32)
        depth = torch.empty((F, P, 1, res, res), device=dev, dtype=torch.float32)
        wsum = torch.empty((F, P, 1, res, res), device=dev, dtype=torch.float32)
    chunks = []
    step = F if not frames_per_call else max(1, int(frames_per_call))
    with torch.cuda.device(dev):
        if noise is None:
            noise = draw_frame_noise(F, P, m, dc, df, dev, float(rendering_options.get('density_noise', 0) or 0))
        jitter, u = noise[0], noise[1]
        for f0 in range(0, F, step):
            f1 = min(F, f0 + step)
            n = (f1 - f0) * P
            o, d = sampler(cam2world[f0:f1].reshape(n, 4, 4).contiguous(), intrinsics[f0:f1].reshape(n, 3, 3).contiguous(), res)
            nz = (jitter[f0 * P:f1 * P], u[f0 * P * m:f1 * P * m] if u is not None else None)
            if len(noise) == 4:
                nz = nz + (noise[2][f0 * P:f1 * P], noise[3][f0 * P:f1 * P] if noise[3] is not None else None)
            if grad:
                # rgb is the [n,M,32] view of [n,32,M] memory (channels_first): the [f,P,32,res,res] image is a free view
                rgb, dep, ws = _r.ImportanceRenderer.forward(renderer, src, decoder, o, d, opts, noise=nz)
                f = f1 - f0
                chunks.append((rgb.permute(0, 2, 1).view(f, P, 32, res, res), dep.view(f, P, 1, res, res),
                               ws.view(f, P, 1, res, res)))
                continue
            out = (feat[f0:f1].view(n, 32, m).permute(0, 2, 1), depth[f0:f1].view(n, m, 1), wsum[f0:f1].view(n, m, 1))
            _r.ImportanceRenderer.forward(renderer, src, decoder, o, d, opts, noise=nz, out=out)
    if grad:
        feat, depth, wsum = chunks[0] if len(chunks) == 1 else (torch.cat(t, 0) for t in zip(*chunks))
    return {'feature_image': feat, 'depth_image': depth, 'weights_image': wsum}


# ----------------------------------------------------------------------------------------------------------------
# plane cache for an UNMODIFIED caller (gen_videos.py keeps calling G.synthesis(ws, c_d, noise_mode='const') per frame)
# ----------------------------------------------------------------------------------------------------------------
class _BackboneMemo:
    """Stands in for ``G.backbone.synthesis.forward``: while the caller passes the same, unmodified ``ws`` tensor and the same keyword
    arguments with a deterministic noise mode, the planes of the previous call are returned instead of re-running the
    StyleGAN2 backbone (the reference has the same switch, ``cache_backbone`` / ``use_cached_backbone`` at
    training/triplane.py:53,66-71, but gen_videos.py never sets it).  The memo holds a reference to ``ws``, so a hit on
    (address, shape, version counter) cannot be a recycled allocation."""

    def __init__(self, fn):
        self.fn, self.key, self.ws, self.planes = fn, None, None, None
        self.hits = self.misses = 0

    def __call__(self, ws, **kwargs):
        cacheable = (kwargs.get('noise_mode', 'random') in ('const', 'none') and not kwargs.get('update_emas', False)
                     and not (torch.is_grad_enabled() and ws.requires_grad))
        if not cacheable:
            return self.fn(ws, **kwargs)
        key = (ws.data_ptr(), tuple(ws.shape), ws._version, ws.device, tuple(sorted((k, repr(v)) for k, v in kwargs.items())))
        if key == self.key:
            self.hits += 1
            return self.planes
        self.misses += 1
        planes = self.fn(ws, **kwargs)
        self.key, self.ws, self.planes = key, ws, planes
        return planes


def enable_plane_cache(G):
    """Turn on backbone + repack caching on a TriPlaneGenerator instance (fresh or unpickled).  Returns the memo (its
    ``hits`` / ``misses`` counters say what happened)."""
    net = G.backbone.synthesis                      # the SynthesisNetwork module (training/networks_stylegan2.py:461)
    memo = net.__dict__.get('_tpr_memo')
    if memo is None:
        memo = _BackboneMemo(net.forward)           # the bound original
        # instance attributes: the class (possibly re-exec'd from a pickle), its parameters and state_dict stay untouched
        net.__dict__['forward'] = memo
        net.__dict__['_tpr_memo'] = memo
    G.renderer.cache_packed_planes = True
    return memo


def disable_plane_cache(G):
    net = G.backbone.synthesis
    if net.__dict__.pop('_tpr_memo', None) is not None:
        net.__dict__.pop('forward', None)
    G.renderer.cache_packed_planes = False
    G.renderer._plane_cache = None


def synthesize_frames(G, ws, cam2world, intrinsics, neural_rendering_resolution=None, *, frames_per_call=None,
                      superresolution=True, update_emas=False, **synthesis_kwargs):
    """The frame loop of gen_videos.py:153-171 for a reference TriPlaneGenerator ``G`` with the renderer batched:
    backbone once (training/triplane.py:69), all frames through render_frames, then -- still the reference's own code,
    frame by frame -- the super-resolution head (training/triplane.py:86-87).  Returns lists of per-frame dicts with the
    keys ``synthesis`` returns."""
    res = G.neural_rendering_resolution if neural_rendering_resolution is None else neural_rendering_resolution
    G.neural_rendering_resolution = res
    planes = G.backbone.synthesis(ws, update_emas=update_emas, **synthesis_kwargs)      # the call of training/triplane.py:69
    planes = planes.view(len(planes), 3, 32, planes.shape[-2], planes.shape[-1])
    r = render_frames(G.renderer, planes, G.decoder, cam2world, intrinsics, res, G.rendering_kwargs,
                      ray_sampler=G.ray_sampler, frames_per_call=frames_per_call)
    frames = []
    sr_kwargs = {k: v for k, v in synthesis_kwargs.items() if k != 'noise_mode'}
    for f in range(r['feature_image'].shape[0]):
        feature_image, depth_image = r['feature_image'][f], r['depth_image'][f]
        if superresolution:
            rgb_image = feature_image[:, :3]
            sr_image, rgb_image = G.superresolution(rgb_image, feature_image, ws,
                                                    noise_mode=G.rendering_kwargs['superresolution_noise_mode'], **sr_kwargs)
            frames.append({'image': sr_image, 'image_raw': rgb_image, 'image_depth': depth_image})
        else:
            frames.append({'image_raw': feature_image[:, :3], 'image_depth': depth_image})
    return frames
