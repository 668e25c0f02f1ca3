"""Autograd for ImportanceRenderer.forward and run_model: gradients w.r.t. the tri-planes and the OSGDecoder's four tensors.

The reference gets its backward from PyTorch autograd over ~40 ATen ops and ~10 GB of saved activations per forward at
FFHQ training shape (SURVEY.md section 3.2); training back-propagates through the renderer at
training/training_loop.py:335,377.  Here the forward is the fused kernel (nothing per-sample is saved) and the backward is
``tpr_render_backward`` (csrc/tpr_backward.cu): it re-evaluates colours / densities at the forward's sample depths and
runs the march, the decoder and the bilinear gather backwards.  Saved between the two: the packed planes, the packed
decoder, the rays, the S sample depths per ray, the depth range and -- written by the forward kernel's composite on its
way -- the 32 colours and sigma of every sample (132 B per sample; eager autograd keeps ~800 B per sample).

Frame-batched renders (F*P cameras over P plane sets, camera n sampling set n % P: ``TprOptions.plane_sets``, what
frames.render_frames passes) differentiate as one call: the backward reads and scatters set n % P, so every plane set
receives the sum of its F cameras' gradients in one [P,3,H,W,32] buffer.  With ``depth_clamp_group`` = k the depth of a
camera was clamped to the range of its own group of k cameras; the forward keeps those ranges only in its scratch, so they
are re-derived here as the min and max of each group's coarse and importance depths -- the values the forward reduced.
``output_layout='channels_first'``: the rgb returned is the [N,M,32] view of [N,32,M] memory; its upstream gradient is
copied once into the [N,M,32] rows the kernels read.

The graph is the reference's: importance depths are constants (VR/renderer.py:198,210: no_grad + detach), so is the
jitter; ray origins / directions are not differentiated (they raise if they require grad).

Under ``torch.use_deterministic_algorithms(True)`` both backward functions run the library's deterministic backward
(TPR_BWD_DETERMINISTIC): bit-identical gradients for equal inputs on the same GPU model, and a plane gradient that does not
depend on the order of the samples.  The forward is deterministic in either mode.
"""
import ctypes

import torch

from .. import _lib
from . import renderer as _r


class _Render(torch.autograd.Function):
    @staticmethod
    def forward(ctx, renderer, decoder, options, noise, planes, w1, b1, w2, b2, origins, dirs):
        with torch.no_grad():
            rgb, depth, wsum, aux = renderer._forward_impl(planes.detach(), decoder, origins, dirs, options, noise=noise,
                                                           train=True)
        fc1, fc2 = decoder.net[0], decoder.net[2]
        ctx.gains = (float(fc1.weight_gain), float(fc1.bias_gain), float(fc2.weight_gain), float(fc2.bias_gain))
        ctx.packed, ctx.opts = aux['packed'], aux['options']
        ctx.shape = tuple(origins.shape[:2])
        fine = aux['fine'] if aux['fine'] is not None else torch.empty(0, device=rgb.device)
        ctx.has_fine = aux['fine'] is not None
        ctx.has_saved = aux['saved'] is not None
        s_col, s_sig, s_feat = aux['saved'] if ctx.has_saved else (None, None, None)
        ctx.has_feat = s_feat is not None
        empty = torch.empty(0, device=rgb.device)
        rng = _group_ranges(aux['coarse'], aux['fine'], ctx.shape[0], aux['options'].depth_clamp_group, aux['range'])
        ctx.save_for_backward(aux['packed'].data, aux['dec'], origins.contiguous(), dirs.contiguous(), aux['coarse'], fine,
                              rng, s_col if ctx.has_saved else empty, s_sig if ctx.has_saved else empty,
                              s_feat if ctx.has_feat else empty)
        return rgb, depth, wsum

    @staticmethod
    @torch.autograd.function.once_differentiable          # raw CUDA kernels: a double backward must raise, not detach silently
    def backward(ctx, g_rgb, g_depth, g_wsum):
        packed, dec, origins, dirs, coarse, fine, rng, s_col, s_sig, s_feat = ctx.saved_tensors
        n, m = ctx.shape
        pp, o = ctx.packed, ctx.opts
        dev = packed.device
        L = _lib.lib()
        p, st = _r._ptr, _r._stream
        zeros = lambda shape: torch.zeros(shape, device=dev, dtype=torch.float32)
        # (channels-first output: g_rgb usually arrives with the output's [N,32,M] strides; contiguous() is then one copy)
        g_rgb = g_rgb.contiguous().float() if g_rgb is not None else zeros((n, m, 32))
        g_depth = g_depth.contiguous().float() if g_depth is not None else zeros((n, m, 1))
        g_wsum = g_wsum.contiguous().float() if g_wsum is not None else zeros((n, m, 1))
        need = ctx.needs_input_grad
        want_planes, want_dec = need[4], any(need[5:9])
        with torch.cuda.device(dev):
            g_planes = torch.empty_like(packed) if want_planes else None
            g_dec = torch.empty_like(dec) if want_dec else None
            nbytes = L.tpr_render_backward_scratch_bytes(n, m, o.depth_resolution + o.depth_resolution_importance)
            o2 = _lib.TprOptions.from_buffer_copy(o)           # plane_sets / depth_clamp_group as the forward had them
            if torch.are_deterministic_algorithms_enabled():
                o2.flags |= _lib.BWD_DETERMINISTIC
                # the fixed-point accumulator holds the P plane sets, not the N cameras
                nbytes += L.tpr_backward_deterministic_scratch_bytes(pp.n_img, pp.height, pp.width)
            scratch = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            _lib.check(L.tpr_render_backward(p(packed), n, pp.height, pp.width, p(dec), p(origins), p(dirs), m, p(coarse),
                                             p(fine) if ctx.has_fine else None, p(rng), ctypes.byref(o2), p(g_rgb), p(g_depth),
                                             p(g_wsum), p(s_col) if ctx.has_saved else None, p(s_sig) if ctx.has_saved else None,
                                             p(s_feat) if ctx.has_feat else None,
                                             p(g_planes), p(g_dec), p(scratch), nbytes, st()),
                       'tpr_render_backward')
            g_nchw, g_w1, g_b1, g_w2, g_b2 = _unpack_grads(g_planes, g_dec, ctx.gains, pp, dev)
        return (None, None, None, None, g_nchw,
                g_w1 if need[5] else None, g_b1 if need[6] else None, g_w2 if need[7] else None, g_b2 if need[8] else None,
                None, None)


def _group_ranges(coarse, fine, n, k, rng):
    """The depth-clamp ranges the forward used: ``rng`` [2] (its call-wide range) for k == 0, else [2*ceil(n/k)] = the (min,
    max) of the coarse and importance depths of cameras [j k, j k + k) -- the reduction the forward made over the same
    values, so the result is bit-equal to the ranges it clamped with."""
    if k <= 0:
        return rng
    c = coarse.reshape(n, -1)
    lo, hi = c.amin(1), c.amax(1)
    if fine is not None and fine.numel():                           # (min / max commute: no concatenated copy)
        f = fine.reshape(n, -1)
        lo, hi = torch.minimum(lo, f.amin(1)), torch.maximum(hi, f.amax(1))
    g = -(-n // k)
    pad = g * k - n                                                  # a shorter last group
    lo = torch.nn.functional.pad(lo, (0, pad), value=float('inf')).view(g, k).amin(1)
    hi = torch.nn.functional.pad(hi, (0, pad), value=float('-inf')).view(g, k).amax(1)
    return torch.stack([lo, hi], 1).reshape(-1).contiguous()


def _unpack_grads(g_planes, g_dec, gains, pp, dev):
    """Packed gradients (either may be None) -> (planes [N,3,32,H,W], w1, b1, w2, b2) of the module's raw tensors."""
    L, p, st = _lib.lib(), _r._ptr, _r._stream
    g_w1 = g_b1 = g_w2 = g_b2 = None
    if g_dec is not None:
        g_w1 = torch.empty((64, 32), device=dev, dtype=torch.float32)
        g_b1 = torch.empty(64, device=dev, dtype=torch.float32)
        g_w2 = torch.empty((33, 64), device=dev, dtype=torch.float32)
        g_b2 = torch.empty(33, device=dev, dtype=torch.float32)
        _lib.check(L.tpr_unpack_decoder_grad(p(g_dec), *gains, p(g_w1), p(g_b1), p(g_w2), p(g_b2), st()),
                   'tpr_unpack_decoder_grad')
    g_nchw = None
    if g_planes is not None:
        # the plane gradient was scattered in the packed layout [N,3,H,W,32]; the backbone wants [N,3,32,H,W] contiguous
        # (autograd would otherwise make that copy itself, strided: 0.22 ms vs 0.08 ms for 201 MB at config 2)
        g_nchw = torch.empty((pp.n_img, 3, 32, pp.height, pp.width), device=dev, dtype=torch.float32)
        _lib.check(L.tpr_unpack_planes(p(g_planes), pp.n_img, pp.height, pp.width, p(g_nchw), st()), 'tpr_unpack_planes')
    return g_nchw, g_w1, g_b1, g_w2, g_b2


def render_with_grad(renderer, planes, decoder, ray_origins, ray_directions, options, noise=None):
    """ImportanceRenderer.forward with autograd: returns (rgb, depth, weight_sum) attached to ``planes`` and to the
    decoder's parameters.  Takes every forward option: frame batching (N = F*P cameras over P plane sets),
    ``depth_clamp_group`` and ``output_layout='channels_first'`` included."""
    if isinstance(planes, _r.PackedPlanes):
        raise NotImplementedError('autograd needs the planes tensor itself ([N,3,32,H,W]), not PackedPlanes')
    for t, name in ((ray_origins, 'ray_origins'), (ray_directions, 'ray_directions')):
        if isinstance(t, torch.Tensor) and t.requires_grad:
            raise NotImplementedError(f'{name} requires grad: the renderer differentiates w.r.t. planes and decoder only')
    _r.pack_decoder(decoder, allow_grad=True)            # validates the decoder's structure before anything is launched
    fc1, fc2 = decoder.net[0], decoder.net[2]
    return _Render.apply(renderer, decoder, options, noise, planes, fc1.weight, fc1.bias, fc2.weight, fc2.bias,
                         ray_origins, ray_directions)


class _RunModel(torch.autograd.Function):
    """ImportanceRenderer.run_model with autograd: the forward is the inference point query (same kernel, same outputs, the
    same density_noise draw); the backward is ``tpr_run_model_backward`` (the decoder backward kernels in their point-query
    mode: no march, no sort, the features gathered again).  Saved: the packed planes and decoder, the coordinates and rgb."""

    @staticmethod
    def forward(ctx, renderer, decoder, options, want_rgb, sigma_noise, xyz, planes, w1, b1, w2, b2):
        ctx.set_materialize_grads(False)           # an unused output hands in None: rgb unused = the sigma-only backward
        with torch.no_grad():
            out, aux = renderer._run_model_impl(planes.detach(), decoder, xyz, options, want_rgb=want_rgb,
                                                sigma_noise=sigma_noise, train=True)
        fc1, fc2 = decoder.net[0], decoder.net[2]
        ctx.gains = (float(fc1.weight_gain), float(fc1.bias_gain), float(fc2.weight_gain), float(fc2.bias_gain))
        ctx.packed, ctx.want_rgb = aux['packed'], want_rgb
        ctx.box_warp, ctx.flags = float(options['box_warp']), _r._mlp_flag(options)
        rgb, sigma = out['rgb'], out['sigma']
        ctx.save_for_backward(aux['packed'].data, aux['dec'], aux['xyz'],
                              rgb if want_rgb else torch.empty(0, device=sigma.device))
        return (rgb, sigma) if want_rgb else sigma

    @staticmethod
    @torch.autograd.function.once_differentiable          # raw CUDA kernels: a double backward must raise, not detach silently
    def backward(ctx, *grads):
        g_rgb, g_sigma = grads if ctx.want_rgb else (None, grads[0])
        need = ctx.needs_input_grad
        want_planes, want_dec = need[6], any(need[7:11])
        if (g_rgb is None and g_sigma is None) or not (want_planes or want_dec):
            return (None,) * 11
        packed, dec, xyz, rgb = ctx.saved_tensors
        pp, dev = ctx.packed, packed.device
        n, npts, _ = xyz.shape
        L, p, st = _lib.lib(), _r._ptr, _r._stream
        g_rgb = g_rgb.contiguous().float() if g_rgb is not None else None
        g_sigma = g_sigma.contiguous().float() if g_sigma is not None else None
        with torch.cuda.device(dev):
            g_planes = torch.empty_like(packed) if want_planes else None
            g_dec = torch.empty_like(dec) if want_dec else None
            nbytes = L.tpr_run_model_backward_scratch_bytes(n, npts)
            flags = ctx.flags
            if torch.are_deterministic_algorithms_enabled():
                flags |= _lib.BWD_DETERMINISTIC
                nbytes += L.tpr_backward_deterministic_scratch_bytes(n, pp.height, pp.width)
            scratch = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            _lib.check(L.tpr_run_model_backward(p(packed), n, pp.height, pp.width, p(dec), p(xyz), npts, ctx.box_warp,
                                                p(rgb) if g_rgb is not None else None, p(g_rgb), p(g_sigma), flags,
                                                p(g_planes), p(g_dec), p(scratch), nbytes, st()),
                       'tpr_run_model_backward')
            g_nchw, g_w1, g_b1, g_w2, g_b2 = _unpack_grads(g_planes, g_dec, ctx.gains, pp, dev)
        return (None, None, None, None, None, None, g_nchw,
                g_w1 if need[7] else None, g_b1 if need[8] else None, g_w2 if need[9] else None, g_b2 if need[10] else None)


def run_model_with_grad(renderer, planes, decoder, sample_coordinates, options, want_rgb=True, sigma_noise=None):
    """ImportanceRenderer.run_model with autograd: returns {'rgb', 'sigma'} attached to ``planes`` and to the decoder's
    parameters (TriPlaneGenerator.sample / sample_mixed under a training step, e.g. EG3D's density regulariser)."""
    if isinstance(planes, _r.PackedPlanes):
        raise NotImplementedError('autograd needs the planes tensor itself ([N,3,32,H,W]), not PackedPlanes')
    if isinstance(sample_coordinates, torch.Tensor) and sample_coordinates.requires_grad:
        raise NotImplementedError('sample_coordinates requires grad: the renderer differentiates w.r.t. planes and decoder only')
    _r.pack_decoder(decoder, allow_grad=True)            # validates the decoder's structure before anything is launched
    fc1, fc2 = decoder.net[0], decoder.net[2]
    out = _RunModel.apply(renderer, decoder, options, bool(want_rgb), sigma_noise, sample_coordinates, planes, fc1.weight,
                          fc1.bias, fc2.weight, fc2.bias)
    rgb, sigma = out if want_rgb else (None, out)
    return {'rgb': rgb, 'sigma': sigma}
