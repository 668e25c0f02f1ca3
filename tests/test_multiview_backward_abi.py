"""CPU: the argument checks of tpr_render_backward for frame-batched calls (plane_sets, depth_clamp_group), all reported before
any device is touched, and the refusals of the autograd path that remain."""
import ctypes

import pytest
import torch

DET = 0x100


def _call(pkg, n, plane_sets, clamp, scratch_bytes, flags=0, m=16, h=8, w=8):
    lib = pkg._lib.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    o = pkg._lib.TprOptions(ray_start=2.25, ray_end=3.3, box_warp=1.0, depth_resolution=8, depth_resolution_importance=8,
                            flags=flags, plane_sets=plane_sets, depth_clamp_group=clamp)
    return lib.tpr_render_backward(p, n, h, w, p, p, p, m, p, p, p, ctypes.byref(o), p, p, p, None, None, None, p, p, p,
                                   scratch_bytes, None)


def test_plane_sets_must_divide_the_cameras(pkg):
    lib = pkg._lib.lib()
    big = lib.tpr_render_backward_scratch_bytes(6, 16, 16) + lib.tpr_backward_deterministic_scratch_bytes(6, 8, 8)
    assert _call(pkg, 6, 4, 0, big) == -2 and b'multiple of plane_sets' in lib.tpr_last_error()
    assert _call(pkg, 6, -1, 0, big) == -2
    assert _call(pkg, 6, 7, 0, big) == -2


def test_negative_clamp_group_is_refused(pkg):
    lib = pkg._lib.lib()
    big = lib.tpr_render_backward_scratch_bytes(6, 16, 16)
    assert _call(pkg, 6, 3, -1, big) == -3 and b'depth_clamp_group < 0' in lib.tpr_last_error()


def test_deterministic_scratch_counts_plane_sets(pkg):
    """With plane_sets = P the deterministic accumulator holds P sets: scratch for P passes, one byte less fails."""
    lib = pkg._lib.lib()
    base = lib.tpr_render_backward_scratch_bytes(6, 16, 16)
    extra = lib.tpr_backward_deterministic_scratch_bytes(2, 8, 8)
    assert extra < lib.tpr_backward_deterministic_scratch_bytes(6, 8, 8)
    assert _call(pkg, 6, 2, 2, base + extra - 1, DET) == -4 and b'scratch' in lib.tpr_last_error()
    assert _call(pkg, 6, 2, 2, base, DET) == -4


def test_remaining_autograd_refusals(pkg):
    """PackedPlanes, out= and rays that require grad stay refused under autograd, with the messages they had (checked before
    any kernel runs, so CPU tensors suffice where the refusal comes first)."""
    from importlib import import_module
    bw = import_module('g-nerf_b200.volumetric_rendering.backward')
    rr = import_module('g-nerf_b200.volumetric_rendering.renderer')
    R = pkg.ImportanceRenderer()
    dec = pkg.OSGDecoder(32, {'decoder_lr_mul': 1, 'decoder_output_dim': 32})
    pp = rr.PackedPlanes(torch.zeros(1), 1, 8, 8)
    rays = torch.zeros(2, 4, 3)
    with pytest.raises(NotImplementedError, match='not PackedPlanes'):
        bw.render_with_grad(R, pp, dec, rays, rays, {})
    with pytest.raises(NotImplementedError, match='ray_origins requires grad'):
        bw.render_with_grad(R, torch.zeros(1, 3, 32, 8, 8), dec, rays.clone().requires_grad_(True), rays, {})
    with pytest.raises(NotImplementedError, match='inference-only'):
        R(torch.zeros(1, 3, 32, 8, 8, requires_grad=True), dec, rays, rays, {}, out=(None, None, None))


def test_clamp_groups_need_fewer_than_2_32_rays(pkg):
    """The per-group march reads the group of a ray with 32-bit arithmetic: a call that has 2^32 rays or more (far beyond
    any device's memory for the backward's scratch) is refused up front rather than indexed wrongly."""
    lib = pkg._lib.lib()
    assert _call(pkg, 1 << 16, 1, 4, 1 << 40, m=1 << 16) == -2 and b'2^32' in lib.tpr_last_error()
