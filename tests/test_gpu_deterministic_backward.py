"""GPU: the deterministic backward.  Under torch.use_deterministic_algorithms(True) both autograd functions (the render's and
run_model's) accumulate the plane gradient in 64-bit fixed point and the decoder gradient as per-CTA rows summed in a fixed
order: equal inputs give bit-identical gradients, the plane gradient does not depend on the order of the points, and scaling
the upstream gradient by a power of two scales every gradient exactly.  Accuracy is held to the gates of the default mode.
The oracles run with the mode off: torch's grid_sample backward refuses to run in it."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import triplane_oracle as O
from tests.cases import load_bwd_case
from tests.test_gpu_backward import run_backward, rel_err as rel_np
from tests.test_gpu_parity import T, make_decoder, dev
from tests.test_gpu_run_model_backward import SHAPES, VARIANTS, synthetic, weights, ours, oracle, check, rel_err

pytestmark = pytest.mark.gpu
REL = 2e-4
NAMES = ('planes', 'w1', 'b1', 'w2', 'b2')


@contextlib.contextmanager
def deterministic(on):
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


@pytest.fixture(autouse=True)
def det_mode():
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    with deterministic(True):
        yield
    torch.backends.cuda.matmul.allow_tf32 = tf32


def assert_equal(a, b):
    for k, x, y in zip(NAMES, a, b):
        assert x is not None and y is not None and torch.equal(x, y), k


def render(pkg, name, keep_samples=True, scale=1.0):
    scene, opts, gold, (A, B, C) = load_bwd_case(name)
    outs, grads = run_backward(pkg, scene, opts, scale * A, scale * B, scale * C, keep_samples=keep_samples)
    return [o.detach() for o in outs], grads, gold


@pytest.mark.parametrize('impl', ['default', 'hmma'])
@pytest.mark.parametrize('keep_samples', [True, False])
@pytest.mark.parametrize('name', ['bwd_ffhq', 'bwd_white'])
def test_render_is_repeatable(pkg, monkeypatch, name, keep_samples, impl):
    if impl == 'hmma':
        monkeypatch.setenv('TPR_BWD_IMPL', 'hmma')
    outs0, g0, _ = render(pkg, name, keep_samples)
    for _ in range(2):
        outs, g, _ = render(pkg, name, keep_samples)
        for a, b in zip(outs0, outs):
            assert torch.equal(a, b)
        assert_equal(g0, g)


@pytest.mark.parametrize('name', ['bwd_ffhq', 'bwd_white', 'bwd_coarse'])
def test_render_accuracy(pkg, name):
    """Against the reference's gradient fixtures (the default mode's gate) and against the default mode."""
    _, g_det, gold = render(pkg, name)
    with deterministic(False):
        _, g_def, _ = render(pkg, name)
    for g, gd, k in zip(g_det, g_def, ('g_planes', 'g_w1', 'g_b1', 'g_w2', 'g_b2')):
        assert torch.isfinite(g).all(), k
        assert rel_np(g.cpu().numpy(), gold[k]) < REL, k
        assert rel_err(g, gd) < 5e-5, k


@pytest.mark.parametrize('variant', VARIANTS)
@pytest.mark.parametrize('n_img,n_pts', SHAPES)
def test_run_model_repeatable_and_accurate(pkg, n_img, n_pts, variant):
    scene, pts = synthetic(n_img, n_pts)
    A, B = weights(n_img, n_pts)
    opts = dict(O.FFHQ_OPTIONS)
    _, g0 = ours(pkg, scene, pts, opts, A, B, variant)
    _, g1 = ours(pkg, scene, pts, opts, A, B, variant)
    assert_equal(g0, g1)
    with deterministic(False):
        _, g_o = oracle(scene, pts, opts['box_warp'], A, B, variant)
    check(g0, g_o)


@pytest.mark.parametrize('n_img,n_pts', [(2, 3000), (2, 100)])
def test_plane_gradient_does_not_depend_on_the_point_order(pkg, n_img, n_pts):
    """(2, 3000): the tcgen05 kernel; (2, 100): fewer than 128 points per image, the mma.sync kernel."""
    scene, pts = synthetic(n_img, n_pts)
    A, B = weights(n_img, n_pts)
    opts = dict(O.FFHQ_OPTIONS)
    perm = np.stack([np.random.default_rng(40 + i).permutation(n_pts) for i in range(n_img)])
    pts_p = np.take_along_axis(pts, perm[..., None], 1)
    idx = torch.from_numpy(perm).to(dev())
    A_p = torch.gather(A, 1, idx[..., None].expand(-1, -1, A.shape[-1]))
    B_p = torch.gather(B, 1, idx[..., None])
    for variant in ('rgb_sigma', 'sigma_only_query'):
        _, g = ours(pkg, scene, pts, opts, A, B, variant)
        _, g_p = ours(pkg, scene, pts_p, opts, A_p, B_p, variant)
        assert torch.equal(g[0], g_p[0]), variant
        for a, b in zip(g[1:], g_p[1:]):
            assert rel_err(b, a) < 1e-5, variant


def test_exact_scaling_with_the_upstream_gradient(pkg):
    scene, pts = synthetic(2, 1000)
    A, B = weights(2, 1000)
    opts = dict(O.FFHQ_OPTIONS)
    _, g1 = ours(pkg, scene, pts, opts, A, B)
    _, r1, _ = render(pkg, 'bwd_ffhq')
    for f in (2.0 ** -20, 2.0, 2.0 ** 20):
        _, gk = ours(pkg, scene, pts, opts, f * A, f * B)
        assert_equal([f * t for t in g1], gk)
        _, rk, _ = render(pkg, 'bwd_ffhq', scale=f)
        assert_equal([f * t for t in r1], rk)


def test_config5_grid(pkg):
    """A 256^3 sigma-only query on one image (the largest point count per image: the fixed point's coarsest resolution)."""
    g = 256
    scene = O.synthetic_scene(95, 1, 4, 256, 8, 8, 0.5)
    ax = (torch.arange(g, device=dev(), dtype=torch.float32) + 0.5) / g - 0.5
    zz, yy, xx = torch.meshgrid(ax, ax, ax, indexing='ij')
    xyz = torch.stack([xx, yy, zz], -1).reshape(1, -1, 3).contiguous()
    del zz, yy, xx
    B = torch.randn((1, g ** 3, 1), device=dev(), generator=torch.Generator(device=dev()).manual_seed(9))
    opts = dict(O.FFHQ_OPTIONS)

    def run():
        dec = make_decoder(pkg, scene['dec']).requires_grad_(True)
        planes = T(scene['planes']).requires_grad_(True)
        s = pkg.ImportanceRenderer().run_model(planes, dec, xyz, None, opts, want_rgb=False)['sigma']
        (s * B).sum().backward()
        return (planes.grad, dec.net[0].weight.grad, dec.net[0].bias.grad, dec.net[2].weight.grad, dec.net[2].bias.grad)

    g0, g1 = run(), run()
    assert_equal(g0, g1)
    with deterministic(False):
        g_def = run()
    for k, a, b in zip(NAMES, g0, g_def):
        if k == 'b2':          # only its sigma entry is reached; the colour entries are exact zeros in both modes
            assert torch.equal(a[1:], b[1:]) and rel_err(a[:1], b[:1]) < 5e-5
        else:
            assert rel_err(a, b) < 5e-5, k


def test_edge_inputs(pkg):
    scene, pts = synthetic(2, 1000)
    A, B = weights(2, 1000)
    opts = dict(O.FFHQ_OPTIONS)
    B_nan = B.clone()
    B_nan[1, 17, 0] = float('nan')
    _, g = ours(pkg, scene, pts, opts, A, B_nan)
    torch.cuda.synchronize()
    assert not torch.isfinite(g[0]).all()
    _, g = ours(pkg, scene, pts, opts, torch.zeros_like(A), torch.zeros_like(B))
    for k, t in zip(NAMES, g):
        assert torch.equal(t, torch.zeros_like(t)), k
