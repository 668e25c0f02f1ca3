"""GPU: autograd through ImportanceRenderer.run_model (TriPlaneGenerator.sample / sample_mixed, training/triplane.py:92-104):
plane and decoder gradients of point queries (tpr_run_model_backward), against same-device autograd through the torch
restatement TO.decode(TO.gather(...)) -- pinned bit-equal to the reference's run_model fixtures on CPU
(tests/test_torch_oracle.py), so this is autograd through the reference's own ATen ops -- with TF32 off.
Loss: sum(rgb * A) + sum(sigma * B).  Gate: 2e-4 of the largest entry of each of the five gradients (the render backward's)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import triplane_oracle as O
from oracle import torch_oracle as TO
from tests.cases import SCALAR_CASES, load_case
from tests.test_gpu_parity import T, make_decoder, dev

pytestmark = pytest.mark.gpu
REL = 2e-4
NAMES = ('planes', 'w1', 'b1', 'w2', 'b2')
# (n_img, points per image): the regulariser's 1000 + 1000 perturbed points, tiles that straddle images, above the
# 65 536-point threshold of the tcgen05 forward with a partial last tile, fewer than 128 points per image (mma.sync fall-back)
SHAPES = [(1, 2000), (4, 2000), (3, 1000), (2, 148 * 128 * 3 + 77), (1, 127), (2, 100)]
# which upstream gradients reach run_model: rgb + sigma; sigma of a want_rgb=False query; sigma only of a full query (g_rgb is
# None); rgb only (g_sigma is None)
VARIANTS = ['rgb_sigma', 'sigma_only_query', 'sigma_loss', 'rgb_loss']


@pytest.fixture(autouse=True)
def no_tf32():
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = prev


def rel_err(got, want):
    got, want = got.detach().double(), want.detach().double()
    return float((got - want).abs().max() / max(float(want.abs().max()), 1e-12))


def synthetic(n_img, n_pts, seed=90):
    """A synthetic scene and points of which some lie outside the box (zero padding: no gradient from those taps)."""
    scene = O.synthetic_scene(seed, n_img, 4, 40, 8, 8, 0.5)
    pts = np.random.default_rng(n_pts + n_img).uniform(-0.6, 0.6, size=(n_img, n_pts, 3)).astype(np.float32)
    return scene, pts


def weights(n_img, n_pts, seed=0):
    g = torch.Generator().manual_seed(seed + n_pts)
    return torch.randn((n_img, n_pts, 32), generator=g).to(dev()), torch.randn((n_img, n_pts, 1), generator=g).to(dev())


def loss_of(out, A, B, variant):
    if variant in ('sigma_only_query', 'sigma_loss'):
        return (out['sigma'] * B).sum()
    if variant == 'rgb_loss':
        return (out['rgb'] * A).sum()
    return (out['rgb'] * A).sum() + (out['sigma'] * B).sum()


def ours(pkg, scene, pts, opts, A, B, variant='rgb_sigma', planes_grad=True, dec_grad=True):
    dec = make_decoder(pkg, scene['dec']).requires_grad_(dec_grad)
    planes = T(scene['planes']).requires_grad_(planes_grad)
    out = pkg.ImportanceRenderer().run_model(planes, dec, T(pts), None, opts, want_rgb=variant != 'sigma_only_query')
    loss_of(out, A, B, variant).backward()
    return out, (planes.grad, dec.net[0].weight.grad, dec.net[0].bias.grad, dec.net[2].weight.grad, dec.net[2].bias.grad)


def oracle(scene, pts, box_warp, A, B, variant='rgb_sigma'):
    planes = T(scene['planes']).requires_grad_(True)
    w1, b1, w2, b2, lr = TO.decoder_tuple(scene['dec'], dev())
    params = [t.requires_grad_(True) for t in (w1, b1, w2, b2)]
    rgb, sigma = TO.decode(TO.gather(planes, T(pts), box_warp), (*params, lr))
    grads = torch.autograd.grad(loss_of({'rgb': rgb, 'sigma': sigma}, A, B, variant), [planes] + params)
    return {'rgb': rgb.detach(), 'sigma': sigma.detach()}, grads


def check(grads, grads_o, gate=REL):
    errs = {}
    for k, g, go in zip(NAMES, grads, grads_o):
        assert g is not None and g.shape == go.shape and torch.isfinite(g).all(), k
        errs[k] = rel_err(g, go)
    print({k: f'{v:.1e}' for k, v in errs.items()})
    assert max(errs.values()) < gate, errs


@pytest.mark.parametrize('name', SCALAR_CASES)
def test_fixture_points_against_autograd(pkg, name):
    """The points of the reference's run_model fixtures, plus a few far outside the box (all twelve taps padded)."""
    scene, opts, gold = load_case(name)
    far = np.random.default_rng(1).uniform(0.6, 0.9, size=(gold['pts'].shape[0], 16, 3)).astype(np.float32)
    far *= np.sign(np.random.default_rng(2).standard_normal(far.shape)).astype(np.float32)
    pts = np.concatenate([gold['pts'], far], 1)
    A, B = weights(*pts.shape[:2])
    out, grads = ours(pkg, scene, pts, opts, A, B)
    out_o, grads_o = oracle(scene, pts, opts['box_warp'], A, B)
    assert float((out['rgb'].detach() - out_o['rgb']).abs().max()) < 1e-4
    check(grads, grads_o)


@pytest.mark.parametrize('variant', VARIANTS)
@pytest.mark.parametrize('n_img,n_pts', SHAPES)
def test_shapes_and_gradient_variants_against_autograd(pkg, n_img, n_pts, variant):
    scene, pts = synthetic(n_img, n_pts)
    A, B = weights(n_img, n_pts)
    opts = dict(O.FFHQ_OPTIONS)
    out, grads = ours(pkg, scene, pts, opts, A, B, variant)
    _, grads_o = oracle(scene, pts, opts['box_warp'], A, B, variant)
    assert (out['rgb'] is None) == (variant == 'sigma_only_query')
    check(grads, grads_o)
    if variant in ('sigma_only_query', 'sigma_loss'):
        assert float(grads[3][1:].abs().max()) == 0 and float(grads[4][1:].abs().max()) == 0     # colour rows of W2, b2
    if variant == 'rgb_loss':
        assert float(grads[3][0].abs().max()) == 0 and float(grads[4][0].abs().max()) == 0       # sigma row


@pytest.mark.parametrize('n_img', [1, 4])
def test_eg3d_density_regulariser(pkg, n_img):
    """EG3D's density regulariser written out: sigma of 1000 random points and of the same points perturbed by 0.004,
    L1 between the two halves x 0.25, backward -- against the same steps through the oracle."""
    scene = O.synthetic_scene(93, n_img, 4, 64, 8, 8, 0.5)
    opts = dict(O.FFHQ_OPTIONS)
    torch.manual_seed(11)
    c = torch.rand((n_img, 1000, 3), device=dev()) * 2 - 1
    c2 = c + torch.randn_like(c) * 0.004
    xyz = torch.cat([c, c2], 1)
    dec = make_decoder(pkg, scene['dec']).requires_grad_(True)
    planes = T(scene['planes']).requires_grad_(True)
    sigma = pkg.ImportanceRenderer().run_model(planes, dec, xyz, None, opts, want_rgb=False)['sigma']
    loss = F.l1_loss(sigma[:, :1000], sigma[:, 1000:]) * 0.25
    loss.backward()
    grads = (planes.grad, dec.net[0].weight.grad, dec.net[0].bias.grad, dec.net[2].weight.grad, dec.net[2].bias.grad)
    p_o = T(scene['planes']).requires_grad_(True)
    w1, b1, w2, b2, lr = TO.decoder_tuple(scene['dec'], dev())
    params = [t.requires_grad_(True) for t in (w1, b1, w2, b2)]
    _, s_o = TO.decode(TO.gather(p_o, xyz, opts['box_warp']), (*params, lr))
    assert float((sigma.detach() - s_o.detach()).abs().max()) < 1e-4
    # the L1 loss with the signs of the differences this forward produced: a pair whose two sigmas differ by less than the
    # forward's rounding could otherwise take the opposite sign in the oracle (points outside the box tie exactly in both)
    sign = torch.sign(sigma[:, :1000] - sigma[:, 1000:]).detach()
    loss_o = ((s_o[:, :1000] - s_o[:, 1000:]) * sign).sum() / sign.numel() * 0.25
    grads_o = torch.autograd.grad(loss_o, [p_o] + params)
    check(grads[:4], grads_o[:4])
    # b2: sigma moves with b2[0] alike at both points of a pair, so the gradient is exactly zero and both sides hold only the
    # rounding of a cancelling sum -- gated against the sum it cancels, sum |dL/dsigma|, instead of its own largest entry
    sum_abs_gsig = float(2 * sign.abs().sum()) / sign.numel() * 0.25
    assert float((grads[4] - grads_o[4]).abs().max()) < REL * sum_abs_gsig
    assert float(grads[0].abs().max()) > 0


def test_density_noise(pkg):
    """density_noise is additive: the gradients equal the noise-free call's, and the grad-mode call draws exactly what the
    no-grad call draws (the same randn in the same order)."""
    scene, pts = synthetic(2, 1000)
    A, B = weights(2, 1000)
    opts = dict(O.FFHQ_OPTIONS)
    noisy = dict(opts, density_noise=0.5)
    _, g_clean = ours(pkg, scene, pts, opts, A, B)
    torch.manual_seed(5)
    out_g, g_noisy = ours(pkg, scene, pts, noisy, A, B)
    state_grad = torch.cuda.get_rng_state()
    for a, b in zip(g_clean, g_noisy):
        assert rel_err(b, a) < 1e-5
    torch.manual_seed(5)
    with torch.no_grad():
        out_n = pkg.ImportanceRenderer().run_model(T(scene['planes']), make_decoder(pkg, scene['dec']), T(pts), None, noisy)
    assert torch.equal(torch.cuda.get_rng_state(), state_grad)
    assert torch.equal(out_n['sigma'], out_g['sigma'].detach()) and torch.equal(out_n['rgb'], out_g['rgb'].detach())


@pytest.mark.parametrize('n_img,n_pts', [(3, 1000), (1, 127)])
def test_kernel_paths_agree(pkg, monkeypatch, n_img, n_pts):
    """TPR_BWD_IMPL=hmma (the mma.sync kernel, 3xTF32) against the default path; decoder_precision='bf16' (one TF32 product
    where the mma.sync kernel runs, bf16 operands in the forward) in the 1e-2 class of the render backward's bf16 mode."""
    scene, pts = synthetic(n_img, n_pts)
    A, B = weights(n_img, n_pts)
    opts = dict(O.FFHQ_OPTIONS)
    for variant in ('rgb_sigma', 'sigma_only_query'):
        _, g_def = ours(pkg, scene, pts, opts, A, B, variant)
        monkeypatch.setenv('TPR_BWD_IMPL', 'hmma')
        _, g_hmma = ours(pkg, scene, pts, opts, A, B, variant)
        monkeypatch.delenv('TPR_BWD_IMPL')
        for a, b in zip(g_def, g_hmma):
            assert rel_err(b, a) < 5e-5
    _, g_bf = ours(pkg, scene, pts, dict(opts, decoder_precision='bf16'), A, B)
    _, g_o = oracle(scene, pts, opts['box_warp'], A, B)
    check(g_bf, g_o, 1e-2)


def test_linear_in_the_upstream_gradient(pkg):
    """The fp16 gradient-side operands are rescaled by a power of two from the upstream gradient's range: 2, 2^-20 and 2^20
    times the upstream gradient give exactly-scaled gradients."""
    scene, pts = synthetic(2, 1000)
    A, B = weights(2, 1000)
    opts = dict(O.FFHQ_OPTIONS)
    for variant in ('rgb_sigma', 'sigma_only_query'):
        _, g1 = ours(pkg, scene, pts, opts, A, B, variant)
        for f in (2.0, 2.0 ** -20, 2.0 ** 20):
            _, gk = ours(pkg, scene, pts, opts, f * A, f * B, variant)
            for a, b in zip(g1, gk):
                assert rel_err(b, f * a) < 1e-5, (f, variant)


def test_requires_grad_handling(pkg):
    scene, pts = synthetic(2, 1000)
    A, B = weights(2, 1000)
    opts = dict(O.FFHQ_OPTIONS)
    R = pkg.ImportanceRenderer()
    out, full = ours(pkg, scene, pts, opts, A, B)
    # planes only / decoder only: exactly those .grad
    _, g = ours(pkg, scene, pts, opts, A, B, dec_grad=False)
    assert g[0] is not None and all(t is None for t in g[1:])
    assert rel_err(g[0], full[0]) < 1e-5
    _, g = ours(pkg, scene, pts, opts, A, B, planes_grad=False)
    assert g[0] is None and all(t is not None for t in g[1:])
    for a, b in zip(g[1:], full[1:]):
        assert rel_err(a, b) < 1e-5
    dec = make_decoder(pkg, scene['dec']).requires_grad_(True)
    planes = T(scene['planes']).requires_grad_(True)
    # coordinates that require grad and PackedPlanes are refused, not silently detached
    with pytest.raises(NotImplementedError, match='sample_coordinates requires grad'):
        R.run_model(planes, dec, T(pts).requires_grad_(True), None, opts)
    with pytest.raises(NotImplementedError, match='PackedPlanes'):
        R.run_model(pkg.pack_planes(T(scene['planes'])), dec, T(pts), None, opts)
    # a double backward raises
    res = R.run_model(planes, dec, T(pts), None, opts)
    gp, = torch.autograd.grad(loss_of(res, A, B, 'rgb_sigma'), planes, create_graph=True)
    with pytest.raises(RuntimeError):
        gp.sum().backward()
    # no_grad: the inference path, bit-identical outputs
    with torch.no_grad():
        inf = R.run_model(planes, dec, T(pts), None, opts)
        inf_s = R.run_model(planes, dec, T(pts), None, opts, want_rgb=False)
    assert not inf['rgb'].requires_grad and res['rgb'].requires_grad and res['sigma'].requires_grad
    assert torch.equal(inf['rgb'], res['rgb'].detach()) and torch.equal(inf['sigma'], res['sigma'].detach())
    assert torch.equal(inf_s['sigma'], res['sigma'].detach())
    # the sharded query's in-place all-gather carries no gradient: it refuses autograd explicitly
    with pytest.raises(NotImplementedError, match='inference-only'):
        pkg.parallel.run_model_sharded(R, planes, dec, T(pts), None, opts)
