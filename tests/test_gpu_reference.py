"""GPU: parity with the UNMODIFIED reference.

The forward, run_model and marcher / resampling comparisons are self-contained: they compare against the reference's own
outputs stored in tests/golden/ (tests/golden/make_golden.py ran the unmodified reference on each case's seeded inputs, with
its two uniform draws and its density-noise draws replaced by the case's stored ones), so they run in a clean checkout.
The module-level helper test needs the reference's own functions (oracle/_ref/g_nerf, oracle/build_ref.py; see
oracle/ref_loader.py) and skips without them.

Gates (BASELINE.json north_star): fp32 mode max-abs <= 1e-4 on rgb / depth / weight sum; bf16-MLP mode PSNR >= 50 dB."""
import numpy as np
import pytest
import torch

from oracle import ref_loader
from tests.cases import case_noise, density_noise_draws, depth_peak, load_case
from tests.test_gpu_parity import T, dev, make_decoder, psnr, TOL

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(ref_loader.reference_dir() is None,
                                     reason='needs the unmodified reference (oracle/_ref, python oracle/build_ref.py)')


@pytest.fixture(scope='module')
def ref():
    torch.backends.cuda.matmul.allow_tf32 = False        # as the reference sets it (training_loop.py:145-146)
    torch.backends.cudnn.allow_tf32 = False
    return ref_loader.import_reference()


def _decoders(pkg, ref, seed=0, bias_scale=0.5):
    """The reference's OSGDecoder and ours with the same parameters (state_dict interchange, both directions)."""
    theirs = ref_loader.make_decoder(seed)
    with torch.no_grad():
        theirs.net[0].bias.normal_(0, bias_scale); theirs.net[2].bias.normal_(0, bias_scale)
    theirs = theirs.to(dev())
    ours = pkg.OSGDecoder(32, {'decoder_lr_mul': 1, 'decoder_output_dim': 32})
    ours.load_state_dict(theirs.state_dict())
    return theirs, ours.to(dev()).requires_grad_(False)


def _psnr(a, b, peak):
    return 10 * np.log10(peak * peak / max(float(((a.double() - b.double()) ** 2).mean()), 1e-30))


def _both(pkg, ref, planes, theirs, ours, o, d, opts, seed=1):
    """(reference outputs, our outputs, RNG states after each) from the same generator state."""
    with torch.no_grad():
        torch.manual_seed(seed)
        want = ref.renderer.ImportanceRenderer()(planes, theirs, o, d, dict(opts))
        state_ref = torch.cuda.get_rng_state(dev())
        torch.manual_seed(seed)
        got = pkg.ImportanceRenderer()(planes, ours, o, d, dict(opts))
        state_ours = torch.cuda.get_rng_state(dev())
    return want, got, state_ref, state_ours


# test case -> the golden fixture holding the reference's outputs for it (config2_pair: the FFHQ options, two images)
FIXTURES = {'config2_pair': 'ffhq_small', 'inference_96': 'inference_96', 'white_back': 'white_back',
            'auto_limits': 'auto_limits', 'density_noise': 'density_noise', 'coarse_only': 'coarse_only',
            'disparity': 'disparity'}


@pytest.mark.parametrize('name', list(FIXTURES))
def test_forward_matches_the_reference_on_the_same_gpu(pkg, name):
    """RaySampler and ImportanceRenderer.forward on the B200 against the reference's rays and renders, same draws."""
    fixture = FIXTURES[name]
    scene, opts, gold = load_case(fixture)
    res = int(round(gold['origins'].shape[1] ** 0.5))
    o, d = pkg.RaySampler()(T(scene['c2w']), T(scene['K']), res)
    assert np.array_equal(o.cpu().numpy(), gold['origins']) and float(np.abs(d.cpu().numpy() - gold['dirs']).max()) <= 2e-7
    dec = make_decoder(pkg, scene['dec'])
    noise = tuple(T(a) for a in case_noise(fixture, scene))
    planes, o_ref, d_ref = T(scene['planes']), T(gold['origins']), T(gold['dirs'])
    with torch.no_grad():
        got = pkg.ImportanceRenderer()(planes, dec, o_ref, d_ref, dict(opts), noise=noise)
    want = (gold['rgb'], gold['depth'], gold['wsum'])
    errs = {k: float(np.abs(a.cpu().numpy() - b).max()) for k, a, b in zip(('rgb', 'depth', 'wsum'), got, want)}
    print(f'{name} ({fixture}): fp32 max-abs vs the reference:', errs)
    for a, b in zip(got, want):
        assert tuple(a.shape) == b.shape and torch.isfinite(a).all()
    assert max(errs.values()) < TOL, errs
    # bf16-MLP mode, same draws
    with torch.no_grad():
        got16 = pkg.ImportanceRenderer()(planes, dec, o_ref, d_ref, dict(opts, decoder_precision='bf16'), noise=noise)
    ps = {'rgb': psnr(got16[0].cpu().numpy(), gold['rgb'], 2.0),
          'depth': psnr(got16[1].cpu().numpy(), gold['depth'], depth_peak(opts, gold))}
    print(f'{name}: bf16-MLP PSNR (dB):', ps)
    assert min(ps.values()) >= 50.0, ps


def test_run_model_matches_the_reference_on_a_density_grid_slab(pkg):
    """run_model (config 5's query, gen_videos.py:33-55,198-209) at the fixtures' points, rgb and sigma of every point against
    the reference's run_model; with density_noise both add the same stored standard-normal draws."""
    for fixture in ('ffhq_small', 'density_noise'):
        scene, opts, gold = load_case(fixture)
        dn = opts.get('density_noise', 0)
        kw = dict(sigma_noise=T(density_noise_draws(fixture)[2])) if dn > 0 else {}
        with torch.no_grad():
            got = pkg.ImportanceRenderer().run_model(T(scene['planes']), make_decoder(pkg, scene['dec']), T(gold['pts']), None,
                                                     opts, **kw)
        assert float(np.abs(got['sigma'].cpu().numpy() - gold['pts_sigma']).max()) < TOL
        assert float(np.abs(got['rgb'].cpu().numpy() - gold['pts_rgb']).max()) < TOL


@needs_reference
def test_module_level_helpers_match_the_reference(pkg, ref):
    """a2 / a3 / a4 / a12 / a15: generate_planes, project_onto_planes, sample_from_planes, sample_from_3dgrid, sort_samples
    and unify_samples -- the public names of VR/renderer.py that forward() does not call -- against the reference's own."""
    from importlib import import_module
    mine = import_module('g-nerf_b200.volumetric_rendering.renderer')
    theirs = ref.renderer
    assert torch.equal(mine.generate_planes(), theirs.generate_planes())
    axes = theirs.generate_planes().to(dev())
    rng = torch.Generator().manual_seed(7)
    xyz = (torch.rand((2, 501, 3), generator=rng) - 0.5).mul(1.3).to(dev())           # some outside the box
    torch.testing.assert_close(mine.project_onto_planes(axes, xyz), theirs.project_onto_planes(axes, xyz), rtol=0, atol=1e-6)
    planes = torch.randn((2, 3, 32, 40, 56), generator=rng).to(dev())                 # H != W
    want = theirs.sample_from_planes(axes, planes, xyz, padding_mode='zeros', box_warp=1.0)
    got = mine.sample_from_planes(axes, planes, xyz, padding_mode='zeros', box_warp=1.0)
    assert got.shape == want.shape == (2, 3, 501, 32)
    assert float((got - want).abs().max()) < 2e-5
    # the decoder on those features == run_model
    theirs_dec, ours_dec = _decoders(pkg, ref)
    a = ours_dec(got, None)
    b = pkg.ImportanceRenderer().run_model(planes, ours_dec, xyz, None, {'box_warp': 1.0, 'decoder_precision': 'fp32_ffma'})
    assert float((a['rgb'] - b['rgb']).abs().max()) < 2e-5 and float((a['sigma'] - b['sigma']).abs().max()) < 2e-5
    # 3-D grid, shared and per-batch, points beyond the borders
    for gshape in ((1, 5, 6, 7, 8), (2, 3, 4, 9, 5)):
        grid = torch.randn(gshape, generator=rng).to(dev())
        q = (torch.rand((2, 333, 3), generator=rng) * 2.4 - 1.2).to(dev())
        want = theirs.sample_from_3dgrid(grid, q)
        got = mine.sample_from_3dgrid(grid, q)
        assert got.shape == want.shape and float((got - want).abs().max()) < 1e-5
    # sort_samples / unify_samples: 48 + 48 samples with a few exact ties
    d1 = torch.rand((2, 37, 48, 1), generator=rng).to(dev()) + 2
    d2 = torch.rand((2, 37, 48, 1), generator=rng).to(dev()) + 2
    c1, c2 = torch.randn((2, 37, 48, 32), generator=rng).to(dev()), torch.randn((2, 37, 48, 32), generator=rng).to(dev())
    s1, s2 = torch.randn((2, 37, 48, 1), generator=rng).to(dev()), torch.randn((2, 37, 48, 1), generator=rng).to(dev())
    R_mine, R_theirs = pkg.ImportanceRenderer(), theirs.ImportanceRenderer()
    for got, want in zip(R_mine.unify_samples(d1, c1, s1, d2, c2, s2), R_theirs.unify_samples(d1, c1, s1, d2, c2, s2)):
        assert torch.equal(got, want)
    for got, want in zip(R_mine.sort_samples(d1, c1, s1), R_theirs.sort_samples(d1, c1, s1)):
        assert torch.equal(got, want)
    d1[:, :, 5] = d1[:, :, 4]                            # ties: torch.sort is unstable, so compare depths and the multiset only
    ds, cs, ss = R_mine.sort_samples(d1, c1, s1)
    wd, _, _ = R_theirs.sort_samples(d1, c1, s1)
    assert torch.equal(ds, wd) and torch.equal(ss.sort(dim=-2).values, s1.sort(dim=-2).values)


def test_marcher_and_resampling_match_the_reference(pkg):
    """MipRayMarcher2 on the fixtures' sample rows (black and white background) and the importance resampling of the
    fixtures' coarse weights with the same u, against the reference's outputs."""
    for fixture in ('ffhq_small', 'white_back'):
        _, opts, gold = load_case(fixture)
        got = pkg.MipRayMarcher2()(T(gold['march_colors']), T(gold['march_sigma']), T(gold['march_depths']), opts)
        for a, b in zip(got, (gold['march_rgb'], gold['march_depth'], gold['march_w'])):
            assert tuple(a.shape) == b.shape and float(np.abs(a.cpu().numpy() - b).max()) < 1e-5
    scene, _, gold = load_case('ffhq_small')
    fine = pkg.ImportanceRenderer().sample_pdf(T(gold['pdf_bins']), T(gold['pdf_weights']), scene['u'].shape[1],
                                               u=T(scene['u']))
    # a draw within an ulp of a CDF entry may land in the neighbouring bin (SURVEY.md section 7.1); everything else agrees
    # to the last ulps
    diff = np.abs(fine.cpu().numpy() - gold['depths_fine'].reshape(tuple(fine.shape)))
    assert float((diff > 1e-5).mean()) < 1e-4 and float(np.median(diff)) < 5e-7
