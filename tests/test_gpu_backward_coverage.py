"""The render backward on every kernel path its dispatcher can take, against a float64 reference that takes the forward's
own sample depths.

The reference's graph treats the coarse and the importance depths as constants (VR/renderer.py:198,210: no_grad + detach).
So the float64 reference (grads_given_depths) does not re-derive them -- a float64 CDF would put some importance samples in
other bins -- but takes the coarse depths from ImportanceRenderer.sample_stratified (the call the backward itself makes) and
the importance depths the forward drew (ImportanceRenderer.last_fine).  From there on it is the reference's arithmetic in
float64: stable sort, bilinear gather, decoder, march, and autograd to the planes and the four decoder tensors.

What each case exists for is in its id: the bucket E of march_backward_kernel<E> (E = ceil(S / 32), rounded up to
1, 2, 3, 4, 6, 8), the forward kernel (warp-specialised tcgen05 with R = 8 or 4 rays per group, its kept-samples TRAIN
instantiation, or the FFMA kernel), the decoder backward (tcgen05, or mma.sync below 128 samples per image) and the plane
shape.  test_the_matrix_covers_every_dispatch_branch restates the dispatch rules and runs without a GPU.

Gates: 2e-4 of each gradient's largest entry (1e-2 with decoder_precision='bf16'); the forward outputs within 1e-4 of the
float64 forward (5e-2 in bf16 mode, the forward's own bf16 gate); the marcher alone within 2e-5.  Rays whose fp32 weights
underflow or saturate have no fp32-faithful float64 counterpart and are tested against the reference's fp32 arithmetic
(test_empty_and_opaque_rays).  Run with -s to see the worst relative error per case and gradient."""
import ctypes
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

from oracle import triplane_oracle as O
from oracle import torch_oracle as TO
from tests.test_gpu_deterministic_backward import deterministic
from tests.test_gpu_parity import dev, make_decoder
from tests.test_gpu_run_model_backward import no_tf32, rel_err  # noqa: F401  (no_tf32: autouse, fp32 references in full fp32)

gpu = pytest.mark.gpu
NAMES = ('planes', 'w1', 'b1', 'w2', 'b2')
REL, REL_BF16, REL_MARCH = 2e-4, 1e-2, 2e-5
FWD_TOL, FWD_TOL_BF16 = 1e-4, 5e-2


# ----------------------------------------------------------------------------------------------------------------------
# the dispatch rules, restated (csrc/tpr_backward.cu: launch_bwd_march; csrc/tpr_render_ws.cu: ws_rays_per_group,
# ws_keeps_samples; csrc/triplane_b200.cu: tpr_render's dispatch and decoder_backward; csrc/tpr_render_ws_*.cu)
# ----------------------------------------------------------------------------------------------------------------------
MARCH_BUCKETS = (1, 2, 3, 4, 6, 8)
WS_ROWS = 128                                   # samples per tcgen05 tile
WS_SLOTS = {'fp32': 14, 'bf16': 13}             # colour slots: Cols<2>::ns, Cols<1>::ns
TC_TILE = 128                                   # samples per tile of decode_backward_tc_kernel


def march_bucket(s):
    e = (s + 31) // 32
    return next(b for b in MARCH_BUCKETS if e <= b)


def ws_rays_per_group(dc, df, precision):
    if precision == 'fp32_ffma':
        return 0
    for r in (8, 4):
        dpt = WS_ROWS // r
        nc, nf = -(-dc // dpt), (-(-df // dpt) if df > 0 else 0)
        if 2 * nc + nf <= WS_SLOTS[precision]:
            return r
    return 0


def ws_keeps_samples(dc, df):
    return 64 < dc + df <= 96 and ws_rays_per_group(dc, df, 'fp32') == 8


def forward_kernel(dc, df, precision, keep_samples):
    """The kernel instantiation tpr_render_train launches for this case: render_kernel<E> (FFMA) or
    render_ws_kernel<MODE, ...> (tcgen05; MODE 1 = bf16, 2 = fp32), whose rays per group R is a run-time argument."""
    s = dc + df
    if ws_rays_per_group(dc, df, precision) == 0:
        return f'render_kernel<{2 if s <= 64 else 4 if s <= 128 else 8}>'
    mode = 1 if precision == 'bf16' else 2
    if keep_samples and ws_keeps_samples(dc, df):
        return f'render_ws_kernel<{mode},4,3,train>'
    return f'render_ws_kernel<{mode},{"2,2" if s <= 64 else "4,3" if s <= 96 else "4,4" if s <= 128 else "8,6" if s <= 192 else "8,8"}>'


def samples_kept(case):
    """Does the forward keep every sample's colours and sigma for the backward (only render_ws_kernel's train variant can)?"""
    return case.keep_samples and forward_kernel(case.dc, case.df, case.precision, True).endswith('train>')


def decoder_backward_kernel(n_img, n_rays, s):
    """tcgen05 when every image has at least one tile of samples, else mma.sync; 'straddle' = tiles that cross images and a
    partial last tile."""
    per_img = n_rays * s
    if per_img < TC_TILE:
        return 'mma.sync'
    return 'tcgen05_straddle' if n_img >= 2 and per_img % TC_TILE else 'tcgen05'


# ----------------------------------------------------------------------------------------------------------------------
# the matrix
# ----------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    id: str
    dc: int
    df: int
    n_img: int = 1
    n_rays: int = 64
    hw: tuple = (32, 32)
    opts: dict = field(default_factory=dict)
    keep_samples: bool = True
    keep_features: bool = True
    seed: int = 0

    @property
    def precision(self):
        return self.opts.get('decoder_precision', 'fp32')


CASES = [
    # march_backward_kernel<E> end to end, and the forward instantiations those sample counts select
    Case('E1_20+12', 20, 12, seed=1),
    Case('E2_36+27_odd', 36, 27, seed=2),
    Case('E3_40+41_kept_odd_exact_rank', 40, 41, seed=3),
    Case('E4_64+64_S128_R8', 64, 64, seed=4),
    Case('E4_112+16_S128_R4', 112, 16, seed=5),
    Case('E6_100+60_R4', 100, 60, seed=6),
    Case('E8_128+128_S256_R4', 128, 128, seed=7),
    Case('E8_255+0_ffma_fwd', 255, 0, seed=8),
    Case('E8_200+56_ffma_fwd', 200, 56, seed=9),
    # planes: non-square and tiny, rays leaving the box so that taps fall on padding
    Case('planes_16x24', 24, 24, hw=(16, 24), opts=dict(box_warp=0.6), seed=10),
    Case('planes_40x8', 24, 24, hw=(40, 8), opts=dict(box_warp=0.6), seed=11),
    Case('planes_1x64', 24, 24, hw=(1, 64), opts=dict(box_warp=0.6), seed=12),
    Case('planes_7x5', 24, 24, hw=(7, 5), opts=dict(box_warp=0.6), seed=13),
    # ray counts: below one tcgen05 tile per image; tiles straddling images with a partial last tile
    Case('mma_sync_1ray_48+48', 48, 48, n_rays=1, seed=14),
    Case('straddle_3img_37rays_48+48', 48, 48, n_img=3, n_rays=37, seed=15),
    # options
    Case('white_back_48+48', 48, 48, opts=dict(white_back=True), seed=16),
    Case('white_back_E8_128+128', 128, 128, opts=dict(white_back=True), seed=17),
    Case('disparity_40+24', 40, 24, opts=dict(disparity_space_sampling=True), seed=18),
    Case('fp32_ffma_48+48', 48, 48, opts=dict(decoder_precision='fp32_ffma'), seed=19),
    Case('fp32_ffma_planes_7x5', 24, 24, hw=(7, 5), opts=dict(box_warp=0.6, decoder_precision='fp32_ffma'), seed=24),
    Case('bf16_48+48', 48, 48, opts=dict(decoder_precision='bf16'), seed=20),
    Case('bf16_E4_64+64', 64, 64, opts=dict(decoder_precision='bf16'), seed=21),
    Case('bf16_E1_20+12', 20, 12, opts=dict(decoder_precision='bf16'), seed=25),
    Case('bf16_no_kept_samples_40+41', 40, 41, opts=dict(decoder_precision='bf16'), keep_samples=False, seed=26),
    Case('bf16_E6_100+60_R4', 100, 60, opts=dict(decoder_precision='bf16'), seed=27),
    Case('bf16_E8_128+128_R4', 128, 128, opts=dict(decoder_precision='bf16'), seed=28),
    Case('no_kept_samples_40+41', 40, 41, keep_samples=False, seed=22),
    Case('no_kept_features_40+41', 40, 41, keep_features=False, seed=23),
]
MODES = ('default', 'hmma', 'deterministic')


def test_the_matrix_covers_every_dispatch_branch():
    """No GPU needed: every bucket of march_backward_kernel<E>, every forward kernel instantiation the training path can
    launch (with both ray-group sizes) and both decoder-backward kernels are reached by some case, so that a change of the
    dispatch cannot leave a branch untested without this failing.  test_render_backward_against_float64 checks on the GPU
    that each case ran the forward named here."""
    assert len({c.id for c in CASES}) == len(CASES)
    assert {march_bucket(c.dc + c.df) for c in CASES} == set(MARCH_BUCKETS)
    # the bucket edges of march_backward_kernel<E> are the marcher-alone sizes
    edges = {32 * b for b in MARCH_BUCKETS} | {32 * b + 1 for b in MARCH_BUCKETS[:-1]}
    assert edges == set(MARCH_SIZES)
    fwd = {forward_kernel(c.dc, c.df, c.precision, c.keep_samples) for c in CASES}
    want = {f'render_ws_kernel<{m},{t}>' for m in (1, 2) for t in ('2,2', '4,3', '4,3,train', '4,4', '8,6', '8,8')}
    want |= {f'render_kernel<{e}>' for e in (2, 4, 8)}
    assert fwd == want, (want - fwd, fwd - want)
    # rays per group: both sizes in both precisions, and S = 128 with either
    groups = {(c.precision, c.dc + c.df, ws_rays_per_group(c.dc, c.df, c.precision)) for c in CASES}
    for prec in ('fp32', 'bf16'):
        assert {r for p, _, r in groups if p == prec} >= {8, 4}, prec
    assert {('fp32', 128, 8), ('fp32', 128, 4)} <= groups
    # the slot arithmetic itself: 48+48 packs 8 rays per group, 96+96 and 128+128 only 4, 255+0 and 200+56 none
    assert ws_rays_per_group(48, 48, 'fp32') == 8 and ws_rays_per_group(96, 96, 'fp32') == 4
    assert ws_rays_per_group(128, 128, 'fp32') == 4 and ws_rays_per_group(255, 0, 'fp32') == 0
    assert ws_rays_per_group(200, 56, 'fp32') == 0 and ws_rays_per_group(64, 64, 'bf16') == 8
    assert ws_keeps_samples(48, 48) and ws_keeps_samples(40, 41) and not ws_keeps_samples(32, 32)
    assert not ws_keeps_samples(64, 64) and not ws_keeps_samples(96, 96)
    bwd = {decoder_backward_kernel(c.n_img, c.n_rays, c.dc + c.df) for c in CASES}
    assert bwd == {'mma.sync', 'tcgen05', 'tcgen05_straddle'}
    # both rank paths of the marcher (fast: Dc and S multiples of four; exact: otherwise) end to end
    assert any(c.dc % 4 == 0 and (c.dc + c.df) % 4 == 0 for c in CASES)
    assert any((c.dc + c.df) % 4 for c in CASES if samples_kept(c))
    # options
    assert {c.precision for c in CASES} == {'fp32', 'fp32_ffma', 'bf16'}
    for key in ('white_back', 'disparity_space_sampling'):
        assert any(c.opts.get(key) for c in CASES), key
    assert {c.hw for c in CASES} >= {(16, 24), (40, 8), (1, 64), (7, 5)}
    assert any(not c.keep_samples for c in CASES) and any(c.keep_samples and not c.keep_features for c in CASES)


# ----------------------------------------------------------------------------------------------------------------------
# the float64 reference
# ----------------------------------------------------------------------------------------------------------------------
def grads_given_depths(planes, dec, origins, dirs, coarse, fine, opts, A, B, C, dtype=torch.float64):
    """The reference's forward and backward in `dtype` at the given sample depths.
    planes [N,3,32,H,W]; dec (w1, b1, w2, b2, lr_mul); origins / dirs [N,M,3]; coarse [N*M,Dc]; fine [N*M,Df] or None;
    A [N,M,32], B and C [N,M,1]: the loss sum(rgb*A) + sum(depth*B) + sum(wsum*C).
    Returns ((rgb, depth, wsum), (g_planes, g_w1, g_b1, g_w2, g_b2), alpha [N,M,S-1,1]); the depth clamp takes the range
    of the depths given, as VR/ray_marcher.py:50 does."""
    cv = lambda t: t.detach().to(dtype)
    n, m, _ = origins.shape
    planes = cv(planes).requires_grad_(True)
    w1, b1, w2, b2 = (cv(t).requires_grad_(True) for t in dec[:4])
    d = cv(coarse).reshape(n, m, -1)
    if fine is not None and fine.numel():
        d = torch.cat([d, cv(fine).reshape(n, m, -1)], -1)
    d = torch.sort(d, dim=-1, stable=True).values                   # equal depths: coarse first (VR/renderer.py:157-167)
    s = d.shape[-1]
    pts = (cv(origins).unsqueeze(-2) + d.unsqueeze(-1) * cv(dirs).unsqueeze(-2)).reshape(n, m * s, 3)
    rgb_s, sig_s = TO.decode(TO.gather(planes, pts, float(opts['box_warp'])), (w1, b1, w2, b2, dec[4]))
    rgb, depth, w = TO.march(rgb_s.reshape(n, m, s, -1), sig_s.reshape(n, m, s, 1), d.unsqueeze(-1),
                             bool(opts.get('white_back', False)))
    wsum = w.sum(2)
    loss = (rgb * cv(A)).sum() + (depth * cv(B)).sum() + (wsum * cv(C)).sum()
    grads = torch.autograd.grad(loss, (planes, w1, b1, w2, b2))
    with torch.no_grad():                                            # VR/ray_marcher.py:30-40
        sig = sig_s.reshape(n, m, s, 1)
        alpha = 1 - torch.exp(-torch.nn.functional.softplus((sig[:, :, :-1] + sig[:, :, 1:]) / 2 - 1) *
                              (d[:, :, 1:] - d[:, :, :-1]).unsqueeze(-1))
    return (rgb.detach(), depth.detach(), wsum.detach()), grads, alpha


def march_given_range(colors, sigma, depths, white_back, lo, hi):
    """TO.march with the depth clamp to an explicit range [lo, hi] (inside the depths' own range: clamping again to the
    narrower range is the same as clamping to it once, gradient included)."""
    rgb, depth, w = TO.march(colors, sigma, depths, white_back)
    return rgb, torch.clamp(depth, lo, hi), w


def scene_of(case):
    """Random N(0,1) planes of the case's H x W, a decoder with non-trivial biases, the first n_rays rays of a 16 x 16 image
    per orbit camera, seeded draws and upstream gradients."""
    rng = np.random.RandomState(1000 + case.seed)
    h, w = case.hw
    n, m, dc, df = case.n_img, case.n_rays, case.dc, case.df
    planes = rng.standard_normal((n, 3, 32, h, w)).astype(np.float32)
    dec = O.make_decoder_params(rng, 1.0, 0.5)
    c2w, K = O.orbit_cameras(n)
    o, d = O.ray_sample(c2w, K, 16)
    below_one = np.nextafter(np.float32(1), np.float32(0))
    jitter = np.minimum(rng.random_sample((n, m, dc, 1)).astype(np.float32), below_one)
    u = np.minimum(rng.random_sample((n * m, df)).astype(np.float32), below_one)
    A, B, C = (rng.standard_normal((n, m, k)).astype(np.float32) for k in (32, 1, 1))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    opts = dict(O.FFHQ_OPTIONS, depth_resolution=dc, depth_resolution_importance=df, **case.opts)
    return dict(planes=t(planes), dec=dec, origins=t(o[:, :m]), dirs=t(d[:, :m]), jitter=t(jitter), u=t(u) if df else None,
                A=t(A), B=t(B), C=t(C), opts=opts)


def run_kernels(pkg, sc, keep_samples=True, keep_features=True):
    """Forward and backward through ImportanceRenderer; returns (outputs, gradients, the forward's coarse and importance
    depths [N*M, Dc], [N*M, Df] or None, the forward's depth range, (samples kept, features kept) as the forward
    reported them to the backward)."""
    dec = make_decoder(pkg, sc['dec']).requires_grad_(True)
    planes = sc['planes'].clone().requires_grad_(True)
    R = pkg.ImportanceRenderer()
    R.keep_samples, R.keep_features = keep_samples, keep_features
    opts = sc['opts']
    rgb, depth, wsum = R(planes, dec, sc['origins'], sc['dirs'], opts, noise=(sc['jitter'], sc['u']))
    kept = (rgb.grad_fn.has_saved, rgb.grad_fn.has_feat)            # (the grad_fn of an autograd.Function is its ctx)
    ((rgb * sc['A']).sum() + (depth * sc['B']).sum() + (wsum * sc['C']).sum()).backward()
    n, m, _ = sc['origins'].shape
    coarse = R.sample_stratified(sc['origins'], opts['ray_start'], opts['ray_end'], opts['depth_resolution'],
                                 bool(opts.get('disparity_space_sampling', False)), jitter=sc['jitter']).reshape(n * m, -1)
    fine = R.last_fine[0].clone() if opts['depth_resolution_importance'] > 0 else None
    grads = (planes.grad, dec.net[0].weight.grad, dec.net[0].bias.grad, dec.net[2].weight.grad, dec.net[2].bias.grad)
    return (rgb.detach(), depth.detach(), wsum.detach()), grads, coarse, fine, R.last_depth_range.clone(), kept


def reference(sc, coarse, fine, dtype=torch.float64):
    return grads_given_depths(sc['planes'], TO.decoder_tuple(sc['dec'], dev()), sc['origins'], sc['dirs'], coarse, fine,
                              sc['opts'], sc['A'], sc['B'], sc['C'], dtype=dtype)


# ----------------------------------------------------------------------------------------------------------------------
# 1. the matrix, end to end
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('case', CASES, ids=[c.id for c in CASES])
def test_render_backward_against_float64(pkg, monkeypatch, case, mode):
    if mode == 'hmma':
        monkeypatch.setenv('TPR_BWD_IMPL', 'hmma')
    sc = scene_of(case)
    with deterministic(mode == 'deterministic'):
        outs, grads, coarse, fine, rng, kept = run_kernels(pkg, sc, case.keep_samples, case.keep_features)
        if mode == 'deterministic':
            outs2, grads2, _, _, _, _ = run_kernels(pkg, sc, case.keep_samples, case.keep_features)
            for a, b in zip(outs, outs2):
                assert torch.equal(a, b)
            for k, a, b in zip(NAMES, grads, grads2):
                assert torch.equal(a, b), f'{k}: two deterministic runs differ'
    depths = torch.cat([coarse, fine], -1) if fine is not None else coarse
    assert torch.equal(rng, torch.stack([depths.min(), depths.max()])), 'the forward\'s depth range is not its depths\' range'
    outs_r, grads_r, alpha_r = reference(sc, coarse, fine)       # (torch's grid_sample backward refuses the deterministic mode)
    # the case ran the forward its id names: kept samples only from render_ws_kernel's train variant, and the FFMA kernel's
    # output, which does not depend on the decoder_precision flag, bit-equal to an fp32_ffma render iff the FFMA kernel ran
    assert kept == (samples_kept(case), samples_kept(case) and case.keep_features), kept
    if mode == 'default':
        with torch.no_grad():
            rgb_ffma = pkg.ImportanceRenderer()(sc['planes'], make_decoder(pkg, sc['dec']), sc['origins'], sc['dirs'],
                                                dict(sc['opts'], decoder_precision='fp32_ffma'), noise=(sc['jitter'], sc['u']))[0]
        ffma = forward_kernel(case.dc, case.df, case.precision, case.keep_samples).startswith('render_kernel')
        assert torch.equal(outs[0], rgb_ffma) == ffma, 'the forward kernel is not the one the case is for'
    # every ray of the matrix is one that fp32 represents: some weight, and no 1 - alpha + 1e-10 that fp32 rounds to ~1e-10
    assert float(outs_r[2].min()) > 1e-3 and float((1 - alpha_r.float()).min()) > 1e-6
    bf16 = case.precision == 'bf16'
    fwd = [float((a.double() - b).abs().max()) for a, b in zip(outs, outs_r)]
    errs = {k: rel_err(g, gr) for k, g, gr in zip(NAMES, grads, grads_r)}
    print(f'\n{case.id} [{mode}] forward max-abs rgb/depth/wsum {fwd[0]:.1e} {fwd[1]:.1e} {fwd[2]:.1e}; grad rel',
          ' '.join(f'{k} {v:.1e}' for k, v in errs.items()))
    assert max(fwd) < (FWD_TOL_BF16 if bf16 else FWD_TOL), fwd
    for k, g in zip(NAMES, grads):
        assert g is not None and torch.isfinite(g).all(), k
    assert max(errs.values()) < (REL_BF16 if bf16 else REL), errs


# ----------------------------------------------------------------------------------------------------------------------
# 2. the marcher alone, at the edges of its buckets
# ----------------------------------------------------------------------------------------------------------------------
MARCH_SIZES = (32, 33, 64, 65, 96, 97, 128, 129, 192, 193, 256)


def march_split(s, variant):
    """(Dc, Df): 'fast' = both multiples of four (the vector rank count; S % 4 == 0 only); 'ties' = the same split with equal
    depths (the rank sum sends the ray to the exact count); 'odd' = an odd coarse count (the exact count).  At an odd S every
    split is odd."""
    if variant == 'odd' or s % 4:
        dc = s // 2 + (1 - (s // 2) % 2)
        return dc, s - dc
    dc = (s // 2) // 4 * 4
    return dc, s - dc


@gpu
@pytest.mark.parametrize('s,variant', [(s, v) for s in MARCH_SIZES for v in ('fast', 'ties', 'odd', 'white_back', 'narrow_range')
                                       if not (v == 'fast' and s % 4)])        # (odd S: only the exact count exists)
def test_march_backward_at_the_bucket_edges(pkg, s, variant):
    """tpr_march_backward alone against float64 autograd of the march, per sample d/d(sigma) and colour weight omega.
    'narrow_range': a depth range that a third of the rays' depths fall below and a third above, so that the clamp blocks
    their depth gradient."""
    d = dev()
    g = torch.Generator(device=d).manual_seed(100 * s + len(variant))
    r = 29
    dc, df = march_split(s, variant)
    if variant in ('fast', 'ties', 'white_back', 'narrow_range') and s % 4 == 0:
        assert dc % 4 == 0 and df % 4 == 0
    coarse = torch.sort(torch.rand(r, dc, device=d, generator=g) * 0.8 + 2.3, -1).values.contiguous()
    fine = (torch.rand(r, df, device=d, generator=g) * 0.8 + 2.3).contiguous()
    if variant == 'ties':
        fine[:, 3] = fine[:, 7]                      # two equal importance depths
        fine[::2, 0] = coarse[::2, 5]                # an importance depth equal to a coarse one
        coarse[1::3, 11] = coarse[1::3, 10]          # equal coarse depths
    sigma = torch.randn(r, s, device=d, generator=g) * 3
    col = torch.rand(r, s, 32, device=d, generator=g)
    A, B, C = (torch.randn(r, k, device=d, generator=g) for k in (32, 1, 1))
    depths = torch.cat([coarse, fine], -1)
    white = variant == 'white_back'
    d64, order = torch.sort(depths.double(), dim=-1, stable=True)
    lo, hi = float(depths.min()), float(depths.max())
    if variant == 'narrow_range':
        # a third of the rays below the range, a third above: bounds halfway between neighbouring float64 raw depths
        with torch.no_grad():
            _, _, w = TO.march(torch.gather(col.double(), 1, order.unsqueeze(-1).expand(-1, -1, 32)).unsqueeze(0),
                               torch.gather(sigma.double(), 1, order).unsqueeze(0).unsqueeze(-1), d64.unsqueeze(0).unsqueeze(-1))
            raw = torch.sort(((w[0, :, :, 0] * (d64[:, 1:] + d64[:, :-1]) / 2).sum(1) / w[0, :, :, 0].sum(1))).values
        lo, hi = float((raw[r // 3 - 1] + raw[r // 3]) / 2), float((raw[2 * r // 3] + raw[2 * r // 3 + 1]) / 2)
    rng = torch.tensor([lo, hi], device=d, dtype=torch.float32)

    sig64 = sigma.double().requires_grad_(True)
    col64 = col.double().requires_grad_(True)
    rgb, depth, w = march_given_range(torch.gather(col64, 1, order.unsqueeze(-1).expand(-1, -1, 32)).unsqueeze(0),
                                      torch.gather(sig64, 1, order).unsqueeze(0).unsqueeze(-1), d64.unsqueeze(0).unsqueeze(-1),
                                      white, float(rng[0]), float(rng[1]))
    loss = (rgb[0] * A.double()).sum() + (depth[0] * B.double()).sum() + (w.sum(2)[0] * C.double()).sum()
    g_sig, g_col = torch.autograd.grad(loss, (sig64, col64))

    gs = torch.empty(r, s, device=d)
    om = torch.empty(r, s, device=d)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    pkg._lib.check(pkg._lib.lib().tpr_march_backward(P(coarse), P(fine), dc, df, P(sigma), P(col), P(A), P(B), P(C), P(rng),
                                                     int(white), r, P(gs), P(om),
                                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   'tpr_march_backward')
    torch.cuda.synchronize()
    e_sig = rel_err(gs, g_sig)
    e_col = rel_err(2 * A.unsqueeze(1) * om.unsqueeze(-1), g_col)
    print(f'\nmarch S={s} ({dc}+{df}) {variant}: g_sigma {e_sig:.1e} g_colour {e_col:.1e}')
    assert e_sig < REL_MARCH and e_col < REL_MARCH, (e_sig, e_col)


# ----------------------------------------------------------------------------------------------------------------------
# 3. rays whose fp32 weights underflow (empty) or whose alphas round to 1 (opaque)
# ----------------------------------------------------------------------------------------------------------------------
def extreme_scene(n_rays=32, dc=48, df=48):
    """Half the rays moved sideways out of the box: every tap is padding and sigma is the decoder's bias, -60 (softplus
    ~1e-26: exp(-sigma delta) == 1 in fp32, all weights exactly 0).  The planes are 5 in every texel and the decoder maps
    that to sigma ~2800 inside the box, so alpha rounds to 1 from the first sample in it."""
    rng = np.random.RandomState(77)
    dec = O.make_decoder_params(rng, 1.0, 0.5)
    dec.w1[:] = 1.0
    dec.b1[:] = -10.0
    dec.w2[0, :] = 20.0
    dec.b2[0] = -60.0
    planes = np.full((1, 3, 32, 16, 16), 5.0, np.float32)
    c2w, K = O.orbit_cameras(1)
    o, d = O.ray_sample(c2w, K, 16)
    o, d = o[:, :n_rays].copy(), d[:, :n_rays].copy()
    o[:, ::2] += np.cross(d[:, ::2], np.array([0.0, 1.0, 0.0], np.float32)) * 4.0     # sideways, by 4 box lengths
    below_one = np.nextafter(np.float32(1), np.float32(0))
    jitter = np.minimum(rng.random_sample((1, n_rays, dc, 1)).astype(np.float32), below_one)
    u = np.minimum(rng.random_sample((n_rays, df)).astype(np.float32), below_one)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev())
    opts = dict(O.FFHQ_OPTIONS, depth_resolution=dc, depth_resolution_importance=df)
    return dict(planes=t(planes), dec=dec, origins=t(o), dirs=t(d), jitter=t(jitter), u=t(u), opts=opts)


@gpu
@pytest.mark.parametrize('mode', MODES)
def test_empty_and_opaque_rays(pkg, monkeypatch, mode):
    """Against the reference's fp32 arithmetic: grads_given_depths in fp32 at the forward's depths.
    An empty ray's fp32 depth is 0/0 -> nan_to_num -> inf -> clamped to the range, so it passes no depth gradient; float64,
    whose weights do not underflow, gives it a finite depth and an O(1) depth gradient.  fp32 autograd itself turns the
    empty rays' 0/0 into NaN decoder gradients (the division's backward multiplies the blocked gradient, 0, by 0/0), so the
    gradients are compared over the opaque rays and the empty rays get exact properties instead: every gradient is finite,
    and a loss that reaches only their depths has a gradient of exactly zero."""
    if mode == 'hmma':
        monkeypatch.setenv('TPR_BWD_IMPL', 'hmma')
    sc = extreme_scene()
    n, m = 1, sc['origins'].shape[1]
    rng = np.random.RandomState(5)
    t = lambda a: torch.from_numpy(a.astype(np.float32)).to(dev())
    empty = torch.zeros(n, m, 1, device=dev())
    empty[:, ::2] = 1.0
    weights = {
        'all': [t(rng.standard_normal((n, m, k))) for k in (32, 1, 1)],
        'empty_depth_only': [torch.zeros(n, m, 32, device=dev()), t(rng.standard_normal((n, m, 1))) * empty,
                             torch.zeros(n, m, 1, device=dev())],
    }
    for name, (A, B, C) in weights.items():
        sc.update(A=A, B=B, C=C)
        with deterministic(mode == 'deterministic'):
            outs, grads, coarse, fine, _, _ = run_kernels(pkg, sc)
        outs_r, _, alpha_r = reference(sc, coarse, fine, dtype=torch.float32)
        # the scene is what it claims: the moved rays have no weight at all, the others saturate
        assert torch.equal(outs_r[2][:, ::2], torch.zeros_like(outs_r[2][:, ::2]))
        assert float(outs_r[2][:, 1::2].min()) > 0.999 and bool((alpha_r[:, 1::2] == 1.0).any())
        assert torch.equal(outs[2][:, ::2], outs_r[2][:, ::2]) and torch.equal(outs[1][:, ::2], outs_r[1][:, ::2])
        for k, g in zip(NAMES, grads):
            assert torch.isfinite(g).all(), (name, k)
        if name == 'empty_depth_only':
            for k, g in zip(NAMES, grads):
                assert torch.equal(g, torch.zeros_like(g)), k
            continue
        fwd = [float((a - b).abs().max()) for a, b in zip(outs, outs_r)]
        op = slice(1, None, 2)
        _, grads_r, _ = grads_given_depths(sc['planes'], TO.decoder_tuple(sc['dec'], dev()), sc['origins'][:, op],
                                           sc['dirs'][:, op], coarse[op], fine[op], sc['opts'], A[:, op], B[:, op],
                                           C[:, op], dtype=torch.float32)
        errs = {k: rel_err(g, gr) for k, g, gr in zip(NAMES, grads, grads_r)}
        print(f'\nempty/opaque [{mode}] forward max-abs rgb/depth/wsum {fwd[0]:.1e} {fwd[1]:.1e} {fwd[2]:.1e}; grad rel',
              ' '.join(f'{k} {v:.1e}' for k, v in errs.items()))
        assert max(fwd) < FWD_TOL, fwd
        assert max(errs.values()) < REL, errs
