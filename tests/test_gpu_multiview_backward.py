"""The render backward of frame-batched calls -- F frames x P identities as N = F*P cameras over P plane sets (camera n samples
set n % P), with per-group depth clamps and either output layout -- against a float64 reference, and the equivalences that
make it a drop-in for the per-frame loop.

The reference is the loop over clamp groups of grads_given_depths (test_gpu_backward_coverage.py): each call takes one
group's cameras, their planes (planes[n % P]) and the forward's own coarse and importance depths, so its depth clamp is the
group's range, as a per-group reference forward's is; the gradients of the copies are summed back into the P sets.  With
density_noise the same arithmetic adds the forward's standard-normal draws x density_noise to every sample's sigma
(grads_given_noisy_depths; VR/renderer.py:146).  Gates as in the coverage test: gradients 2e-4 of the largest entry (bf16: 1e-2), forward 1e-4 (bf16: 5e-2)."""
import ctypes
from dataclasses import dataclass, field
from importlib import import_module

import numpy as np
import pytest
import torch

from oracle import triplane_oracle as O
from oracle import torch_oracle as TO
from tests.test_gpu_backward_coverage import (FWD_TOL, FWD_TOL_BF16, NAMES, REL, REL_BF16, decoder_backward_kernel,
                                              grads_given_depths, samples_kept, ws_keeps_samples)
from tests.test_gpu_deterministic_backward import deterministic
from tests.test_gpu_parity import dev, make_decoder
from tests.test_gpu_run_model_backward import no_tf32, rel_err  # noqa: F401  (no_tf32: autouse)

gpu = pytest.mark.gpu


@dataclass(frozen=True)
class Case:
    id: str
    P: int
    F: int
    dc: int = 48
    df: int = 48
    n_rays: int = 64
    clamp: int = -1                    # depth_clamp_group; -1 = P (one range per frame, what render_frames uses)
    opts: dict = field(default_factory=dict)
    keep_samples: bool = True
    keep_features: bool = True
    seed: int = 0
    density_noise: float = 0.0

    @property
    def k(self):
        return self.P if self.clamp < 0 else self.clamp

    @property
    def precision(self):
        return self.opts.get('decoder_precision', 'fp32')


CASES = [
    Case('P1_F2_kept', 1, 2, seed=1),
    Case('P2_F3_kept', 2, 3, seed=2),
    Case('P3_F5_kept_channels_first', 3, 5, n_rays=32, opts=dict(output_layout='channels_first'), seed=3),
    Case('P2_F3_one_range', 2, 3, clamp=0, seed=4),
    Case('P2_F5_ragged_groups_of_3', 2, 5, clamp=3, seed=5),
    Case('P3_F2_no_kept_samples', 3, 2, 40, 41, keep_samples=False, seed=6),
    Case('P2_F3_no_kept_features', 2, 3, keep_features=False, seed=7),
    Case('P2_F2_64+64_white_back', 2, 2, 64, 64, opts=dict(white_back=True), seed=8),
    Case('P3_F2_coarse_only', 3, 2, 40, 0, seed=9),
    Case('P2_F3_auto_limits', 2, 3, opts=dict(ray_start='auto', ray_end='auto'), seed=10),
    Case('P2_F3_mma_sync_1ray', 2, 3, n_rays=1, seed=11),
    Case('P2_F2_bf16', 2, 2, opts=dict(decoder_precision='bf16'), seed=12),
    Case('P1_F3_bf16_channels_first', 1, 3, opts=dict(decoder_precision='bf16', output_layout='channels_first'), seed=13),
    Case('P3_F2_kept_density_noise', 3, 2, density_noise=0.5, seed=14),
]
MODES = ('default', 'hmma', 'deterministic')


def _cov(c):
    from tests.test_gpu_backward_coverage import Case as CovCase
    return CovCase(c.id, c.dc, c.df, c.F * c.P, c.n_rays, opts=c.opts, keep_samples=c.keep_samples,
                   keep_features=c.keep_features)


def test_the_matrix_reaches_every_branch():
    """No GPU needed: the cases reach the plane-set counts, frame counts, clamp groupings, kept-sample classes, options and
    decoder-backward kernels the frame-batched backward has."""
    assert len({c.id for c in CASES}) == len(CASES)
    assert {c.P for c in CASES} >= {1, 2, 3} and {c.F for c in CASES} >= {2, 3, 5}
    assert any(c.k == c.P for c in CASES) and any(c.k == 0 for c in CASES)
    assert any(c.k > 0 and (c.P * c.F) % c.k for c in CASES), 'a ragged last clamp group'
    kept = [c for c in CASES if samples_kept(_cov(c))]
    assert any(c.keep_features for c in kept) and any(not c.keep_features for c in kept)
    assert any(not c.keep_samples for c in CASES)
    assert any(c.keep_samples and not ws_keeps_samples(c.dc, c.df) for c in CASES), 'a sample count outside the kept class'
    assert any(c.df == 0 for c in CASES)
    assert any(c.opts.get('ray_start') == 'auto' for c in CASES)
    assert any(c.opts.get('white_back') for c in CASES)
    assert {c.precision for c in CASES} >= {'fp32', 'bf16'}
    assert {c.opts.get('output_layout', 'channels_last') for c in CASES} == {'channels_last', 'channels_first'}
    kernels = {decoder_backward_kernel(c.P * c.F, c.n_rays, c.dc + c.df) for c in CASES}
    assert kernels == {'mma.sync', 'tcgen05', 'tcgen05_straddle'}, kernels
    assert any(c.density_noise > 0 and samples_kept(_cov(c)) for c in CASES)      # (density_noise needs kept samples)


def scene_of(case, density_noise=None):
    density_noise = case.density_noise if density_noise is None else density_noise
    rng = np.random.RandomState(2000 + case.seed)
    n, m, dc, df, P = case.P * case.F, case.n_rays, case.dc, case.df, case.P
    planes = rng.standard_normal((P, 3, 32, 32, 32)).astype(np.float32)
    dec = O.make_decoder_params(rng, 1.0, 0.5)
    c2w, K = O.orbit_cameras(n)
    o, d = O.ray_sample(c2w, K, 16)
    below_one = np.nextafter(np.float32(1), np.float32(0))
    jitter = np.minimum(rng.random_sample((n, m, dc, 1)).astype(np.float32), below_one)
    u = np.minimum(rng.random_sample((n * m, df)).astype(np.float32), below_one)
    A, B, C = (rng.standard_normal((n, m, k)).astype(np.float32) for k in (32, 1, 1))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    opts = dict(O.FFHQ_OPTIONS, depth_resolution=dc, depth_resolution_importance=df, depth_clamp_group=case.k, **case.opts)
    noise = (t(jitter), t(u) if df else None)
    if density_noise > 0:
        opts['density_noise'] = density_noise
        noise = noise + (t(rng.standard_normal((n, m * dc, 1)).astype(np.float32)),
                         t(rng.standard_normal((n, m * df, 1)).astype(np.float32)) if df else None)
    return dict(planes=t(planes), dec=dec, origins=t(o[:, :m]), dirs=t(d[:, :m]), noise=noise, A=t(A), B=t(B), C=t(C),
                opts=opts, P=P)


def run_kernels(pkg, sc, keep_samples=True, keep_features=True, planes=None):
    """Forward + backward of the whole batch; returns (outputs, gradients, coarse [N*M,Dc], fine or None, the clamp ranges
    the backward used, (samples kept, features kept)).  ``planes``: another plane tensor to render (replicated sets)."""
    dec = make_decoder(pkg, sc['dec']).requires_grad_(True)
    src = (sc['planes'] if planes is None else planes).clone().requires_grad_(True)
    R = pkg.ImportanceRenderer()
    R.keep_samples, R.keep_features = keep_samples, keep_features
    rgb, depth, wsum = R(src, dec, sc['origins'], sc['dirs'], sc['opts'], noise=sc['noise'])
    ctx = rgb.grad_fn
    saved = ctx.saved_tensors
    coarse, fine, ranges = saved[4].clone(), (saved[5].clone() if ctx.has_fine else None), saved[6].clone()
    kept = (ctx.has_saved, ctx.has_feat)
    ((rgb * sc['A']).sum() + (depth * sc['B']).sum() + (wsum * sc['C']).sum()).backward()
    grads = (src.grad, dec.net[0].weight.grad, dec.net[0].bias.grad, dec.net[2].weight.grad, dec.net[2].bias.grad)
    return (rgb.detach(), depth.detach(), wsum.detach()), grads, coarse, fine, ranges, kept, R


def groups(n, k):
    return [(0, n)] if k == 0 else [(g, min(n, g + k)) for g in range(0, n, k)]


def grads_given_noisy_depths(planes, dec, origins, dirs, coarse, fine, opts, A, B, C, nz_c, nz_f, dn):
    """grads_given_depths with density noise: sigma of every sample + dn x its draw (nz_c [N,M*Dc,1] for the coarse samples,
    nz_f [N,M*Df,1] for the importance samples, in the forward's sample order), carried through the stable depth sort."""
    cv = lambda t: t.detach().double()
    n, m, _ = origins.shape
    planes = cv(planes).requires_grad_(True)
    w1, b1, w2, b2 = (cv(t).requires_grad_(True) for t in dec[:4])
    d, nz = cv(coarse).reshape(n, m, -1), cv(nz_c).reshape(n, m, -1)
    if fine is not None and fine.numel():
        d, nz = torch.cat([d, cv(fine).reshape(n, m, -1)], -1), torch.cat([nz, cv(nz_f).reshape(n, m, -1)], -1)
    d, order = torch.sort(d, dim=-1, stable=True)
    nz = torch.gather(nz, -1, order)
    s = d.shape[-1]
    pts = (cv(origins).unsqueeze(-2) + d.unsqueeze(-1) * cv(dirs).unsqueeze(-2)).reshape(n, m * s, 3)
    rgb_s, sig_s = TO.decode(TO.gather(planes, pts, float(opts['box_warp'])), (w1, b1, w2, b2, dec[4]))
    sig_s = sig_s.reshape(n, m, s, 1) + nz.unsqueeze(-1) * dn
    rgb, depth, w = TO.march(rgb_s.reshape(n, m, s, -1), sig_s, d.unsqueeze(-1), bool(opts.get('white_back', False)))
    wsum = w.sum(2)
    loss = (rgb * cv(A)).sum() + (depth * cv(B)).sum() + (wsum * cv(C)).sum()
    grads = torch.autograd.grad(loss, (planes, w1, b1, w2, b2))
    return (rgb.detach(), depth.detach(), wsum.detach()), grads, None


def reference(sc, coarse, fine, k):
    """grads_given_depths per clamp group in float64, the plane gradients of the copies summed into the P sets."""
    n, m, _ = sc['origins'].shape
    P = sc['P']
    dec = TO.decoder_tuple(sc['dec'], dev())
    outs, g_planes, g_dec = [[], [], []], torch.zeros(sc['planes'].shape, dtype=torch.float64, device=dev()), None
    for g0, g1 in groups(n, k):
        idx = torch.arange(g0, g1, device=dev()) % P
        r = slice(g0 * m, g1 * m)
        args = (sc['planes'][idx], dec, sc['origins'][g0:g1], sc['dirs'][g0:g1], coarse[r], fine[r] if fine is not None else None,
                sc['opts'], sc['A'][g0:g1], sc['B'][g0:g1], sc['C'][g0:g1])
        if len(sc['noise']) == 4:
            nz_f = sc['noise'][3][g0:g1] if sc['noise'][3] is not None else None
            o, grads, _ = grads_given_noisy_depths(*args, sc['noise'][2][g0:g1], nz_f, sc['opts']['density_noise'])
        else:
            o, grads, _ = grads_given_depths(*args)
        for i in range(3):
            outs[i].append(o[i])
        g_planes.index_add_(0, idx, grads[0])
        g_dec = list(grads[1:]) if g_dec is None else [a + b for a, b in zip(g_dec, grads[1:])]
    return tuple(torch.cat(t) for t in outs), (g_planes, *g_dec)


def _depths(coarse, fine, n):
    return torch.cat([coarse.reshape(n, -1), fine.reshape(n, -1)], 1) if fine is not None else coarse.reshape(n, -1)


# ----------------------------------------------------------------------------------------------------------------------
# 1. the matrix against float64
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('case', CASES, ids=[c.id for c in CASES])
def test_frame_batched_backward_against_float64(pkg, monkeypatch, case, mode):
    if mode == 'hmma':
        monkeypatch.setenv('TPR_BWD_IMPL', 'hmma')
    sc = scene_of(case)
    with deterministic(mode == 'deterministic'):
        outs, grads, coarse, fine, ranges, kept, _ = run_kernels(pkg, sc, case.keep_samples, case.keep_features)
        if mode == 'deterministic':
            outs2, grads2 = run_kernels(pkg, sc, case.keep_samples, case.keep_features)[:2]
            for a, b in zip(outs, outs2):
                assert torch.equal(a, b)
            for k, a, b in zip(NAMES, grads, grads2):
                assert torch.equal(a, b), f'{k}: two deterministic runs differ'
    assert kept == (samples_kept(_cov(case)), samples_kept(_cov(case)) and case.keep_features), kept
    n = case.P * case.F
    d = _depths(coarse, fine, n)
    want_ranges = torch.stack([torch.stack([d[g0:g1].min(), d[g0:g1].max()]) for g0, g1 in groups(n, case.k)]).reshape(-1)
    assert torch.equal(ranges, want_ranges)
    outs_r, grads_r = reference(sc, coarse, fine, case.k)
    bf16 = case.precision == 'bf16'
    assert float(outs_r[2].min()) > 1e-3
    fwd = [float((a.double() - b).abs().max()) for a, b in zip(outs, outs_r)]
    errs = {k: rel_err(g, gr) for k, g, gr in zip(NAMES, grads, grads_r)}
    print(f'\n{case.id} [{mode}] forward max-abs rgb/depth/wsum {fwd[0]:.1e} {fwd[1]:.1e} {fwd[2]:.1e}; grad rel',
          ' '.join(f'{k} {v:.1e}' for k, v in errs.items()))
    assert max(fwd) < (FWD_TOL_BF16 if bf16 else FWD_TOL), fwd
    for k, g in zip(NAMES, grads):
        assert g is not None and torch.isfinite(g).all(), k
    assert max(errs.values()) < (REL_BF16 if bf16 else REL), errs


# ----------------------------------------------------------------------------------------------------------------------
# 2. the per-group ranges are the ones the forward clamped with, bit for bit
# ----------------------------------------------------------------------------------------------------------------------
def _ordered_to_float(u):
    u = u.astype(np.uint32)
    bits = np.where(u & 0x80000000, u & 0x7fffffff, ~u).astype(np.uint32)
    return bits.view(np.float32)


@gpu
@pytest.mark.parametrize('dc,df,k,precision', [(48, 48, 2, 'fp32'), (48, 48, 3, 'fp32'), (48, 48, 4, 'fp32'),
                                                (64, 64, 3, 'fp32'), (48, 48, 3, 'fp32_ffma')])
def test_group_ranges_equal_the_forwards(pkg, dc, df, k, precision):
    """The forward's per-group (min, max) pairs live in its scratch (from word 64, order-preserving encoding); the ranges
    the backward re-derives from the saved depths equal them bit for bit.  P = 2, F = 5: n = 10 cameras, so k = 3 and 4
    leave a ragged last group; 48+48 runs the forward's kept-samples kernel, 64+64 its default tcgen05 kernel (samples
    not kept) and fp32_ffma the FFMA kernel."""
    case = Case('ranges', 2, 5, dc, df, clamp=k, opts=dict(decoder_precision=precision), seed=20 + k)
    sc = scene_of(case)
    _, _, _, _, ranges, kept, R = run_kernels(pkg, sc)
    assert kept[0] == (dc + df == 96 and precision == 'fp32')
    n_slots = -(-10 // k)
    words = R.last_scratch[256:256 + 8 * n_slots].cpu().numpy().view(np.uint32)
    assert np.array_equal(_ordered_to_float(words), ranges.cpu().numpy())


# ----------------------------------------------------------------------------------------------------------------------
# 3. equivalences
# ----------------------------------------------------------------------------------------------------------------------
EQUIV = [  # (id, P, F, dc, df, density_noise)
    ('P2_F3_48+48', 2, 3, 48, 48, 0.0),
    ('P3_F2_48+48_density_noise', 3, 2, 48, 48, 0.5),
    ('P2_F2_64+64', 2, 2, 64, 64, 0.0),
]


@gpu
@pytest.mark.parametrize('mode', ('default', 'deterministic'))
@pytest.mark.parametrize('eid,P,F,dc,df,dn', EQUIV, ids=[e[0] for e in EQUIV])
def test_frame_batched_equals_replicated_planes(pkg, mode, eid, P, F, dc, df, dn):
    """The same batch with the planes replicated per camera (planes[n % P], N = F*P sets): outputs bit-equal, and the
    replicated copies' gradients summed per set within the gate."""
    case = Case(eid, P, F, dc, df, seed=40 + P * F)
    sc = scene_of(case, dn)
    with deterministic(mode == 'deterministic'):
        outs, grads = run_kernels(pkg, sc)[:2]
        idx = torch.arange(P * F, device=dev()) % P
        outs_r, grads_r = run_kernels(pkg, sc, planes=sc['planes'][idx].contiguous())[:2]
    for a, b in zip(outs, outs_r):
        assert torch.equal(a, b)
    summed = torch.zeros_like(grads[0]).index_add_(0, idx, grads_r[0])
    errs = {k: rel_err(g, gr) for k, g, gr in zip(NAMES, grads, (summed,) + tuple(grads_r[1:]))}
    print(f'\n{eid} [{mode}] frame-batched vs replicated:', ' '.join(f'{k} {v:.1e}' for k, v in errs.items()))
    assert max(errs.values()) < REL, errs


@gpu
@pytest.mark.parametrize('mode', ('default', 'deterministic'))
def test_channels_first_equals_channels_last(pkg, mode):
    case = Case('layout', 2, 3, seed=60)
    sc = scene_of(case)
    with deterministic(mode == 'deterministic'):
        outs, grads = run_kernels(pkg, sc)[:2]
        sc_cf = dict(sc, opts=dict(sc['opts'], output_layout='channels_first'))
        outs_cf, grads_cf = run_kernels(pkg, sc_cf)[:2]
    for a, b in zip(outs, outs_cf):
        assert torch.equal(a, b)
    for k, a, b in zip(NAMES, grads, grads_cf):
        if mode == 'deterministic':
            assert torch.equal(a, b), k
        else:
            assert rel_err(a, b) < REL, k


@gpu
def test_deterministic_plane_gradient_ignores_the_frame_order(pkg):
    """Reversing the frames (same per-frame rays, noise and upstream gradients) gives a bit-identical plane gradient."""
    case = Case('order', 2, 4, seed=70)
    sc = scene_of(case)
    P, F, m = 2, 4, case.n_rays
    perm = torch.cat([torch.arange(f * P, f * P + P) for f in reversed(range(F))]).to(dev())
    rev = dict(sc)
    for key in ('origins', 'dirs', 'A', 'B', 'C'):
        rev[key] = sc[key][perm].contiguous()
    jitter, u = sc['noise']
    rev['noise'] = (jitter[perm].contiguous(), u.view(P * F, m, -1)[perm].reshape(P * F * m, -1).contiguous())
    with deterministic(True):
        g = run_kernels(pkg, sc)[1][0]
        g_rev = run_kernels(pkg, rev)[1][0]
    assert torch.equal(g, g_rev)


# ----------------------------------------------------------------------------------------------------------------------
# 4. the per-group clamp at the C ABI
# ----------------------------------------------------------------------------------------------------------------------
@gpu
def test_per_group_clamp_at_the_c_abi(pkg):
    """tpr_render_backward with hand-chosen ranges: group 0's range cuts some of its rays' depths (their depth gradient is
    blocked), group 1's holds all of them.  Against float64 autograd of the march with the group's range."""
    case = Case('abi', 2, 2, seed=80)
    sc = scene_of(case)
    lib, P_ = pkg._lib.lib(), lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    n, m = 4, case.n_rays
    outs, _, coarse, fine, ranges, _, R = run_kernels(pkg, sc, keep_samples=False)
    # ranges: group 0 = cameras 0-1 narrowed to the middle of its raw depths, group 1 = cameras 2-3 widened
    d0 = outs[1][:2].reshape(-1).sort().values
    mine = torch.tensor([float(d0[m // 3]), float(d0[-m // 3]), float(ranges[2]) - 1.0, float(ranges[3]) + 1.0],
                        device=dev())
    dec = make_decoder(pkg, sc['dec'])
    packed = pkg.pack_planes(sc['planes']).data
    dec_p = pkg.pack_decoder(dec)
    o = pkg._lib.TprOptions(ray_start=2.25, ray_end=3.3, box_warp=1.0, depth_resolution=48, depth_resolution_importance=48,
                            plane_sets=2, depth_clamp_group=2, flags=pkg._lib.MLP_FP32)
    g_planes = torch.empty_like(packed)
    g_dec = torch.empty_like(dec_p)
    nbytes = lib.tpr_render_backward_scratch_bytes(n, m, 96)
    scratch = torch.empty(nbytes, device=dev(), dtype=torch.uint8)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    pkg._lib.check(lib.tpr_render_backward(P_(packed), n, 32, 32, P_(dec_p), P_(sc['origins']), P_(sc['dirs']), m, P_(coarse),
                                           P_(fine), P_(mine), ctypes.byref(o), P_(sc['A']), P_(sc['B']), P_(sc['C']), None,
                                           None, None, P_(g_planes), P_(g_dec), P_(scratch), nbytes, st), 'tpr_render_backward')
    g_nchw = torch.empty_like(sc['planes'])
    pkg._lib.check(lib.tpr_unpack_planes(P_(g_planes), 2, 32, 32, P_(g_nchw), st), 'tpr_unpack_planes')
    # float64: the group's reference with its clamp narrowed to the chosen range (march_given_range semantics)
    dec_t = TO.decoder_tuple(sc['dec'], dev())
    want = torch.zeros(sc['planes'].shape, dtype=torch.float64, device=dev())
    blocked = 0
    for j, (g0, g1) in enumerate(((0, 2), (2, 4))):
        idx = torch.arange(g0, g1, device=dev()) % 2
        lo, hi = float(mine[2 * j]), float(mine[2 * j + 1])
        planes = sc['planes'][idx].double().requires_grad_(True)
        w = [t.detach().double() for t in dec_t[:4]]
        dd = torch.cat([coarse[g0 * m:g1 * m], fine[g0 * m:g1 * m]], -1).double().reshape(2, m, -1)
        dd = torch.sort(dd, dim=-1, stable=True).values
        pts = (sc['origins'][g0:g1].double().unsqueeze(-2) + dd.unsqueeze(-1) * sc['dirs'][g0:g1].double().unsqueeze(-2))
        rgb_s, sig_s = TO.decode(TO.gather(planes, pts.reshape(2, -1, 3), 1.0), (*w, dec_t[4]))
        s = dd.shape[-1]
        rgb, depth, wts = TO.march(rgb_s.reshape(2, m, s, -1), sig_s.reshape(2, m, s, 1), dd.unsqueeze(-1), False)
        blocked += int(((depth < lo) | (depth > hi)).sum())
        depth = torch.clamp(depth, lo, hi)
        loss = (rgb * sc['A'][g0:g1].double()).sum() + (depth * sc['B'][g0:g1].double()).sum() + \
            (wts.sum(2) * sc['C'][g0:g1].double()).sum()
        want.index_add_(0, idx, torch.autograd.grad(loss, planes)[0])
        if j == 1:
            assert not bool(((depth <= lo) | (depth >= hi)).any())
    assert blocked > 0
    err = rel_err(g_nchw, want)
    print(f'\nper-group clamp at the C ABI: {blocked} rays clamped, plane gradient rel {err:.1e}')
    assert err < REL


# ----------------------------------------------------------------------------------------------------------------------
# 5. render_frames under autograd
# ----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('wants', ['planes', 'decoder', 'both'])
@pytest.mark.parametrize('fpc', [1, 2, None])
def test_render_frames_under_grad(pkg, fpc, wants):
    """The planes, the decoder or both require grad.  The frames are attached to them (with only the planes requiring grad
    the frames used to come back detached; with the decoder, render_frames raised), equal bit for bit to the same call under
    no_grad, and the gradients of whatever requires grad match a per-frame loop of autograd forwards from the same
    generator seed.  The generator ends in the same state."""
    P, F, res = 2, 3, 8
    rng = np.random.RandomState(90)
    planes = torch.from_numpy(rng.standard_normal((P, 3, 32, 32, 32)).astype(np.float32)).to(dev())
    dec = make_decoder(pkg, O.make_decoder_params(rng, 1.0, 0.5))
    c2w, K = O.orbit_cameras(F)
    c2w, K = torch.from_numpy(c2w.astype(np.float32)).to(dev()), torch.from_numpy(K[0].astype(np.float32)).to(dev())
    opts = dict(O.FFHQ_OPTIONS)
    R = pkg.ImportanceRenderer()
    Wf = torch.from_numpy(rng.standard_normal((F, P, 32, res, res)).astype(np.float32)).to(dev())
    Wd = torch.from_numpy(rng.standard_normal((F, P, 1, res, res)).astype(np.float32)).to(dev())

    torch.manual_seed(5)
    with torch.no_grad():
        ref = pkg.render_frames(R, planes, dec, c2w, K, res, opts, frames_per_call=fpc)
    state_nograd = torch.cuda.get_rng_state()

    want_pl, want_dec = wants in ('planes', 'both'), wants in ('decoder', 'both')
    dec.requires_grad_(want_dec)
    torch.manual_seed(5)
    pl = planes.clone().requires_grad_(want_pl)
    got = pkg.render_frames(R, pl, dec, c2w, K, res, opts, frames_per_call=fpc)
    assert torch.equal(torch.cuda.get_rng_state(), state_nograd)
    assert got['feature_image'].requires_grad and got['depth_image'].requires_grad
    for key in ('feature_image', 'depth_image', 'weights_image'):
        assert torch.equal(got[key].detach(), ref[key]), key
    ((got['feature_image'] * Wf).sum() + (got['depth_image'] * Wd).sum()).backward()
    assert (pl.grad is not None) == want_pl
    params = list(dec.parameters())
    g_dec = [p.grad.clone() if p.grad is not None else None for p in params]
    assert all((g is not None) == want_dec for g in g_dec)
    for p in params:
        p.grad = None

    # the per-frame loop: one reference-style forward of the P-batch per frame, same generator
    torch.manual_seed(5)
    pl2 = planes.clone().requires_grad_(want_pl)
    loss = 0
    RS = import_module('g-nerf_b200.volumetric_rendering.ray_sampler').RaySampler()
    for f in range(F):
        o, d = RS(c2w[f:f + 1].expand(P, -1, -1).contiguous(), K[None].expand(P, -1, -1).contiguous(), res)
        rgb, depth, _ = R(pl2, dec, o, d, opts)
        loss = loss + (rgb.permute(0, 2, 1).reshape(P, 32, res, res) * Wf[f]).sum() + \
            (depth.permute(0, 2, 1).reshape(P, 1, res, res) * Wd[f]).sum()
    loss.backward()
    assert torch.equal(torch.cuda.get_rng_state(), state_nograd)
    if want_pl:
        assert rel_err(pl.grad, pl2.grad) < REL
    if want_dec:
        for i, (g, p) in enumerate(zip(g_dec, params)):
            assert rel_err(g, p.grad) < REL, i


# ----------------------------------------------------------------------------------------------------------------------
# 6. the deterministic scratch holds P plane sets, not N cameras
# ----------------------------------------------------------------------------------------------------------------------
@gpu
def test_deterministic_scratch_is_sized_for_the_plane_sets(pkg, monkeypatch):
    """A deterministic frame-batched backward (P = 2, F = 4) hands tpr_render_backward the base scratch plus the fixed-point
    accumulator of the 2 plane sets: the accumulator of all 8 cameras would be 4x larger than the library uses."""
    case = Case('scratch', 2, 4, seed=95)
    sc = scene_of(case)
    lib = pkg._lib.lib()
    real, seen = lib.tpr_render_backward, []

    def spy(*args):
        seen.append(args[-2])                                        # scratch_bytes
        return real(*args)
    monkeypatch.setattr(lib, 'tpr_render_backward', spy)
    with deterministic(True):
        run_kernels(pkg, sc)
    n, m = 8, case.n_rays
    want = lib.tpr_render_backward_scratch_bytes(n, m, 96) + lib.tpr_backward_deterministic_scratch_bytes(2, 32, 32)
    assert seen == [want], (seen, want)
