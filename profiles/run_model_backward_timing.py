"""Autograd through ImportanceRenderer.run_model (point queries: TriPlaneGenerator.sample / sample_mixed) on one B200.

  * regulariser shape: EG3D's density regulariser, N = 4 images x (1000 + 1000 perturbed) points, sigma only, 256^2 planes:
    forward + L1 + backward per call (CUDA events), the fused path next to eager autograd through the torch restatement
    (oracle/torch_oracle.py: the reference's ATen ops);
  * config-5 grid (bench.py's config5 workload: 256^3 voxel centres of one identity, 256^2 planes), sigma only and rgb + sigma,
    random upstream gradient: tpr_run_model_backward alone (ms, G points/s), its plane-gradient scatter (12 x 128 B of
    red.global.add per point) as a fraction of the scatter ceiling measured in the same run (tpr_scatter_microbench on an
    L2-resident 25 MB target, as profiles/scatter_shapes.py), the decode kernel alone (torch.profiler), fused forward +
    backward against eager autograd (sigma only), and the render backward's decode kernel (keep_features=False, config 2)
    per sample beside it.
Measurement script, not product code.  Usage: python profiles/run_model_backward_timing.py > profiles/r03_run_model_backward_timing.json
``--roles``: one backward per variant with TPR_BWD_PROFILE=1 set by the caller (the per-role cycle table goes to stderr)."""
import argparse, ctypes, importlib, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F
import bench
from oracle import torch_oracle as TO
pkg = importlib.import_module('g-nerf_b200')
ap = argparse.ArgumentParser(); ap.add_argument('--reps', type=int, default=20); ap.add_argument('--roles', action='store_true')
args = ap.parse_args()
torch.backends.cuda.matmul.allow_tf32 = False
dev = torch.device('cuda:0')
L, P, ST = pkg._lib.lib(), (lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None), \
    (lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
opts = dict(bench.OPTS)
SCATTER_BYTES = 12 * 128


def timed(fn, warm=3, reps=args.reps):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def kernel_ms(fn, name, reps=5):
    """Mean device time of the kernels whose name contains `name`, per call of fn (torch.profiler, its own window)."""
    fn(); torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps): fn()
        torch.cuda.synchronize()
    tot = sum(e.device_time_total for e in prof.key_averages() if name in e.key)
    return tot / 1e3 / reps


def decoder_params():
    dec = bench.make_decoder(torch, pkg, dev, 0).requires_grad_(True)
    fc1, fc2 = dec.net[0], dec.net[2]
    raw = tuple(t.detach().clone().requires_grad_(True) for t in (fc1.weight, fc1.bias, fc2.weight, fc2.bias))
    return dec, raw + (float(fc1.bias_gain),)                 # (lr_mul: the runtime gains are the restatement's too)


out = {}
smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
out['gpu'] = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else f'nvidia-smi failed: {smi.stderr.strip()}'
dec, dec_raw = decoder_params()

# ---- config-5 grid: inputs of the backward (bench.py leg_config5)
g = 256
planes5 = torch.randn((1, 3, 32, bench.PLANE_RES, bench.PLANE_RES), device=dev, generator=torch.Generator(device=dev).manual_seed(500))
ax = (torch.arange(g, device=dev, dtype=torch.float32) + 0.5) / g - 0.5
zz, yy, xx = torch.meshgrid(ax, ax, ax, indexing='ij')
xyz5 = torch.stack([xx, yy, zz], -1).reshape(1, -1, 3).contiguous()
del zz, yy, xx
n5 = g ** 3
pp5 = pkg.pack_planes(planes5)
dec_p = pkg.pack_decoder(dec, allow_grad=True)
with torch.no_grad():
    rgb5 = pkg.ImportanceRenderer().run_model(planes5, dec, xyz5, None, opts)['rgb']
gen = torch.Generator(device=dev).manual_seed(7)
g_rgb5 = torch.randn((1, n5, 32), device=dev, generator=gen)
g_sig5 = torch.randn((1, n5, 1), device=dev, generator=gen)
g_planes5 = torch.empty_like(pp5.data)
g_dec5 = torch.empty_like(dec_p)
nbytes = L.tpr_run_model_backward_scratch_bytes(1, n5)
scratch5 = torch.empty(nbytes, device=dev, dtype=torch.uint8)


def backward5(with_rgb):
    pkg._lib.check(L.tpr_run_model_backward(P(pp5.data), 1, pp5.height, pp5.width, P(dec_p), P(xyz5), n5, float(opts['box_warp']),
                                            P(rgb5) if with_rgb else None, P(g_rgb5) if with_rgb else None, P(g_sig5), 0,
                                            P(g_planes5), P(g_dec5), P(scratch5), nbytes, ST()), 'tpr_run_model_backward')


if args.roles:
    for with_rgb in (False, True):
        print(f'[roles] config-5 grid, {"rgb + sigma" if with_rgb else "sigma only"}', file=sys.stderr)
        backward5(with_rgb); torch.cuda.synchronize()
    sys.exit(0)

# scatter ceiling, live: the best of the microbenchmark's CTA shapes on a 25 MB (one image's plane gradient) target
B = pkg._lib.bench_lib()
sms = torch.cuda.get_device_properties(0).multi_processor_count
n_lines = 25 * (1 << 20) // 128
buf = torch.zeros(n_lines * 32, device=dev)
ceiling = 0.0
for threads, per_sm in ((256, 1), (512, 1), (1024, 1), (1024, 2)):
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); lines = B.tpr_scatter_microbench(P(buf), n_lines, sms * per_sm, threads, 12, 64, ST()); e1.record()
        torch.cuda.synchronize()
        ceiling = max(ceiling, lines * 128 / e0.elapsed_time(e1) / 1e9)
out['scatter_ceiling_TBps'] = ceiling
del buf

grid = {}
for with_rgb in (False, True):
    ms = timed(lambda: backward5(with_rgb))
    k_ms = kernel_ms(lambda: backward5(with_rgb), 'decode_backward_tc_kernel')
    grid['rgb_sigma' if with_rgb else 'sigma_only'] = {
        'backward_ms': ms, 'G_points_per_s': n5 / ms / 1e6, 'decode_kernel_ms': k_ms,
        'scatter_TBps': n5 * SCATTER_BYTES / k_ms / 1e9, 'fraction_of_scatter_ceiling': n5 * SCATTER_BYTES / k_ms / 1e9 / ceiling}
del g_rgb5, rgb5

# fused vs eager forward + backward at the config-5 grid, sigma only (the density grid of sample_mixed under autograd)
pg5 = planes5.clone().requires_grad_(True)
w5 = torch.randn((1, n5, 1), device=dev, generator=gen)


def fused5():
    pg5.grad = None; dec.zero_grad(set_to_none=True)
    s = pkg.ImportanceRenderer().run_model(pg5, dec, xyz5, None, opts, want_rgb=False)['sigma']
    (s * w5).sum().backward()


def eager5():
    pg5.grad = None
    _, s = TO.decode(TO.gather(pg5, xyz5, opts['box_warp']), dec_raw)
    torch.autograd.grad((s * w5).sum(), [pg5] + list(dec_raw[:4]))


grid['fwd_bwd_sigma_only_fused_ms'] = timed(fused5, reps=5)
torch.cuda.empty_cache()
grid['fwd_bwd_sigma_only_eager_autograd_ms'] = timed(eager5, warm=1, reps=3)
torch.cuda.empty_cache()
grid['points'] = n5
out['config5_grid'] = grid
del pg5, w5, scratch5, g_planes5

# ---- the regulariser shape
n_img = 4
planes_r = torch.randn((n_img, 3, 32, bench.PLANE_RES, bench.PLANE_RES), device=dev,
                       generator=torch.Generator(device=dev).manual_seed(501)).requires_grad_(True)
torch.manual_seed(3)
c = torch.rand((n_img, 1000, 3), device=dev) * 2 - 1
xyz_r = torch.cat([c, c + torch.randn_like(c) * 0.004], 1)


def fused_reg():
    planes_r.grad = None; dec.zero_grad(set_to_none=True)
    s = pkg.ImportanceRenderer().run_model(planes_r, dec, xyz_r, None, opts, want_rgb=False)['sigma']
    (F.l1_loss(s[:, :1000], s[:, 1000:]) * 0.25).backward()


def eager_reg():
    _, s = TO.decode(TO.gather(planes_r, xyz_r, opts['box_warp']), dec_raw)
    torch.autograd.grad(F.l1_loss(s[:, :1000], s[:, 1000:]) * 0.25, [planes_r] + list(dec_raw[:4]))


out['regulariser'] = {'shape': f'{n_img} x (1000 + 1000) points, sigma only, 3x32x256^2 planes',
                      'fwd_bwd_fused_ms': timed(fused_reg, reps=50), 'fwd_bwd_eager_autograd_ms': timed(eager_reg, reps=50)}

# ---- the render backward's decode kernel at config 2, features gathered again (keep_features=False), per sample
planes_h, c2w, K = bench.make_inputs(torch, 100)
planes2 = planes_h.to(dev).requires_grad_(True)
o, d = pkg.RaySampler()(c2w.to(dev), K.to(dev), bench.RES)
R = pkg.ImportanceRenderer(); R.keep_features = False
A2 = torch.randn(o.shape[0], o.shape[1], 32, device=dev)


def render_step():
    planes2.grad = None; dec.zero_grad(set_to_none=True)
    rgb, _, _ = R(planes2, dec, o, d, opts)
    (rgb * A2).sum().backward()


samples = o.shape[0] * o.shape[1] * (bench.DC + bench.DF)
k2 = kernel_ms(render_step, 'decode_backward_tc_kernel')
out['render_backward_decode_kernel_keep_features_false'] = {
    'workload': 'config2: 8 x 128^2 rays x (48+48) samples', 'samples': samples, 'kernel_ms': k2, 'ns_per_sample': k2 * 1e6 / samples,
    'scatter_TBps': samples * SCATTER_BYTES / k2 / 1e9, 'fraction_of_scatter_ceiling': samples * SCATTER_BYTES / k2 / 1e9 / ceiling}
for k in ('sigma_only', 'rgb_sigma'):
    out['config5_grid'][k]['ns_per_point'] = out['config5_grid'][k]['decode_kernel_ms'] * 1e6 / n5
print(json.dumps(out, indent=1))
