"""The deterministic backward (torch.use_deterministic_algorithms(True) -> TPR_BWD_DETERMINISTIC) against the default backward
on one B200, the modes alternated call by call in one process (CUDA events, median):

  * config-2 train step in fp32 (bench.py's workload: 8 x 128^2 rays x (48+48) samples, 256^2 planes, kept samples):
    forward + sum(rgb * A) + backward, and the decode-backward kernel alone (torch.profiler, its own window);
  * EG3D's density regulariser: 4 images x (1000 + 1000 perturbed) points, sigma only: forward + L1 + backward;
  * the config-5 grid (256^3 voxel centres of one identity), sigma only: tpr_run_model_backward alone.

The deterministic mode is timed twice: with torch.utils.deterministic.fill_uninitialized_memory on (torch's default in that
mode: every torch.empty is NaN-filled, the train step's kept samples included) and off.  Measurement script, not product code.
Usage: python profiles/deterministic_backward_timing.py > profiles/r04_deterministic_backward_timing.json"""
import argparse, ctypes, importlib, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F
import torch.utils.deterministic
import bench
pkg = importlib.import_module('g-nerf_b200')
ap = argparse.ArgumentParser(); ap.add_argument('--reps', type=int, default=15)
args = ap.parse_args()
dev = torch.device('cuda:0')
L, P, ST = pkg._lib.lib(), (lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None), \
    (lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
opts = dict(bench.OPTS)
MODES = ('default', 'deterministic', 'deterministic_no_fill')


def set_mode(mode):
    torch.use_deterministic_algorithms(mode != 'default')
    torch.utils.deterministic.fill_uninitialized_memory = mode != 'deterministic_no_fill'


def once(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def alternated(fn, warm=2, reps=args.reps):
    """Median ms per mode; the modes take turns call by call."""
    for mode in MODES:
        set_mode(mode)
        for _ in range(warm): fn()
    torch.cuda.synchronize()
    ts = {m: [] for m in MODES}
    for _ in range(reps):
        for mode in MODES:
            set_mode(mode)
            ts[mode].append(once(fn))
    set_mode('default')
    res = {m: sorted(v)[len(v) // 2] for m, v in ts.items()}
    res['ratio_deterministic'] = res['deterministic'] / res['default']
    res['ratio_deterministic_no_fill'] = res['deterministic_no_fill'] / res['default']
    return res


def kernel_ms(fn, name, mode, reps=5):
    set_mode(mode)
    fn(); torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps): fn()
        torch.cuda.synchronize()
    set_mode('default')
    return sum(e.device_time_total for e in prof.key_averages() if name in e.key) / 1e3 / reps


out = {}
smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
out['gpu'] = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else f'nvidia-smi failed: {smi.stderr.strip()}'
out['reps'] = args.reps
dec = bench.make_decoder(torch, pkg, dev, 0).requires_grad_(True)

# ---- config-2 train step, fp32
planes_h, c2w, K = bench.make_inputs(torch, 100)
planes2 = planes_h.to(dev).requires_grad_(True)
o, d = pkg.RaySampler()(c2w.to(dev), K.to(dev), bench.RES)
R = pkg.ImportanceRenderer()
A2 = torch.randn(o.shape[0], o.shape[1], 32, device=dev, generator=torch.Generator(device=dev).manual_seed(1))


def train_step():
    planes2.grad = None; dec.zero_grad(set_to_none=True)
    rgb, _, _ = R(planes2, dec, o, d, opts)
    (rgb * A2).sum().backward()


step = alternated(train_step)
step['decode_backward_kernel_ms'] = {m: kernel_ms(train_step, 'decode_backward_tc_kernel', m) for m in ('default', 'deterministic')}
step['decode_backward_kernel_ratio'] = step['decode_backward_kernel_ms']['deterministic'] / step['decode_backward_kernel_ms']['default']
step['workload'] = 'config2: 8 x 128^2 rays x (48+48) samples, 3x32x256^2 planes, fp32, forward + backward'
out['config2_train_step_ms'] = step
del planes2, o, d, A2
torch.cuda.empty_cache()

# ---- the regulariser shape
n_img = 4
planes_r = torch.randn((n_img, 3, 32, bench.PLANE_RES, bench.PLANE_RES), device=dev,
                       generator=torch.Generator(device=dev).manual_seed(501)).requires_grad_(True)
torch.manual_seed(3)
c = torch.rand((n_img, 1000, 3), device=dev) * 2 - 1
xyz_r = torch.cat([c, c + torch.randn_like(c) * 0.004], 1)


def regulariser():
    planes_r.grad = None; dec.zero_grad(set_to_none=True)
    s = pkg.ImportanceRenderer().run_model(planes_r, dec, xyz_r, None, opts, want_rgb=False)['sigma']
    (F.l1_loss(s[:, :1000], s[:, 1000:]) * 0.25).backward()


reg = alternated(regulariser, reps=max(args.reps, 50))
reg['workload'] = f'{n_img} x (1000 + 1000) points, sigma only, 3x32x256^2 planes, forward + L1 + backward'
out['regulariser_ms'] = reg
del planes_r

# ---- config-5 grid, sigma only: the C-ABI backward alone (scratch allocated once, so the fill setting does not apply)
g = 256
planes5 = torch.randn((1, 3, 32, bench.PLANE_RES, bench.PLANE_RES), device=dev, generator=torch.Generator(device=dev).manual_seed(500))
ax = (torch.arange(g, device=dev, dtype=torch.float32) + 0.5) / g - 0.5
zz, yy, xx = torch.meshgrid(ax, ax, ax, indexing='ij')
xyz5 = torch.stack([xx, yy, zz], -1).reshape(1, -1, 3).contiguous()
del zz, yy, xx
n5 = g ** 3
pp5 = pkg.pack_planes(planes5)
dec_p = pkg.pack_decoder(dec, allow_grad=True)
g_sig5 = torch.randn((1, n5, 1), device=dev, generator=torch.Generator(device=dev).manual_seed(7))
g_planes5, g_dec5 = torch.empty_like(pp5.data), torch.empty_like(dec_p)
nbytes = L.tpr_run_model_backward_scratch_bytes(1, n5) + L.tpr_backward_deterministic_scratch_bytes(1, pp5.height, pp5.width)
scratch5 = torch.empty(nbytes, device=dev, dtype=torch.uint8)


def backward5():
    flags = pkg._lib.BWD_DETERMINISTIC if torch.are_deterministic_algorithms_enabled() else 0
    pkg._lib.check(L.tpr_run_model_backward(P(pp5.data), 1, pp5.height, pp5.width, P(dec_p), P(xyz5), n5, float(opts['box_warp']),
                                            None, None, P(g_sig5), flags, P(g_planes5), P(g_dec5), P(scratch5), nbytes, ST()),
                   'tpr_run_model_backward')


grid = alternated(backward5)
del grid['deterministic_no_fill'], grid['ratio_deterministic_no_fill']
grid['decode_backward_kernel_ms'] = {m: kernel_ms(backward5, 'decode_backward_tc_kernel', m) for m in ('default', 'deterministic')}
grid['decode_backward_kernel_ratio'] = grid['decode_backward_kernel_ms']['deterministic'] / grid['decode_backward_kernel_ms']['default']
grid['workload'] = '256^3 points of one image, sigma only, 3x32x256^2 planes, tpr_run_model_backward'
out['config5_sigma_backward_ms'] = grid
print(json.dumps(out, indent=1))
