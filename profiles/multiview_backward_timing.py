"""A multi-view training step on one B200: P = 4 identities x F = 8 views, 48+48 samples (the training depths), 256^2 planes,
at 64^2 and 128^2 rays per view, forward + sum(rgb * A) + sum(depth * B) + backward, two ways alternated call by call in one
process (CUDA events, median):

  * frame_batched: the planes tensor [P,3,32,H,W] rendered once for the F*P cameras (plane_sets = P, depth_clamp_group = P,
    channels-first output, as render_frames calls it): one backward scatters every view into the P plane sets;
  * replicated: planes[idx] with N = F*P copies (same rays, noise and upstream gradients, one depth range per frame as
    well): F*P packed copies and plane gradients, summed back by autograd.

Each in the default and the deterministic backward (torch.use_deterministic_algorithms(True)), with the peak memory of one
step (torch.cuda.max_memory_allocated after reset_peak_memory_stats).  Also: the one copy of the channels-first upstream
gradient into the [N,M,32] rows the backward reads (g_rgb.contiguous()), alone.  Measurement script, not product code.
Usage: python profiles/multiview_backward_timing.py > profiles/r05_multiview_backward_timing.json"""
import argparse, importlib, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
pkg = importlib.import_module('g-nerf_b200')
ap = argparse.ArgumentParser(); ap.add_argument('--reps', type=int, default=9)
args = ap.parse_args()
dev = torch.device('cuda:0')
P, F = 4, 8
VARIANTS = ('frame_batched', 'replicated')


def once(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def steps(res, det):
    torch.use_deterministic_algorithms(det)
    planes0, _, _ = bench.make_inputs(torch, 1, n_img=P)
    planes0 = planes0.to(dev)
    c2w, K = bench._camera_utils().orbit_cameras(F * P)
    o, d = pkg.RaySampler()(torch.as_tensor(c2w, device=dev), torch.as_tensor(K, device=dev), res)
    dec = bench.make_decoder(torch, pkg, dev, 2).requires_grad_(True)
    R = pkg.ImportanceRenderer()
    n, m = F * P, res * res
    noise = pkg.frames.draw_frame_noise(F, P, m, 48, 48, dev)
    g = torch.Generator(device=dev).manual_seed(3)
    A = torch.randn((n, m, 32), device=dev, generator=g)
    B = torch.randn((n, m, 1), device=dev, generator=g)
    idx = torch.arange(n, device=dev) % P
    base = dict(bench.OPTS, depth_clamp_group=P)

    def frame_batched():
        planes = planes0.clone().requires_grad_(True)
        rgb, depth, _ = R(planes, dec, o, d, dict(base, output_layout='channels_first'), noise=noise)
        ((rgb * A).sum() + (depth * B).sum()).backward()

    def replicated():
        planes = planes0.clone().requires_grad_(True)
        rgb, depth, _ = R(planes[idx], dec, o, d, base, noise=noise)
        ((rgb * A).sum() + (depth * B).sum()).backward()

    return {'frame_batched': frame_batched, 'replicated': replicated}, (n, m)


def measure(res, det):
    fns, (n, m) = steps(res, det)
    for fn in fns.values():
        fn(); fn()
    torch.cuda.synchronize()
    ts = {v: [] for v in VARIANTS}
    for _ in range(args.reps):
        for v in VARIANTS:
            ts[v].append(once(fns[v]))
    out = {f'{v}_ms': sorted(t)[len(t) // 2] for v, t in ts.items()}
    out.update({f'{v}_ms_min_max': [min(t), max(t)] for v, t in ts.items()})
    for v in VARIANTS:
        torch.cuda.synchronize(); torch.cuda.reset_peak_memory_stats()
        fns[v](); torch.cuda.synchronize()
        out[f'{v}_peak_mb'] = torch.cuda.max_memory_allocated() / 1e6
    out['ratio_replicated_over_batched'] = out['replicated_ms'] / out['frame_batched_ms']
    torch.use_deterministic_algorithms(False)
    return out


def channels_first_copy_ms(res):
    """g_rgb [N,M,32] with the strides of the channels-first output ([N,32,M] memory) -> contiguous, alone."""
    n, m = F * P, res * res
    g = torch.randn((n, 32, m), device=dev).permute(0, 2, 1)
    for _ in range(3): g.contiguous()
    t = sorted(once(lambda: g.contiguous()) for _ in range(21))
    return {'ms': t[len(t) // 2], 'bytes_moved': 2 * n * m * 32 * 4}


out = {'P': P, 'F': F, 'samples': '48+48', 'plane_res': bench.PLANE_RES, 'reps': args.reps}
smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
out['gpu'] = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else f'nvidia-smi failed: {smi.stderr.strip()}'
for res in (64, 128):
    for det in (False, True):
        out[f'{res}x{res}_{"deterministic" if det else "default"}'] = measure(res, det)
    out[f'{res}x{res}_channels_first_grad_copy'] = channels_first_copy_ms(res)
print(json.dumps(out, indent=1))
