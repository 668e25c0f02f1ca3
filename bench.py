#!/usr/bin/env python
"""Benchmark of the tri-plane render hot path (BASELINE.json metric: ray-samples/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mode fp32|bf16] [--legs a,b,...]
                    [--dump-outputs DIR]

A "step" is one ImportanceRenderer.forward over one batch of synthetic input of the BASELINE config-2 shape: 8 images x
128^2 rays x (48 coarse + 48 importance) samples, 3x32x256^2 planes per image, random-init OSGDecoder.  One process per
GPU (torchrun for N > 1); every rank renders its own batch of 8 images (weak scaling) and the rendered features / depth /
weight sums are gathered to every GPU, as BASELINE.json's north_star describes.  Prints ONE JSON line on rank 0.

Besides the headline (`value`, `e2e`, `roofline`) the line carries the other configurations BASELINE.json names, each as
its own object (`--legs` selects them; all are on by default and bounded to seconds):
  cpu_baseline   the UNMODIFIED reference renderer (oracle/_ref) on the host cores: 2 of config 2's 8 images per forward (+ config 1 beside it; N = 1 only)
  gpu_baseline   the UNMODIFIED reference renderer on this GPU, config 2, TF32 off -- SURVEY.md section 8(d)'s "real bar"
  train_step     forward + backward at config 2 (N = 1 only)
  config3        gen_videos.py's 120-frame orbit through the reference TriPlaneGenerator (random init) with the renderer
                 dropped in; backbone / renderer / super-resolution timed separately; one identity per GPU
  config4        batch 32 x 256^2 rays x (96+96) samples, image-sharded, outputs gathered by the render kernel
  config5        256^3 density grid through run_model, point-slab-sharded, sigma all-gathered
  strong         config 2 with the 8 images split over the N GPUs (strong scaling)
  gather_check   N > 1: the in-kernel NVLink gather equals the NCCL all-gather bit for bit, also when consumed a step late
  h2d_ceiling    bare concurrent pinned-memory cudaMemcpyAsync of the e2e path's bytes, no render

`--impl reference` runs the UNMODIFIED reference's ImportanceRenderer.forward (oracle/_ref, the byte-for-byte copy that
oracle/build_ref.py makes of the cited files) on the host cores at the same config-2 workload and prints the same line.
"""
import argparse
import importlib
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_IMG, RES, PLANE_RES, DC, DF = 8, 128, 256, 48, 48
BYTES_PER_SAMPLE = 1536            # 3 planes x 4 taps x 32 channels x 4 B  (SURVEY.md section 8(d))
METRIC = 'ray-samples/sec'
WORKLOAD = 'config2: batch 8 x 128^2 rays x (48+48) samples, 3x32x256^2 fp32 planes/image'
ALL_LEGS = ('cpu_baseline', 'gpu_baseline', 'train_step', 'config3', 'config4', 'config5', 'strong', 'gather_check',
            'h2d_ceiling')
DUMP_MAX_BYTES = 64 << 20

OPTS = {'ray_start': 2.25, 'ray_end': 3.3, 'box_warp': 1, 'depth_resolution': DC, 'depth_resolution_importance': DF,
        'disparity_space_sampling': False, 'clamp_mode': 'softplus'}        # train.py:312-313,328-332


def config_dict(mode, world):
    """The `config` object: identical for the GPU arm and the reference arm of the same command line."""
    return {'workload': WORKLOAD, 'per_gpu_batch': N_IMG, 'rays_per_image': RES * RES, 'samples_per_ray': DC + DF,
            'planes': '3x32x256^2 fp32 per image (N(0,1)), random-init OSGDecoder, cameras on the gen_videos orbit',
            'decoder_precision': mode,
            'parallelism': 'single GPU' if world == 1 else
            f'image-batch sharding x{world} (weak scaling: {N_IMG} images per GPU), outputs gathered to every GPU',
            'l2': 'inputs larger than L2: 201 MB planes + 201 MB repack + 50 MB noise per step (126 MB L2)',
            'step': 'ImportanceRenderer.forward incl. plane repack, decoder pack, both torch.rand draws'}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return json.load(open(p)), 'measured'
    return {'hbm_gbs': 6650.0}, 'fallback'


def ncu_traffic(mode):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the newest committed
    `ncu --set full` summary of this same command (profiles/); None if there is no capture for this mode."""
    tot = None
    for rnd in ('r02', 'r01'):
        path = os.path.join(ROOT, 'profiles', f'{rnd}_render_ws_{mode}_ncu_full_summary.txt')
        if not os.path.exists(path):
            continue
        tot = 0.0
        for line in open(path):
            for key in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                if line.startswith(key):
                    unit = line[line.index('[') + 1:line.index(']')]
                    tot += float(line.split('=')[1]) * {'Mbyte': 1e6, 'Gbyte': 1e9, 'Kbyte': 1e3, 'byte': 1.0}[unit]
        break
    return tot or None


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '20', '-i', str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(',')]))

    def window(self, t0, t1):
        self.t0, self.t1 = t0, t1

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.05)
        self.proc.terminate()
        t0, t1 = getattr(self, 't0', 0.0), getattr(self, 't1', float('inf'))
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.03] or [r for _, r in self.rows[-3:]]
        sm = [float(r[0]) for r in rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        pw = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith('active')})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(pw) if pw else None, 'reasons': reasons, 'samples': len(sm)}


# ----------------------------------------------------------------------------------------------
# synthetic workload (shared by both arms: same seeds, same cameras)
# ----------------------------------------------------------------------------------------------
def _camera_utils():
    """g-nerf_b200/camera_utils.py loaded as a plain file (numpy only): the reference arm must not import the package."""
    spec = importlib.util.spec_from_file_location('_tpr_bench_cameras', os.path.join(ROOT, 'g-nerf_b200', 'camera_utils.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_inputs(torch, seed, n_img=N_IMG, plane_res=PLANE_RES):
    g = torch.Generator(device='cpu').manual_seed(seed)
    planes = torch.randn((n_img, 3, 32, plane_res, plane_res), generator=g, dtype=torch.float32)
    c2w, K = _camera_utils().orbit_cameras(n_img)
    return planes, torch.from_numpy(c2w), torch.from_numpy(K)


def make_decoder(torch, pkg, dev, seed):
    torch.manual_seed(seed)
    return pkg.OSGDecoder(32, {'decoder_lr_mul': 1, 'decoder_output_dim': 32}).to(dev).requires_grad_(False)


def dump_outputs(out_dir, outputs):
    """--dump-outputs: what the last timed step returned -- rgb [N,M,32], depth [N,M,1], weight sum [N,M,1] -- as
    out_dir/<name>.npy in float32, so that two builds can be compared output for output.  Inputs and noise are seeded, so
    the same arguments give the same inputs.  Beyond 64 MB in all (N > 1 gathers every rank's images) every array keeps the
    same fixed, seeded sample of rays, flattened to [rays, channels]."""
    arrays = {name: np.ascontiguousarray(t.detach().cpu().numpy(), dtype=np.float32)
              for name, t in zip(('rgb', 'depth', 'weight_sum'), outputs)}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_MAX_BYTES - 4096                   # room for the .npy headers
    if total > budget:
        rays = arrays['depth'].shape[0] * arrays['depth'].shape[1]
        keep = np.sort(np.random.default_rng(0).choice(rays, rays * budget // total, replace=False))
        arrays = {name: np.ascontiguousarray(a.reshape(rays, -1)[keep]) for name, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


# ----------------------------------------------------------------------------------------------
# the reference on the host cores (bench.py's only uses of oracle/: this arm and the cpu_baseline leg)
# ----------------------------------------------------------------------------------------------
def reference_cpu_forward(torch, n_img, res, seed=100, threads=None):
    """Returns (callable running ONE reference ImportanceRenderer.forward on the CPU, ray-samples per call, threads)."""
    from oracle import ref_loader
    ref = ref_loader.import_reference()
    threads = threads or len(os.sched_getaffinity(0))
    torch.set_num_threads(threads)               # torchrun exports OMP_NUM_THREADS=1; the baseline uses every core it may
    planes, c2w, K = make_inputs(torch, seed, n_img)
    dec = ref_loader.make_decoder(0)
    R = ref.renderer.ImportanceRenderer()
    with torch.no_grad():
        o, d = ref.ray_sampler.RaySampler()(c2w, K, res)

    def fwd(k=n_img):
        with torch.no_grad():
            return R(planes[:k], dec, o[:k], d[:k], dict(OPTS))
    return fwd, res * res * (DC + DF), threads


def run_reference(args):
    """`--impl reference`: the unmodified reference's CPU implementation of the path, all host threads, on this arm's
    config.  A step is one ImportanceRenderer.forward over the 8-image batch; if the host is so slow that K + W such steps
    would take more than ~4 minutes, a step renders the first k of the 8 images instead (stated in `sample`).  With
    --dump-outputs a step always renders all 8, so that the dumped arrays do not depend on the host's speed."""
    if int(os.environ.get('RANK', '0')) != 0:
        return 0
    import torch
    fwd, per_image, threads = reference_cpu_forward(torch, N_IMG, RES)
    t0 = time.perf_counter()
    fwd(1)
    t1 = time.perf_counter() - t0                      # one image, cold: an upper bound of the per-image cost
    budget = 240.0
    k = N_IMG
    while not args.dump_outputs and k > 1 and (args.steps + args.warmup) * k * t1 > budget:
        k //= 2
    for _ in range(args.warmup):
        fwd(k)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        last = fwd(k)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    dt = float(np.mean(times))
    value = k * per_image / dt
    sample = (f'{k} of the {N_IMG} images per step x {RES}^2 rays x ({DC}+{DF}) samples, 3x32x256^2 planes: the unmodified '
              f'reference ImportanceRenderer.forward (oracle/_ref, torch {torch.__version__} CPU, {threads} threads, '
              f'{cpu_model()}); {dt:.2f} s/step')
    base = {'value': value, 'unit': METRIC, 'cores': threads, 'kind': 'reference', 'sample': sample, 'cpu_model': cpu_model()}
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': METRIC, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': config_dict(args.mode, args.gpus), 'cpu_baseline': base,
            'e2e': {'value': value, 'unit': METRIC, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))
    return 0


def leg_cpu_baseline(torch):
    """The unmodified reference on the host's cores, on a bounded sample of THIS workload: the first 2 of config 2's 8 images
    (128^2 rays x 48+48 each) per forward, ~10 s of CPU work in all.  (`--impl reference` runs the same code over more images per
    step; BASELINE config 1 -- 1 image x 64^2 rays, the reference's own CPU-runnable case -- is timed beside it.)"""
    k = 2
    fwd, per_image, threads = reference_cpu_forward(torch, k, RES)
    fwd()
    times = []
    t_end = time.perf_counter() + 12.0
    while len(times) < 10 and (len(times) < 3 or time.perf_counter() < t_end):
        t0 = time.perf_counter()
        fwd()
        times.append(time.perf_counter() - t0)
    dt = float(np.median(times))
    out = {'value': k * per_image / dt, 'unit': METRIC, 'cores': threads, 'kind': 'reference', 'cpu_model': cpu_model(),
           'sample': f'{k} of the {N_IMG} images of config 2 ({RES}^2 rays x ({DC}+{DF}) samples each, 3x32x256^2 planes): the '
                     f'unmodified reference ImportanceRenderer.forward (oracle/_ref, torch {torch.__version__} CPU, {threads} '
                     f'threads); median of {len(times)} forwards, {dt:.3f} s each'}
    try:
        fwd1, per1, _ = reference_cpu_forward(torch, 1, 64)
        fwd1()
        t1 = []
        for _ in range(5):
            t0 = time.perf_counter()
            fwd1()
            t1.append(time.perf_counter() - t0)
        out['config1'] = {'value': per1 / float(np.median(t1)), 'unit': METRIC,
                          'sample': f'BASELINE config 1: 1 image x 64^2 rays x ({DC}+{DF}) samples; median of 5 forwards, '
                                    f'{float(np.median(t1)):.3f} s each'}
    except Exception as e:       # noqa: BLE001
        out['config1'] = {'error': str(e)[:200]}
    return out


def bind_to_gpu_numa_node(torch, index):
    """Pin this process to the CPU cores of the NUMA node its GPU hangs off, so that the pinned host buffers of the e2e path
    are allocated next to the GPU's PCIe root (torchrun does not bind ranks).  Returns the node, or None if unknown."""
    try:
        p = torch.cuda.get_device_properties(index)
        dev = f'{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0'
        node = int(open(f'/sys/bus/pci/devices/{dev}/numa_node').read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            lo, _, hi = part.partition('-')
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------
# GPU arm: helpers
# ----------------------------------------------------------------------------------------------
class Ctx:
    """What every leg needs: torch, the package, device, rank / world, barrier and max-over-ranks."""

    def __init__(self, torch, dist, pkg, dev, rank, world, args):
        self.torch, self.dist, self.pkg, self.dev, self.rank, self.world, self.args = torch, dist, pkg, dev, rank, world, args

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return list(vals)
        t = self.torch.tensor(vals, device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def all_ok(self, ok):
        """Every rank reached this point in a state to run a collective leg?"""
        if self.world == 1:
            return bool(ok)
        t = self.torch.tensor([1.0 if ok else 0.0], device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item() > 0.5)

    def time_steps(self, fn, steps, warmup=3):
        """ms per call of fn: warm-up, barrier + synchronize on both sides, CUDA events, max over ranks."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1) / steps)[0]


def l2_gather_ceiling(cx):
    """Random-128-byte-line gather bandwidth with the working set in L2 (one image's 25 MB of planes), measured NOW on this GPU
    with the render kernels' access shape (8 lanes x LDG.128 per line): the ceiling SURVEY.md section 8(d) asks to report the
    gather against.  tpr_gather_microbench_ex (libtriplane_b200_bench.so); best cell of a small warps x lines-in-flight sweep."""
    import ctypes
    torch = cx.torch
    L = cx.pkg._lib.bench_lib()
    n_lines = 25 * (1 << 20) // 128
    buf = torch.randn(n_lines * 32, device=cx.dev)
    sink = torch.empty(65536, device=cx.dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    best, cells = 0.0, {}
    for threads, fl in ((1024, 4), (1024, 6), (768, 4), (512, 4)):
        top = 0.0
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            lines = L.tpr_gather_microbench_ex(ctypes.c_void_p(buf.data_ptr()), n_lines, 148, threads, fl, 1200 // fl,
                                               ctypes.c_void_p(sink.data_ptr()), st)
            e1.record()
            torch.cuda.synchronize()
            if lines <= 0:
                raise RuntimeError(f'tpr_gather_microbench_ex failed: {lines}')
            top = max(top, lines * 128 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        cells[f'{threads // 32}warps_x_{fl}inflight'] = round(top, 1)
        best = max(best, top)
    return best, cells


# ----------------------------------------------------------------------------------------------
# legs
# ----------------------------------------------------------------------------------------------
def leg_gpu_baseline(cx, planes, origins, dirs):
    """SURVEY.md section 8(d) "GPU baseline (the real bar)": the unmodified reference renderer on this GPU, config 2, fp32 with
    TF32 off as the reference sets it (training_loop.py:145-146), same timing protocol."""
    torch = cx.torch
    from oracle import ref_loader
    ref = ref_loader.import_reference()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dec = ref_loader.make_decoder(0).to(cx.dev)
    R = ref.renderer.ImportanceRenderer()

    def fwd():
        with torch.no_grad():
            return R(planes, dec, origins, dirs, dict(OPTS))
    torch.cuda.reset_peak_memory_stats()
    ms = cx.time_steps(fwd, steps=10, warmup=3)
    samples = N_IMG * RES * RES * (DC + DF)
    return {'ms_per_step': ms, 'value': samples / (ms * 1e-3), 'unit': METRIC, 'steps': 10, 'warmup': 3, 'tf32': False,
            'peak_mem_GB': torch.cuda.max_memory_allocated() / 1e9, 'torch': torch.__version__,
            'what': 'the unmodified reference ImportanceRenderer.forward (oracle/_ref, ~40 ATen launches) on this GPU, '
                    'config 2, same inputs'}


def leg_train_step(cx, planes, origins, dirs, opts):
    torch, pkg = cx.torch, cx.pkg
    m = RES * RES
    renderer = pkg.ImportanceRenderer()
    planes_g = planes.detach().clone().requires_grad_(True)
    dec_g = make_decoder(torch, pkg, cx.dev, seed=0).requires_grad_(True)
    ups = (torch.randn(N_IMG, m, 32, device=cx.dev), torch.randn(N_IMG, m, 1, device=cx.dev), torch.randn(N_IMG, m, 1, device=cx.dev))

    def train_step():
        planes_g.grad = None
        for prm in dec_g.parameters():
            prm.grad = None
        torch.autograd.backward(renderer(planes_g, dec_g, origins, dirs, opts), ups)
    n_train = max(3, min(cx.args.steps, 10))
    ms = cx.time_steps(train_step, n_train, warmup=3)
    return {'ms_per_step': ms, 'value': N_IMG * m * (DC + DF) / (ms * 1e-3), 'unit': METRIC, 'steps': n_train,
            'what': 'ImportanceRenderer.forward + backward (gradients of planes and the four decoder tensors), '
                    'inputs resident in HBM; forward as above, backward = tpr_render_backward'}


class SharedHostOutputs:
    """N > 1: ONE host buffer for the whole job's outputs (a POSIX shared-memory file mapped by every rank and registered with
    CUDA as pinned memory); rank r's device -> host copies land in slice r, so that after the step's barrier the gathered
    [world * N_IMG, M, 32 | 1 | 1] result sits in host memory that rank 0 -- the caller -- reads.  No extra copy: the gather is
    where the D2H copies point."""

    def __init__(self, cx, n_img, m):
        import mmap
        torch = cx.torch
        self.cx, self.torch = cx, torch
        self.path = f'/dev/shm/tpr_bench_{os.environ.get("MASTER_PORT", "0")}'
        shapes = [(cx.world * n_img, m, c) for c in (32, 1, 1)]
        sizes = [int(np.prod(sh)) * 4 for sh in shapes]
        total = sum(sizes)
        if cx.rank == 0:
            with open(self.path, 'wb') as f:
                f.truncate(total)
        cx.barrier()
        self.fd = os.open(self.path, os.O_RDWR)
        self.mm = mmap.mmap(self.fd, total)
        whole = torch.from_numpy(np.frombuffer(self.mm, dtype=np.float32))
        rc = torch.cuda.cudart().cudaHostRegister(whole.data_ptr(), total, 0)
        if int(rc) != 0:
            raise RuntimeError(f'cudaHostRegister failed: {rc}')
        self.whole = whole
        self.all, off = [], 0
        for sh, sz in zip(shapes, sizes):
            self.all.append(whole[off // 4:(off + sz) // 4].view(sh))
            off += sz
        self.mine = tuple(t[cx.rank * n_img:(cx.rank + 1) * n_img] for t in self.all)      # contiguous slices
        cx.barrier()
        if cx.rank == 0:
            os.unlink(self.path)                     # mapped everywhere by now: the name can go

    def close(self):
        self.torch.cuda.synchronize()
        self.torch.cuda.cudart().cudaHostUnregister(self.whole.data_ptr())
        self.mine = self.all = self.whole = None
        try:
            self.mm.close()
        except BufferError:                          # (a numpy view still alive: the mapping goes with the process)
            pass
        os.close(self.fd)


def leg_h2d_ceiling(cx, planes_pin, out_pin):
    """Bare concurrent copies of the e2e path's bytes (pinned host -> device of this rank's planes, device -> pinned host of
    its outputs), all ranks at once, nothing rendered: what the host can feed N GPUs."""
    torch = cx.torch
    dst = torch.empty(planes_pin.shape, device=cx.dev)
    src = tuple(torch.empty(t.shape, device=cx.dev) for t in out_pin)
    s_out = torch.cuda.Stream()

    def copies():
        dst.copy_(planes_pin, non_blocking=True)
        s_out.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s_out):
            for h, d in zip(out_pin, src):
                h.copy_(d, non_blocking=True)
        torch.cuda.current_stream().wait_stream(s_out)
    ms = cx.time_steps(copies, steps=5, warmup=2)
    h2d = planes_pin.numel() * 4
    return {'ms_per_step': ms, 'h2d_GBps_per_gpu': h2d / (ms * 1e-3) / 1e9, 'h2d_GBps_aggregate': cx.world * h2d / (ms * 1e-3) / 1e9,
            'what': f'{cx.world} rank(s) x concurrent cudaMemcpyAsync of {h2d / 1e6:.0f} MB pinned planes in + outputs back, no render'}


def leg_gather_check(cx, renderer, planes, decoder, origins, dirs, opts, peer):
    """N > 1 correctness under the driver: the render kernel's NVLink peer stores deliver exactly what render + NCCL
    all-gather delivers, on every buffer set, also when a step's outputs are consumed one call late (the lifetime contract
    of parallel.PeerGather) with this rank delayed."""
    torch, P = cx.torch, cx.pkg.parallel
    n, m = origins.shape[:2]
    ok, detail = True, []
    held = None
    for step in range(4):
        g = torch.Generator(device=cx.dev).manual_seed(1000 + 17 * step + cx.rank)
        noise = (torch.rand((n, m, DC, 1), device=cx.dev, generator=g), torch.rand((n * m, DF), device=cx.dev, generator=g))
        want = tuple(t.clone() for t in P.render_sharded(renderer, planes, decoder, origins, dirs, opts, noise=noise))
        got = P.render_sharded(renderer, planes, decoder, origins, dirs, opts, noise=noise, peer=peer)
        same = all(torch.equal(a, b) for a, b in zip(got, want))
        if cx.rank % 2 == 1:
            torch.cuda._sleep(10_000_000)              # odd ranks fall ~5 ms behind their peers
        late = True
        if held is not None:
            late = all(torch.equal(a, b) for a, b in zip(*held))       # step-1's outputs, read after this step's exchange
        held = (got, want)
        ok = ok and same and late
        detail.append((same, late))
    torch.cuda.synchronize()
    return cx.all_ok(ok), detail


def leg_strong(cx, decoder, opts):
    """Config 2 with its 8 images split over the N GPUs (strong scaling): 8 / N images per GPU, outputs gathered by the
    render kernel."""
    torch, pkg = cx.torch, cx.pkg
    if N_IMG % cx.world != 0:
        return {'unavailable': f'{N_IMG} images do not split evenly over {cx.world} GPUs'}
    n_local = N_IMG // cx.world
    planes_h, c2w, K = make_inputs(torch, 100)                       # the SAME 8 images whatever N is
    sl = slice(cx.rank * n_local, (cx.rank + 1) * n_local)
    planes = planes_h[sl].to(cx.dev)
    o, d = pkg.RaySampler()(c2w[sl].to(cx.dev), K[sl].to(cx.dev), RES)
    renderer = pkg.ImportanceRenderer()
    peer = pkg.parallel.PeerGather(n_local, RES * RES)
    try:
        ms = cx.time_steps(lambda: pkg.parallel.render_sharded(renderer, planes, decoder, o, d, opts, peer=peer),
                           steps=max(5, min(cx.args.steps, 20)), warmup=3)
    finally:
        peer.close()
    total = N_IMG * RES * RES * (DC + DF)
    return {'ms_per_step': ms, 'value': total / (ms * 1e-3), 'unit': METRIC, 'images_per_gpu': n_local, 'scaling': 'strong',
            'what': 'config 2, 8 images in total; every GPU ends up with all 8 rendered images'}


def leg_config4(cx, decoder, mode):
    """BASELINE configs[3]: batch 32 x 256^2 rays x (96+96) samples -- the depths gen_videos.py:127-128 really renders with --
    image-sharded over the N GPUs (32 / N images each), rendered features / depth gathered to every GPU by the kernel."""
    torch, pkg = cx.torch, cx.pkg
    total_img, res, dc, df = 32, 256, 96, 96
    if total_img % cx.world != 0:
        return {'unavailable': f'{total_img} images do not split evenly over {cx.world} GPUs'}
    n_local = total_img // cx.world
    g = torch.Generator(device=cx.dev).manual_seed(400 + cx.rank)
    planes = torch.randn((n_local, 3, 32, PLANE_RES, PLANE_RES), device=cx.dev, generator=g)
    cams = _camera_utils()
    c2w, K = cams.orbit_cameras(total_img)
    sl = slice(cx.rank * n_local, (cx.rank + 1) * n_local)
    o, d = pkg.RaySampler()(torch.from_numpy(c2w[sl]).to(cx.dev), torch.from_numpy(K[sl]).to(cx.dev), res)
    opts = dict(OPTS, depth_resolution=dc, depth_resolution_importance=df, decoder_precision=mode)
    renderer = pkg.ImportanceRenderer()
    peer = pkg.parallel.PeerGather(n_local, res * res) if cx.world > 1 else None
    kernel_events = []

    def step(record=False):
        if record:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            renderer._timing_events = ev
            kernel_events.append(ev)
        if peer is not None:
            out = pkg.parallel.render_sharded(renderer, planes, decoder, o, d, opts, peer=peer)
        else:
            out = renderer(planes, decoder, o, d, opts)
        renderer._timing_events = None
        return out
    try:
        for _ in range(2):
            step()
        cx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = 4
        e0.record()
        for _ in range(steps):
            step(record=True)
        e1.record()
        cx.barrier()
        ms = e0.elapsed_time(e1) / steps
        kern = float(np.mean([a.elapsed_time(b) for a, b in kernel_events]))
        ms, kern = cx.max_over_ranks(ms, kern)
    finally:
        if peer is not None:
            peer.close()
    total = total_img * res * res * (dc + df)
    per_gpu = n_local * res * res * (dc + df)
    return {'workload': 'config4: batch 32 x 256^2 rays x (96+96) samples', 'ms_per_step': ms, 'value': total / (ms * 1e-3),
            'unit': METRIC, 'images_per_gpu': n_local, 'scaling': 'strong', 'kernel_ms': kern,
            'per_gpu_value': per_gpu / (ms * 1e-3), 'kernel_GBps_algorithmic': per_gpu * BYTES_PER_SAMPLE / (kern * 1e-3) / 1e9,
            'gather': 'render kernel peer stores + 2-float all-reduce' if peer is not None else 'single GPU', 'steps': steps}


def leg_config5(cx, decoder, mode):
    """BASELINE configs[4]: the 256^3 density grid of gen_videos.py:33-55,189-209 (sample_mixed -> run_model, sigma only), cut
    into contiguous z-slabs over the N GPUs (parallel.run_model_sharded), sigma all-gathered."""
    torch, pkg = cx.torch, cx.pkg
    g = 256
    planes = torch.randn((1, 3, 32, PLANE_RES, PLANE_RES), device=cx.dev, generator=torch.Generator(device=cx.dev).manual_seed(500))
    # create_samples (gen_videos.py:33-55): voxel centres of a cube of side box_warp, x fastest, z slowest
    ax = (torch.arange(g, device=cx.dev, dtype=torch.float32) + 0.5) / g - 0.5
    zz, yy, xx = torch.meshgrid(ax, ax, ax, indexing='ij')
    xyz = torch.stack([xx, yy, zz], -1).reshape(1, -1, 3).contiguous()
    del zz, yy, xx
    opts = dict(OPTS, decoder_precision=mode)
    renderer = pkg.ImportanceRenderer()
    pp = pkg.pack_planes(planes)                                       # packed once per identity (the plane cache)

    def query():
        return pkg.parallel.run_model_sharded(renderer, pp, decoder, xyz, None, opts, want_rgb=False)
    ms = cx.time_steps(query, steps=10, warmup=3)
    ms_local = cx.time_steps(lambda: pkg.parallel.run_model_sharded(renderer, pp, decoder, xyz, None, opts, gather=False),
                             steps=10, warmup=2)
    pts = g ** 3
    return {'workload': 'config5: 256^3 sample_mixed queries (sigma only), z-slab sharded', 'ms_per_step': ms,
            'value': pts / (ms * 1e-3), 'unit': 'points/sec', 'points_per_gpu': pts // cx.world, 'scaling': 'strong',
            'ms_query_only': ms_local, 'GBps_algorithmic': pts * BYTES_PER_SAMPLE / (ms * 1e-3) / 1e9,
            'gather': 'in-place NCCL all-gather of sigma (4 B/point)' if cx.world > 1 else 'single GPU'}


class _Split:
    """CUDA-event time spent inside each of a set of modules' __call__ (forward pre / post hooks on this stream)."""

    def __init__(self, torch, mods):
        self.torch, self.ev, self.handles = torch, {k: [] for k in mods}, []
        for name, m in mods.items():
            self.handles.append(m.register_forward_pre_hook(lambda mod, a, _n=name: self._start(_n)))
            self.handles.append(m.register_forward_hook(lambda mod, a, out, _n=name: self._stop(_n)))

    def _start(self, name):
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev[name].append([e, None])

    def _stop(self, name):
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev[name][-1][1] = e

    def reset(self):
        for k in self.ev:
            self.ev[k] = []

    def totals(self):
        self.torch.cuda.synchronize()
        return {k: float(sum(a.elapsed_time(b) for a, b in v if b is not None)) for k, v in self.ev.items()}

    def remove(self):
        for h in self.handles:
            h.remove()


def leg_config3(cx, frames=120, res=64):
    """BASELINE configs[2]: the gen_videos.py:147-171 loop -- 120-frame orbit of one identity through the reference's
    TriPlaneGenerator (random init, FFHQ shape, 512^2 super-resolution head; depths doubled to 96+96 as gen_videos.py:127-128
    does) -- one identity per GPU.  Four ways, backbone / renderer / super-resolution timed separately with CUDA events:
      stock        the unmodified reference, its own renderer (~40 ATen launches per frame)
      drop_in      install(): the reference's loop untouched, ImportanceRenderer / RaySampler replaced by the sm_100a kernels
      plane_cache  + launch.py's default: backbone and plane repack once per identity (the loop re-runs them per frame)
      batched      frames.synthesize_frames: backbone once, all 120 frames in ONE renderer call, then the SR head per frame
    The reference's backbone and super-resolution stay on the reference path (its own bias_act / upfirdn2d plugins)."""
    torch, pkg = cx.torch, cx.pkg
    from oracle import ref_loader
    ref = ref_loader.import_reference()
    torch.backends.cuda.matmul.allow_tf32 = False          # training_loop.py:145-146
    torch.backends.cudnn.allow_tf32 = False
    pkg.enable_reference_plugins()                        # the reference's bias_act / upfirdn2d JIT plugins under torch 2.x
    G = ref_loader.make_generator(seed=10 + cx.rank).to(cx.dev)
    G.rendering_kwargs['depth_resolution'] = int(G.rendering_kwargs['depth_resolution'] * 2)                  # gen_videos.py:127
    G.rendering_kwargs['depth_resolution_importance'] = int(G.rendering_kwargs['depth_resolution_importance'] * 2)   # :128
    dc, df = G.rendering_kwargs['depth_resolution'], G.rendering_kwargs['depth_resolution_importance']
    LookAt = ref.camera_utils.LookAtPoseSampler
    intr = torch.tensor([[4.2647, 0, 0.5], [0, 4.2647, 0.5], [0, 0, 1]], device=cx.dev)                      # gen_videos.py:135
    z = torch.randn((1, 512), generator=torch.Generator().manual_seed(20 + cx.rank)).to(cx.dev)   # stands for E(id_image), :131
    pose_s = LookAt.sample(3.14 / 2, 3.14 / 2, radius=G.rendering_kwargs['avg_camera_radius'], device=cx.dev)
    c_s = torch.cat([pose_s.reshape(-1, 16), intr.reshape(-1, 9)], 1)
    with torch.no_grad():
        ws = G.mapping(z=z, c=torch.zeros_like(c_s))                                                         # :150

    def pose(i):                                                                                              # :155-158
        return LookAt.sample(3.14 / 2 + 0.7 * np.sin(2 * 3.14 * i / frames), 3.14 / 2 - 0.05 + 0.3 * np.cos(2 * 3.14 * i / frames),
                             radius=G.rendering_kwargs['avg_camera_radius'], device=cx.dev)

    def frame_loop(n):
        """gen_videos.py:153-178: per frame a pose, G.synthesis, uint8 conversion and the copy to the host."""
        with torch.no_grad():
            for i in range(n):
                c_d = torch.cat([pose(i).reshape(-1, 16), intr.reshape(-1, 9)], 1)
                out = G.synthesis(ws=ws, c=c_d, noise_mode='const', neural_rendering_resolution=res)          # :171
                (out['image'] * 127.5 + 128).clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).cpu()          # :173
                (out['image_raw'] * 127.5 + 128).clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).cpu()      # :174

    split = _Split(torch, {'backbone': G.backbone.synthesis, 'renderer': G.renderer, 'superresolution': G.superresolution})
    per_frame = res * res * (dc + df)
    out = {'workload': f'config3: {frames}-frame gen_videos orbit, 1 identity per GPU, {res}^2 rays x ({dc}+{df}) samples, 512^2 SR',
           'frames': frames, 'ray_samples_per_frame': per_frame}

    def timed(run, name, extra_renderer_events=None):
        run(4)                                             # warm-up: plugin JIT / cuDNN autotune / allocator
        cx.barrier()
        split.reset()
        if extra_renderer_events is not None:
            extra_renderer_events.clear()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        run(frames)
        e1.record()
        cx.barrier()
        wall = (time.perf_counter() - t0) * 1e3
        tot = split.totals()
        if extra_renderer_events is not None:
            tot['renderer'] = float(sum(a.elapsed_time(b) for a, b in extra_renderer_events))
        ms = e0.elapsed_time(e1)
        ms, wall, bb, rr, sr = cx.max_over_ranks(ms, wall, tot['backbone'], tot['renderer'], tot['superresolution'])
        out[name] = {'orbit_ms': ms, 'orbit_wall_ms': wall, 'backbone_ms': bb, 'renderer_ms': rr, 'superresolution_ms': sr,
                     'other_ms': ms - bb - rr - sr, 'frames_per_s': cx.world * frames / (wall * 1e-3),
                     'renderer_ray_samples_per_s': cx.world * frames * per_frame / (rr * 1e-3) if rr > 0 else None}

    try:
        timed(frame_loop, 'stock')
        pkg.install()
        try:
            timed(frame_loop, 'drop_in')
            pkg.enable_plane_cache(G)
            timed(frame_loop, 'plane_cache')
            pkg.disable_plane_cache(G)
            # batched: poses built on the host once (camera_utils.orbit_cameras mirrors gen_videos.py:155-158), one renderer call
            cams = _camera_utils()
            c2w_all = torch.from_numpy(cams.orbit_cameras(frames, frames=frames)[0]).to(cx.dev)
            rf_events = []
            real_rf = pkg.frames.render_frames

            def timed_rf(*a, **k):
                ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                ev[0].record()
                r = real_rf(*a, **k)
                ev[1].record()
                rf_events.append(ev)
                return r

            def batched(n):
                with torch.no_grad():
                    pkg.frames.render_frames = timed_rf
                    try:
                        fr = pkg.synthesize_frames(G, ws, c2w_all[:n], intr, res, noise_mode='const')
                    finally:
                        pkg.frames.render_frames = real_rf
                    for f in fr:
                        (f['image'] * 127.5 + 128).clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).cpu()
                        (f['image_raw'] * 127.5 + 128).clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).cpu()
            timed(batched, 'batched', extra_renderer_events=rf_events)
        finally:
            pkg.uninstall()
    finally:
        split.remove()
    out['renderer_speedup_vs_stock'] = {k: out['stock']['renderer_ms'] / out[k]['renderer_ms'] for k in ('drop_in', 'plane_cache', 'batched')}
    out['orbit_speedup_vs_stock'] = {k: out['stock']['orbit_wall_ms'] / out[k]['orbit_wall_ms'] for k in ('drop_in', 'plane_cache', 'batched')}
    out['note'] = ('value of each object: max over ranks; frames_per_s is the aggregate of all ranks (one identity each). '
                   'other_ms = pose construction, ray sampling, uint8 conversion and the per-frame copies to the host '
                   '(gen_videos.py:155-178)')
    return out


def merge_config3(per_rank):
    """Ranks ran the orbit concurrently, one identity each: times = max over ranks, rates = the whole job's."""
    errs = [r['error'] for r in per_rank if 'error' in r]
    if errs:
        return {'error': errs[0], 'ranks_failed': len(errs)}
    out = dict(per_rank[0])
    world = len(per_rank)
    for name in ('stock', 'drop_in', 'plane_cache', 'batched'):
        o = {}
        for k in ('orbit_ms', 'orbit_wall_ms', 'backbone_ms', 'renderer_ms', 'superresolution_ms', 'other_ms'):
            o[k] = max(r[name][k] for r in per_rank)
        o['frames_per_s'] = world * out['frames'] / (o['orbit_wall_ms'] * 1e-3)
        o['renderer_ray_samples_per_s'] = world * out['frames'] * out['ray_samples_per_frame'] / (o['renderer_ms'] * 1e-3)
        out[name] = o
    out['renderer_speedup_vs_stock'] = {k: out['stock']['renderer_ms'] / out[k]['renderer_ms'] for k in ('drop_in', 'plane_cache', 'batched')}
    out['orbit_speedup_vs_stock'] = {k: out['stock']['orbit_wall_ms'] / out[k]['orbit_wall_ms'] for k in ('drop_in', 'plane_cache', 'batched')}
    out['identities'] = world
    return out


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--mode', default='fp32', choices=['fp32', 'bf16', 'fp32_ffma'])
    ap.add_argument('--legs', default='all', help='comma-separated subset of ' + ','.join(ALL_LEGS) + ' (or all / none)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-train-step', action='store_true', help='skip the forward+backward timing (N = 1 only)')
    ap.add_argument('--gather', default='peer', choices=['peer', 'nccl'],
                    help='N > 1: peer = the render kernel stores into every GPU\'s gather buffers over NVLink; '
                         'nccl = render, then an in-place all-gather (A/B)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the rgb / depth / weight sum of the last timed step to DIR/<name>.npy (float32, at most '
                         '64 MB in all: a fixed, seeded sample of rays beyond that)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)
    legs = set(ALL_LEGS) if args.legs == 'all' else set() if args.legs == 'none' else set(args.legs.split(','))
    unknown = legs - set(ALL_LEGS)
    if unknown:
        raise SystemExit(f'unknown legs: {sorted(unknown)}')
    if args.no_cpu_baseline:
        legs.discard('cpu_baseline')
    if args.no_train_step:
        legs.discard('train_step')

    import torch
    import torch.distributed as dist
    pkg = importlib.import_module('g-nerf_b200')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: the renderer has no CPU path')
    # stdout carries the ONE JSON line and nothing else: libraries that print there (NCCL's version banner) go to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(torch, local)       # before any pinned allocation: first touch decides the node
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    cx = Ctx(torch, dist, pkg, dev, rank, world, args)
    warmup = max(args.warmup, 3)

    planes_h, c2w_h, K_h = make_inputs(torch, seed=100 + rank)
    decoder = make_decoder(torch, pkg, dev, seed=0)
    renderer, sampler = pkg.ImportanceRenderer(), pkg.RaySampler()
    opts = dict(OPTS, decoder_precision=args.mode)
    planes = planes_h.to(dev)
    origins, dirs = sampler(c2w_h.to(dev), K_h.to(dev), RES)
    m = RES * RES
    samples_per_step = N_IMG * m * (DC + DF)

    kernel_events = []
    peer = pkg.parallel.PeerGather(N_IMG, m) if world > 1 and args.gather == 'peer' else None

    def step(record=False):
        """The hot path as a user calls it, inputs resident in HBM.  N > 1: every rank renders its batch into
        its slice of EVERY rank's gather buffers (peer stores in the render kernel's epilogue), the depth range is
        all-reduced (which also completes the exchange) and the gathered depths are clamped."""
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            renderer._timing_events = (e0, e1)
            kernel_events.append((e0, e1))
        if world > 1:
            out = pkg.parallel.render_sharded(renderer, planes, decoder, origins, dirs, opts, peer=peer)
        else:
            out = renderer(planes, decoder, origins, dirs, opts)
        renderer._timing_events = None
        return out

    sampler_clk = ClockSampler(local)
    if rank == 0:
        sampler_clk.start()              # nvidia-smi needs ~100 ms to start: begin before the warm-up
    for _ in range(warmup):
        step()
    cx.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cx.barrier()
    t_wall0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        last = step(record=True)
    ev1.record()
    cx.barrier()
    sampler_clk.window(t_wall0, time.time())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    ms = ev0.elapsed_time(ev1) / args.steps
    clocks = sampler_clk.stop() if rank == 0 else None
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in kernel_events]))

    # ---- end to end: the forward with HOST buffers (ImportanceRenderer.forward_host -> tpr_render_host): every step
    # copies that step's planes and rays from pinned host memory and reads rgb / depth / weight sums back to the host
    planes_pin, o_pin, d_pin = planes_h.pin_memory(), origins.cpu().pin_memory(), dirs.cpu().pin_memory()
    shared_out = SharedHostOutputs(cx, N_IMG, m) if world > 1 else None
    out_pin = shared_out.mine if world > 1 else tuple(torch.empty((N_IMG, m, c), dtype=torch.float32).pin_memory() for c in (32, 1, 1))
    h2d = planes_pin.numel() * 4 + o_pin.numel() * 4 + d_pin.numel() * 4
    d2h = sum(t.numel() * 4 for t in out_pin)

    def e2e_step():
        if world == 1:
            renderer.forward_host(planes_pin, decoder, o_pin, d_pin, opts, out=out_pin)
            return
        # N > 1: the same per-image pipeline; the depth clamp needs the all-reduced range, so depth leaves the device last
        renderer.forward_host(planes_pin, decoder, o_pin, d_pin, opts, out=out_pin, defer_depth=True)
        rng = renderer.last_depth_range
        lo, hi = rng[0:1].clone(), rng[1:2].clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        renderer.finish_host_depth(torch.cat([lo, hi]))

    e2e_steps = max(3, min(args.steps, 10))
    e2e_ms = cx.time_steps(e2e_step, e2e_steps, warmup=2)
    e2e_gathered = None
    if world > 1:
        # the gathered result is in rank 0's address space: the file starts zero-filled, so finite non-zero data in EVERY rank's
        # slice, seen from rank 0, is every rank's D2H copies having landed in the one buffer
        cx.barrier()
        filled = True
        if rank == 0:
            for r in range(world):
                for t in shared_out.all:
                    sl = t[r * N_IMG:(r + 1) * N_IMG]
                    filled = filled and bool(torch.isfinite(sl).all()) and float(sl.abs().max()) > 0.0
        e2e_gathered = cx.all_ok(filled)
    ms, kern_ms = cx.max_over_ranks(ms, kern_ms)

    # ---- the other configurations / baselines, each bounded to seconds; a failing leg reports its error, never kills the line
    extra = {}

    def run_leg(name, fn, collective=False):
        if name not in legs:
            return
        try:
            extra[name] = fn()
        except Exception as e:       # noqa: BLE001
            if collective and world > 1:
                raise                # the ranks would deadlock on the next collective: fail the run loudly instead
            extra[name] = {'error': f'{type(e).__name__}: {e}'[:400]}

    if world > 1:
        run_leg('gather_check', lambda: dict(zip(('ok', 'per_step_same_and_late'),
                                                 leg_gather_check(cx, renderer, planes, decoder, origins, dirs, opts, peer)))
                if peer is not None else {'unavailable': '--gather nccl'}, collective=True)
    run_leg('h2d_ceiling', lambda: leg_h2d_ceiling(cx, planes_pin, out_pin), collective=True)
    if peer is not None:
        peer.close()
        peer = None
    if shared_out is not None:
        out_pin = None
        shared_out.close()
    if world == 1:
        run_leg('train_step', lambda: leg_train_step(cx, planes, origins, dirs, opts) if args.mode != 'fp32_ffma'
                else {'unavailable': 'fp32_ffma'})
        run_leg('gpu_baseline', lambda: leg_gpu_baseline(cx, planes, origins, dirs))
    del planes, planes_pin
    torch.cuda.empty_cache()
    if world > 1:
        run_leg('strong', lambda: leg_strong(cx, decoder, opts), collective=True)
    run_leg('config4', lambda: leg_config4(cx, decoder, args.mode), collective=True)
    torch.cuda.empty_cache()
    run_leg('config5', lambda: leg_config5(cx, decoder, args.mode), collective=True)
    torch.cuda.empty_cache()
    if 'config3' in legs:
        # One identity per GPU, no data-path collective: every rank times its own orbit with LOCAL synchronisation only (the
        # reference's plugins JIT-compile on first use; a rank that fails must not leave the others waiting in a collective),
        # then ONE all_gather_object that every rank reaches, whatever happened, merges the ranks (max of the times).
        try:
            res3 = leg_config3(Ctx(torch, dist, pkg, dev, rank, 1, args))
        except Exception as e:       # noqa: BLE001
            res3 = {'error': f'rank {rank}: {type(e).__name__}: {e}'[:400]}
        if world > 1:
            allr = [None] * world
            dist.all_gather_object(allr, res3)
            res3 = merge_config3(allr)
        extra['config3'] = res3

    if rank == 0:
        pk, pk_kind = peaks()
        value = world * samples_per_step / (ms * 1e-3)
        achieved = samples_per_step * BYTES_PER_SAMPLE / (kern_ms * 1e-3) / 1e9
        try:
            l2_peak, l2_cells = l2_gather_ceiling(cx)
            l2_kind = 'measured live (tpr_gather_microbench_ex, 25 MB working set, one CTA per SM)'
        except Exception as e:       # noqa: BLE001
            l2_peak, l2_cells, l2_kind = 16590.3, None, f'profiles/r01_gather_roofline.json (live measurement failed: {e})'
        line = {
            'metric': METRIC, 'value': value, 'unit': METRIC, 'n_gpus': world, 'steps': args.steps, 'warmup': warmup,
            'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16-mlp' if args.mode == 'bf16' else 'f32', 'data': 'synthetic',
            'config': config_dict(args.mode, world),
            'roofline': {'bound': 'l2_gather', 'achieved': achieved, 'peak': l2_peak, 'unit': 'GB/s', 'frac': achieved / l2_peak,
                         'traffic': ncu_traffic(args.mode), 'peak_kind': l2_kind, 'peak_cells': l2_cells,
                         'why_not_hbm': 'one image\'s 25 MB of planes stays L2-resident (ncu: DRAM traffic ~1 % of the algorithmic '
                                        'bytes, L2 hit 97 %), so the 1536 B/sample are L2 -> SM traffic; the HBM copy peak is not the '
                                        'ceiling (SURVEY.md section 8(d)) and is reported beside it',
                         'hbm_peak': pk['hbm_gbs'], 'hbm_peak_kind': pk_kind, 'frac_of_hbm': achieved / pk['hbm_gbs'],
                         'kernel': ('render_kernel' if args.mode == 'fp32_ffma' else 'render_ws_kernel') + ' (tpr_render: +2 helper launches of ~2 us)',
                         'kernel_ms': kern_ms, 'algorithmic_bytes_per_launch': samples_per_step * BYTES_PER_SAMPLE},
            'e2e': {'value': world * samples_per_step / (e2e_ms * 1e-3), 'unit': METRIC, 'ms_per_step': e2e_ms,
                    'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'api': 'ImportanceRenderer.forward_host (tpr_render_host: per-image H2D / repack+render / D2H pipeline)'
                    if world == 1 else 'ImportanceRenderer.forward_host(defer_depth) + 2-float all-reduce + finish_host_depth; every rank\'s '
                    'D2H copies land in its slice of ONE shared pinned host buffer (the gathered result, readable by rank 0)',
                    'outputs_gathered_on_host': e2e_gathered},
            'gpu_launches': 5 * args.steps,                    # pack_planes, pack_decoder, range_init, render_ws, finish
            'clocks': clocks,
            'notes': {'gather': ('outputs gathered by the render kernel (NVLink peer stores) + 2-float all-reduce' if args.gather == 'peer'
                                 else 'NCCL all-gather of outputs') if world > 1 else None, 'host_numa_node': numa},
        }
        if 'h2d_ceiling' in extra and 'ms_per_step' in extra['h2d_ceiling']:
            line['e2e']['copy_ceiling'] = extra.pop('h2d_ceiling')
            line['e2e']['frac_of_copy_ceiling'] = line['e2e']['copy_ceiling']['ms_per_step'] / e2e_ms
        if world == 1 and 'cpu_baseline' in legs:
            os.sched_setaffinity(0, all_cpus)            # the CPU baseline uses every host core
            try:
                line['cpu_baseline'] = leg_cpu_baseline(torch)
            except Exception as e:       # noqa: BLE001
                line['cpu_baseline'] = {'error': f'{type(e).__name__}: {e}'[:400]}
        line.update(extra)
        os.write(real_stdout, (json.dumps(line) + '\n').encode())
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
