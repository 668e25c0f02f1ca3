"""Drop the B200 renderer into an UNMODIFIED reference checkout.

The reference's TriPlaneGenerator constructs ImportanceRenderer() / RaySampler() itself
(training/triplane.py:38-39) and unpickled generators resolve those classes by module path
(SURVEY.md section 8(b)), so the swap is done at CLASS level: the reference classes' ``forward`` /
``run_model`` are rebound to the implementations in this package.  That covers freshly constructed
and unpickled instances alike, touches no state_dict (the renderer has no parameters or buffers),
and leaves training/triplane.py and gen_videos.py untouched.

    import sys; sys.path.insert(0, '<reference>/g_nerf')
    import importlib; importlib.import_module('g-nerf_b200').install()

``uninstall()`` restores the originals.  CPU tensors keep going to the reference implementation
(the reference's own plugins pick 'cuda' vs 'ref' by device the same way, torch_utils/ops/bias_act.py:86-88);
CUDA tensors go to the kernels and never fall back.
"""
import importlib

from .volumetric_rendering import renderer as _r, ray_sampler as _s, ray_marcher as _m

_saved = {}


def _dispatch(ours, theirs, probe_arg):
    def method(self, *args, **kwargs):
        t = args[probe_arg] if len(args) > probe_arg else None
        on_cuda = getattr(t, 'is_cuda', False) or isinstance(t, _r.PackedPlanes)
        return (ours if on_cuda else theirs)(self, *args, **kwargs)
    method.__wrapped__ = theirs
    return method


def install(reference_package: str = 'training.volumetric_rendering'):
    """Rebind the reference's hot-path methods.  ``reference_package`` must already be importable."""
    if _saved:
        return
    ref_r = importlib.import_module(reference_package + '.renderer')
    ref_s = importlib.import_module(reference_package + '.ray_sampler')
    ref_m = importlib.import_module(reference_package + '.ray_marcher')
    targets = [
        (ref_r.ImportanceRenderer, 'forward', _r.ImportanceRenderer.forward, 2),       # probe ray_origins
        (ref_r.ImportanceRenderer, 'run_model', _r.ImportanceRenderer.run_model, 2),   # probe sample_coordinates
        (ref_s.RaySampler, 'forward', _s.RaySampler.forward, 0),
        (ref_m.MipRayMarcher2, 'run_forward', _m.MipRayMarcher2.run_forward, 0),
    ]
    for cls, name, ours, probe in targets:
        _saved[(cls, name)] = getattr(cls, name)
        setattr(cls, name, _dispatch(ours, _saved[(cls, name)], probe))
    # attributes our forward() sets/reads on the (reference-constructed) instance
    for attr, val in (('last_depth_range', None), ('last_fine', None), ('debug_outputs', False),
                      ('defer_depth_clamp', False), ('_timing_events', None), ('cache_packed_planes', False),
                      ('_plane_cache', None), ('_packed', _r.ImportanceRenderer._packed),
                      ('_forward_impl', _r.ImportanceRenderer._forward_impl),
                      ('_run_model_impl', _r.ImportanceRenderer._run_model_impl)):
        setattr(ref_r.ImportanceRenderer, attr, val)


def uninstall():
    for (cls, name), fn in _saved.items():
        setattr(cls, name, fn)
    _saved.clear()
