"""CPU: the deterministic backward's C-ABI surface (TPR_BWD_DETERMINISTIC): its scratch size, and the argument errors of both
backward entry points with the flag set, all reported before any device is touched."""
import ctypes

DET = 0x100
ROWS, DEC_FLOATS = 512, 4452


def test_scratch_size_formula(pkg):
    lib = pkg._lib.lib()
    assert pkg._lib.BWD_DETERMINISTIC == DET
    align = lambda n: (n + 255) // 256 * 256
    for n, h, w in ((1, 8, 8), (2, 256, 256), (3, 17, 5)):
        want = 256 + align(ROWS * DEC_FLOATS * 4) + align(n * 3 * h * w * 32 * 8)
        assert lib.tpr_backward_deterministic_scratch_bytes(n, h, w) == want
    assert lib.tpr_backward_deterministic_scratch_bytes(0, 8, 8) == 0
    assert lib.tpr_backward_deterministic_scratch_bytes(1, 0, 8) == 0
    assert lib.tpr_backward_deterministic_scratch_bytes(1, 8, -1) == 0


def test_run_model_backward_flag(pkg):
    lib = pkg._lib.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    base = lib.tpr_run_model_backward_scratch_bytes(2, 1000)
    extra = lib.tpr_backward_deterministic_scratch_bytes(2, 8, 8)

    def call(flags, scratch_bytes):
        return lib.tpr_run_model_backward(p, 2, 8, 8, p, p, 1000, 1.0, p, p, p, flags, p, p, p, scratch_bytes, None)

    assert call(DET, base) == -4 and b'scratch' in lib.tpr_last_error()           # the existing size is not enough
    assert call(DET, base + extra - 1) == -4
    assert call(DET | pkg._lib.MLP_BF16, base + extra - 1) == -4
    assert call(0x200, base + extra) == -3 and call(DET | 0x4, base + extra) == -3  # other unknown bits stay refused
    assert call(DET | 7, base + extra) == -3


def test_render_backward_flag(pkg):
    lib = pkg._lib.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    n, m, h, w = 2, 16, 8, 8
    base = lib.tpr_render_backward_scratch_bytes(n, m, 8 + 8)
    extra = lib.tpr_backward_deterministic_scratch_bytes(n, h, w)

    def call(flags, scratch_bytes):
        o = pkg._lib.TprOptions(ray_start=2.25, ray_end=3.3, box_warp=1.0, depth_resolution=8, depth_resolution_importance=8,
                                flags=flags)
        return lib.tpr_render_backward(p, n, h, w, p, p, p, m, p, p, p, ctypes.byref(o), p, p, p, None, None, None, p, p, p,
                                       scratch_bytes, None)

    assert call(DET, base) == -4 and b'scratch' in lib.tpr_last_error()
    assert call(DET, base + extra - 1) == -4
    assert call(0x200, base + extra) == -3 and call(DET | 0x4, base + extra) == -3
