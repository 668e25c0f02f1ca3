"""CPU: argument errors of tpr_run_model_backward (the backward of a point query) are reported before any device is touched."""
import ctypes


def test_run_model_backward_argument_errors(pkg):
    lib = pkg._lib.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    nbytes = lib.tpr_run_model_backward_scratch_bytes(2, 1000)
    assert nbytes >= 2 * 1000 * 4 + 16 and lib.tpr_run_model_backward_scratch_bytes(0, 1000) == 0

    def call(planes=p, dec=p, xyz=p, n_pts=1000, rgb=p, g_rgb=p, g_sigma=p, g_planes=p, g_dec=p, scratch=p, scratch_bytes=nbytes,
             box_warp=1.0):
        return lib.tpr_run_model_backward(planes, 2, 8, 8, dec, xyz, n_pts, box_warp, rgb, g_rgb, g_sigma, 0, g_planes, g_dec,
                                          scratch, scratch_bytes, None)

    assert call(planes=None) == -1 and b'NULL' in lib.tpr_last_error()
    assert call(xyz=None) == -1
    assert call(g_planes=None, g_dec=None) == -1                    # no output asked for
    assert call(rgb=None) == -1 and b'rgb' in lib.tpr_last_error()  # g_rgb needs the forward's rgb
    assert call(g_rgb=None, g_sigma=None) == -1
    assert call(n_pts=0) == -2 and call(n_pts=-5) == -2
    assert call(box_warp=0.0) == -3
    assert call(scratch_bytes=nbytes - 1) == -4
