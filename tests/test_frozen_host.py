"""CPU suite: argument checks of the frozen-BatchNorm backward entries (gfs_bn_act_bwd_frozen, gfs_bn_act_bwd_argmax_frozen).
They return their status before anything reaches a device, so this runs without a GPU."""
import ctypes


def _buf():
    buf = (ctypes.c_float * 64)()
    return ctypes.cast(buf, ctypes.c_void_p), buf


def test_bn_act_bwd_frozen_validates_its_arguments():
    from gfs3d._lib import lib
    l = lib()
    p, _keep = _buf()
    coeffs = [p] * 4                                           # mean, invstd, gamma, beta
    rc = l.gfs_bn_act_bwd_frozen(p, 100, p, 100, None, 100, 64, 100, *coeffs, 0.2, p, p, p, None)
    assert rc == 1 and b"null pointer" in l.gfs_last_error_string()
    rc = l.gfs_bn_act_bwd_frozen(p, 100, p, 100, p, 100, 64, 100, *coeffs, 0.2, None, p, p, None)
    assert rc == 1 and b"null pointer" in l.gfs_last_error_string()
    rc = l.gfs_bn_act_bwd_frozen(p, 100, p, 100, p, 100, 0, 100, *coeffs, 0.2, p, p, p, None)
    assert rc == 1 and b"C=0" in l.gfs_last_error_string()
    rc = l.gfs_bn_act_bwd_frozen(p, 100, p, 100, p, 100, 64, -5, *coeffs, 0.2, p, p, p, None)
    assert rc == 1 and b"M=-5" in l.gfs_last_error_string()


def test_bn_act_bwd_argmax_frozen_validates_its_arguments():
    from gfs3d._lib import lib
    l = lib()
    p, _keep = _buf()
    coeffs = [p] * 4
    rc = l.gfs_bn_act_bwd_argmax_frozen(p, 100, None, 20, p, 2000, p, 2000, 64, 100, *coeffs, 0.2, p, p, p, None)
    assert rc == 1 and b"null pointer" in l.gfs_last_error_string()
    rc = l.gfs_bn_act_bwd_argmax_frozen(p, 100, p, 20, p, 2000, p, 2000, 64, 100, *coeffs, 0.2, p, p, None, None)
    assert rc == 1 and b"null pointer" in l.gfs_last_error_string()
    for C, Mp, k in ((0, 100, 20), (64, 0, 20), (64, 100, 0), (64, 100, 256)):
        rc = l.gfs_bn_act_bwd_argmax_frozen(p, 100, p, k, p, 2000, p, 2000, C, Mp, *coeffs, 0.2, p, p, p, None)
        assert rc == 1 and f"C={C} Mp={Mp} k={k}".encode() in l.gfs_last_error_string(), (C, Mp, k)
    rc = l.gfs_bn_act_bwd_argmax_frozen(p, 100, p, 64, p, 2000, p, 2000, 64, 1 << 25, *coeffs, 0.2, p, p, p, None)   # Mp*k = 2^31
    assert rc == 2 and b"2^31" in l.gfs_last_error_string()
