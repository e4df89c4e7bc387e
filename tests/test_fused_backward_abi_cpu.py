"""CPU-side checks of pws_warp2d_backward_fused's argument validation.  No GPU compute is issued: every call below is
rejected before the library selects a device, so the data pointers are placeholders that are never dereferenced."""
import ctypes

import pytest

FAKE = 0x1000   # never dereferenced: validation fails first


def tensor(_lib, dtype, sizes, strides=None):
    t = _lib.PwsTensor()
    t.data = FAKE
    t.dtype = dtype
    t.device = 0
    if strides is None:
        strides, s = [], 1
        for sz in reversed(sizes):
            strides.insert(0, s)
            s *= sz
    for i in range(4):
        t.size[i] = sizes[i]
        t.stride[i] = strides[i]
    return t


@pytest.fixture()
def abi():
    from pwstablenet_b200 import _lib
    lib = _lib.load()
    N, C, H, W, Ho, Wo, h, w = 2, 3, 16, 24, 32, 48, 8, 12
    drift = tensor(_lib, _lib.PWS_F32, (N, h, w, 2))
    spec = _lib.PwsMapSpec()
    spec.drift = ctypes.pointer(drift)
    spec.theta = FAKE
    spec.base = _lib.PWS_BASE_AFFINE
    spec.upsample = _lib.PWS_UP_ALIGNED
    spec.map_h, spec.map_w = h, w
    spec.pre_add, spec.pre_mul, spec.post_div, spec.post_add = 0.0, 1.0, 1.0, 0.0
    d = dict(lib=lib, _lib=_lib, spec=spec, drift=drift,
             frame=tensor(_lib, _lib.PWS_F32, (N, C, H, W)), frame_u8=tensor(_lib, _lib.PWS_U8, (N, C, H, W)),
             gout=tensor(_lib, _lib.PWS_F32, (N, C, Ho, Wo)), gin=tensor(_lib, _lib.PWS_F32, (N, C, H, W)),
             glat=tensor(_lib, _lib.PWS_F32, (N, h, w, 2)))

    def call(gout, frame, gin=None, glat=None, gtheta=None, spec=spec):
        return lib.pws_warp2d_backward_fused(ctypes.byref(gout), ctypes.byref(frame), ctypes.byref(spec),
                                             ctypes.byref(gin) if gin is not None else None,
                                             ctypes.byref(glat) if glat is not None else None,
                                             gtheta, 0, 0, None)
    d["call"] = call
    return d


def err(a):
    return a["lib"].pws_last_error().decode()


def test_backward_fused_is_exported(abi):
    assert "pws_warp2d_backward_fused" in abi["_lib"].EXPORTS and hasattr(abi["lib"], "pws_warp2d_backward_fused")


def test_uint8_frame_has_no_frame_gradient(abi):
    _lib = abi["_lib"]
    rc = abi["call"](abi["gout"], abi["frame_u8"], gin=abi["gin"])
    assert rc == _lib.PWS_EINVAL and "uint8 frame" in err(abi)


def test_uint8_output_is_not_differentiable(abi):
    _lib = abi["_lib"]
    gout8 = tensor(_lib, _lib.PWS_U8, tuple(abi["gout"].size))
    rc = abi["call"](gout8, abi["frame_u8"], glat=abi["glat"])
    assert rc == _lib.PWS_EINVAL and "not differentiable" in err(abi)


def test_gout_dtype_follows_the_forward_output(abi):
    _lib = abi["_lib"]
    f16 = tensor(_lib, _lib.PWS_F16, tuple(abi["frame"].size))
    rc = abi["call"](abi["gout"], f16, glat=abi["glat"])      # a 16-bit frame's output has the frame's type
    assert rc == _lib.PWS_EINVAL and "grad_output" in err(abi)


def test_gtheta_needs_the_affine_base_and_glattice(abi):
    _lib, spec = abi["_lib"], abi["spec"]
    rc = abi["call"](abi["gout"], abi["frame"], gtheta=FAKE)
    assert rc == _lib.PWS_EINVAL and "glattice" in err(abi)
    spec.base = _lib.PWS_BASE_IDENTITY
    rc = abi["call"](abi["gout"], abi["frame"], glat=abi["glat"], gtheta=FAKE)
    assert rc == _lib.PWS_EINVAL and "affine" in err(abi)


def test_glattice_shape_dtype_and_layout(abi):
    _lib = abi["_lib"]
    N, h, w = 2, 8, 12
    for bad, what in ((tensor(_lib, _lib.PWS_F32, (N, h + 1, w, 2)), "expected sizes"),
                      (tensor(_lib, _lib.PWS_F16, (N, h, w, 2)), "f32"),
                      (tensor(_lib, _lib.PWS_F32, (N, h, w, 2), (h * w * 2, 2, 2 * h, 1)), "contiguous")):
        rc = abi["call"](abi["gout"], abi["frame"], glat=bad)
        assert rc == _lib.PWS_EINVAL and what in err(abi), err(abi)


def test_glattice_must_be_8_byte_aligned(abi):
    # a dense f32 buffer at an odd float offset (a slice of a caller's pool): every node is one 8-byte pair access
    _lib = abi["_lib"]
    glat = tensor(_lib, _lib.PWS_F32, (2, 8, 12, 2))
    glat.data = FAKE + 4
    rc = abi["call"](abi["gout"], abi["frame"], glat=glat)
    assert rc == _lib.PWS_EINVAL and "8-byte aligned" in err(abi), err(abi)


def test_gin_shape_dtype_and_layout(abi):
    _lib = abi["_lib"]
    N, C, H, W = 2, 3, 16, 24
    for bad, what in ((tensor(_lib, _lib.PWS_F32, (N, C, H, W + 1)), "expected sizes"),
                      (tensor(_lib, _lib.PWS_F16, (N, C, H, W)), "f32"),
                      (tensor(_lib, _lib.PWS_F32, (N, C, H, W), (C * H * W, 1, W * C, C)), "contiguous")):
        rc = abi["call"](abi["gout"], abi["frame"], gin=bad)
        assert rc == _lib.PWS_EINVAL and what in err(abi), err(abi)


def test_gout_shape_and_modes(abi):
    _lib = abi["_lib"]
    gout = tensor(_lib, _lib.PWS_F32, (2, 4, 32, 48))
    rc = abi["call"](gout, abi["frame"], glat=abi["glat"])
    assert rc == _lib.PWS_EINVAL and "batch/channels" in err(abi)
    rc = abi["lib"].pws_warp2d_backward_fused(ctypes.byref(abi["gout"]), ctypes.byref(abi["frame"]), ctypes.byref(abi["spec"]),
                                              None, None, None, 2, 0, None)
    assert rc == _lib.PWS_EUNSUPPORTED and "reflection" in err(abi)
