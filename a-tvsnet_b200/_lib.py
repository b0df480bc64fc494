"""ctypes binding of libatvs.so (include/atvs.h).  There is NO fallback: if the library
is missing or a call fails, a RuntimeError is raised."""
import ctypes as C
import functools
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libatvs.so")
_lib = None

F32, BF16, F16 = 0, 1, 2
_p, _i, _ll, _f = C.c_void_p, C.c_int, C.c_longlong, C.c_float

_SIGS = {
    "atvs_get_homographies": [_p, _p, _i, _i, _p, _p, _i, _p, _p],
    "atvs_homography_warping": [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p],
    "atvs_homography_warping_by_depth": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, _p],
    "atvs_build_cost_volume": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    "atvs_build_cost_volume_src16": [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    "atvs_conv3d_fp32": [_p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p],
    "atvs_pack_conv_weights_tc": [_p, _i, _i, _i, _i, _p, _p],
    "atvs_conv3d_tc": [_p, _i, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _p],
    "atvs_conv3d_tc_bias": [_p, _i, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _i, _p, _p],
    "atvs_bn_relu_add": [_p, _i, _p, _ll, _i, _f, _i, _p, _p, _p, _p, _i, _p],
    "atvs_bn_relu_add_pair": [_p, _p, _p, _p, _i, _ll, _i, _f, _i, _p, _p, _p, _i, _p],
    "atvs_set_concurrency": [_i],
    "atvs_cast": [_p, _i, _p, _i, _ll, _p],
    "atvs_pad_cast": [_p, _ll, _i, _i, _p, _i, _p],
    "atvs_add": [_p, _p, _p, _i, _ll, _p],
    "atvs_attention_combine": [_p, _p, _i, _ll, _i, _i, _p, _p],
    "atvs_attention_local_max": [_p, _i, _ll, _i, _i, _p, _p],
    "atvs_attention_partial": [_p, _p, _i, _ll, _i, _i, _p, _p, _p],
    "atvs_attention_finish": [_p, _ll, _i, _p, _p],
    "atvs_attention_raw": [_p, _i, _p, _i, _ll, _i, _i, _i, _p, _p, _p],
    "atvs_attention_fused": [_p, _i, _i, _p, _i, _i, _i, _i, _i, _p, _p],
    "atvs_conv2d_fp32": [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    "atvs_channel_moments": [_p, _ll, _i, _p, _p],
    "atvs_bn2d_apply": [_p, _p, _p, _ll, _i, _f, _i, _p, _i, _p],
    "atvs_pack_conv2d_weights_tc": [_p, _i, _i, _i, _i, _p, _p],
    "atvs_conv2d_tc": [_p, _i, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p, _p],
    "atvs_avg_pool_same": [_p, _i, _i, _i, _i, _i, _i, _p, _p],
    "atvs_resize_bilinear_align": [_p, _i, _i, _i, _i, _i, _i, _p, _p],
    "atvs_transform_depth": [_p, _p, _p, _i, _i, _i, _i, _p, _p],
    "atvs_refine_geo_group": [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p],
    "atvs_refine_photo_group": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p],
    "atvs_visual_hull": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p],
    "atvs_prob2depth": [_p, _i, _i, _i, _i, _p, _p, _i, _p, _p, _p],
    "atvs_fuse_depth_maps": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _f, _f, _i, _i, _p, _ll, _p, _p, _p, _p, _p],
}
EXPORTS = sorted(list(_SIGS) + ["atvs_version", "atvs_last_error", "atvs_device_sm_count",
                                "atvs_packed_weight_bytes", "atvs_packed_weight2d_bytes", "atvs_launch_count",
                                "atvs_fuse_workspace_bytes", "atvs_crc32c",
                                "atvs_saturation_count"])


def lib_path():
    return _SO


def load():
    """Load libatvs.so (building nothing: use __graft_entry__.build() / _build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise RuntimeError("libatvs.so not found at %s - run `python a-tvsnet_b200/_build.py` "
                               "(there is no CPU fallback)" % _SO)
        lib = C.CDLL(_SO)
        for name, sig in _SIGS.items():
            fn = getattr(lib, name)
            fn.argtypes = sig
            fn.restype = _i
        lib.atvs_version.restype = _i
        lib.atvs_last_error.restype = C.c_char_p
        lib.atvs_device_sm_count.restype = _i
        lib.atvs_packed_weight_bytes.argtypes = [_i, _i, _i]
        lib.atvs_packed_weight_bytes.restype = C.c_size_t
        lib.atvs_launch_count.restype = C.c_longlong
        lib.atvs_packed_weight2d_bytes.argtypes = [_i, _i, _i]
        lib.atvs_packed_weight2d_bytes.restype = C.c_size_t
        lib.atvs_fuse_workspace_bytes.argtypes = [_i, _i, _i]
        lib.atvs_fuse_workspace_bytes.restype = C.c_size_t
        lib.atvs_crc32c.argtypes = [_p, C.c_size_t, C.c_uint]
        lib.atvs_crc32c.restype = C.c_uint
        lib.atvs_saturation_count.argtypes = [_i]
        lib.atvs_saturation_count.restype = C.c_longlong
        _lib = lib
    return _lib


def call(name, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError("%s failed (rc=%d): %s" % (name, rc, lib.atvs_last_error().decode()))


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _cuda_devices(obj, found):
    if isinstance(obj, torch.Tensor):
        if obj.is_cuda:
            found.add(obj.device.index)
    elif isinstance(obj, (list, tuple)):
        for o in obj:
            _cuda_devices(o, found)
    elif isinstance(obj, dict):
        for o in obj.values():
            _cuda_devices(o, found)
    else:      # e.g. network.SplitCostVolume
        d = getattr(obj, 'device', None)
        if isinstance(d, torch.device) and d.type == 'cuda':
            found.add(d.index)


def input_device(args, who='a-tvsnet_b200'):
    """``with input_device(args):`` makes the device of the CUDA tensors in ``args`` (tensors, lists, tuples, dicts,
    objects with a ``.device``) the current one, so that every launch goes to that device's current stream and the
    variable store hands out that device's weights (variables.get_variable), and restores the caller's current device
    on exit.  CUDA tensors on different devices raise ValueError before anything is launched; without CUDA tensors
    the current device stays."""
    found = set()
    _cuda_devices(args, found)
    if len(found) > 1:
        raise ValueError("%s: CUDA inputs on different devices (%s); move them to one device"
                         % (who, ', '.join('cuda:%d' % i for i in sorted(found))))
    return torch.cuda.device(found.pop() if found else -1)


def on_input_device(fn):
    """decorator of a public entry point: the call runs under input_device(its arguments)."""
    @functools.wraps(fn)
    def entry(*args, **kwargs):
        with input_device((args, kwargs), fn.__name__):
            return fn(*args, **kwargs)
    return entry


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("a-tvsnet_b200 ops run on CUDA tensors only (no CPU fallback); got %s" % t.device)


def dtype_code(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    if t.dtype == torch.float16:
        return F16
    raise RuntimeError("unsupported dtype %s" % t.dtype)


def f32c(t):
    """contiguous fp32 view/copy on the same device (tensor plumbing only)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()
