"""CPU: the C-ABI library loads without a GPU and exports every symbol include/atvs.h declares;
argument validation works without touching a device."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    import atvsnet_b200 as A
    return A._lib.load()


def test_header_symbols_exported(lib):
    hdr = open(os.path.join(ROOT, 'include', 'atvs.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    names = set(re.findall(r'\b(atvs_[a-z0-9_]+)\s*\(', hdr))
    assert len(names) >= 19
    for n in sorted(names):
        assert hasattr(lib, n), 'libatvs.so does not export %s' % n
    import atvsnet_b200 as A
    assert names == set(A._lib.EXPORTS)


def test_version_and_error_string(lib):
    assert lib.atvs_version() >= 100
    assert isinstance(lib.atvs_last_error(), bytes)


def test_argument_errors_without_gpu(lib):
    # NULL pointers / bad shapes are rejected before any CUDA call
    rc = lib.atvs_get_homographies(None, None, 1, 8, None, None, 1, None, None)
    assert rc == -4 and b'NULL' in lib.atvs_last_error()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert lib.atvs_prob2depth(p, 1, 8, 4, 4, p, p, 3, p, None, None) == -5          # up must be 1 or 4
    assert lib.atvs_build_cost_volume(p, p, p, None, 1, 8, 4, 4, 6, 0, 0, p, None) == -1  # F % 4
    assert lib.atvs_conv3d_fp32(p, p, 1, 2, 2, 2, 8, 5, 1, 0, p, None, None) == -5       # Cout
    for xd in (1, 2):                                                                      # bf16 and fp16 operands
        assert lib.atvs_conv3d_tc(p, xd, p, 1, 2, 2, 2, 12, 8, 1, 0, p, 0, None, None) == -5      # Cin
        assert lib.atvs_conv3d_tc(p, xd, p, 1, 3, 2, 2, 16, 8, 2, 0, p, 0, None, None) == -3      # odd D, stride 2
        assert lib.atvs_conv3d_tc(p, xd, p, 1, 2, 2, 2, 16, 8, 1, 0, p, 1, None, None) == -2      # raw dtype must be f32 | f16
    assert lib.atvs_conv3d_tc(p, 0, p, 1, 2, 2, 2, 16, 8, 1, 0, p, 0, None, None) == -2           # operands must be 16-bit
    assert lib.atvs_pack_conv_weights_tc(p, 16, 8, 0, 0, p, None) == -2
    assert lib.atvs_conv3d_tc_bias(p, 2, p, 1, 2, 2, 2, 16, 8, 1, None, p, 0, None, None) == -4   # plane bias NULL
    # raw dtype / view table / FEM validation before any launch
    assert lib.atvs_bn_relu_add(p, 7, p, 8, 8, 1e-3, 1, None, None, p, None, 0, None) == -2              # raw dtype
    assert lib.atvs_attention_raw(p, 0, None, 2, 8, 8, 0, 0, None, p, None) == -4                        # views NULL
    assert lib.atvs_attention_raw(p, 0, p, 9, 8, 8, 0, 0, None, p, None) == -1                           # N > 8
    assert lib.atvs_bn_relu_add(p, 0, p, 8, 8, 1e-3, 1, None, None, p, None, 7, None) == -2              # act dtype
    assert lib.atvs_cast(p, 2, p, 1, 8, None) == -2                                                      # fp16 -> bf16: via fp32
    assert lib.atvs_conv2d_fp32(p, p, None, 1, 8, 8, 4, 8, 5, 1, 1, 2, 2, 8, 8, 0, p, None) == -5        # kernel size 5
    assert lib.atvs_conv2d_fp32(None, p, None, 1, 8, 8, 4, 8, 3, 1, 1, 1, 1, 8, 8, 0, p, None) == -4
    assert lib.atvs_channel_moments(p, 0, 8, p, None) == -1 and lib.atvs_bn2d_apply(p, None, None, 4, 8, 1e-3, 0, p, 0, None) == -4
    assert lib.atvs_bn2d_apply(p, p, None, 4, 8, 1e-3, 0, p, 1, None) == -2                              # fp32 | fp16 output
    assert lib.atvs_conv2d_tc(p, 2, p, None, 1, 8, 8, 48, 32, 3, 1, 0, p, 0, None, None) == -5           # Cin 32 | 64k
    assert lib.atvs_conv2d_tc(p, 0, p, None, 1, 8, 8, 64, 32, 3, 1, 0, p, 0, None, None) == -2           # 16-bit operands
    assert lib.atvs_packed_weight2d_bytes(128, 128, 3) == 4 * 18 * 32 * 64 * 2 and lib.atvs_packed_weight2d_bytes(48, 8, 3) == 0
    assert lib.atvs_avg_pool_same(p, 1, 8, 8, 4, 0, 1, p, None) == -1
    assert lib.atvs_resize_bilinear_align(p, 1, 8, 8, 4, 0, 4, p, None) == -1
    assert lib.atvs_transform_depth(p, p, None, 1, 4, 4, 1, p, None) == -4
    assert lib.atvs_visual_hull(p, p, p, p, p, 1, 4, 4, 4, 3, 1, p, None) == -5                        # view_num must be 2
    assert lib.atvs_refine_geo_group(p, p, p, p, p, p, p, 1, 4, 1, 4, 16, p, None) == -1               # H > 1
    assert lib.atvs_refine_photo_group(p, p, None, p, 1, 4, 4, 4, 16, p, None) == -4
    # per-tap TMA image + halo-ring images (stride 1, and stride 2 for Cin <= 16)
    assert lib.atvs_packed_weight_bytes(64, 64, 0) == 2 * 27 * 2 * 32 * 64 + 2 * 36 * 2 * 96 * 16
    assert lib.atvs_packed_weight_bytes(8, 8, 0) == 28 * 16 * 8 * 2 + 5 * 2 * 64 * 16 + 5 * 2 * 48 * 16
    assert lib.atvs_packed_weight_bytes(32, 16, 0) == 27 * 16 * 32 * 2 + 18 * 2 * 48 * 16
    # per-class image + fused 8-class image + plane-ring image [4 shifts][2 chunks][3 planes x 4 classes x 8][8]
    assert lib.atvs_packed_weight_bytes(16, 8, 1) == 27 * 16 * 16 * 2 * 2 + 4 * 2 * 96 * 16


def test_ops_refuse_cpu_tensors():
    import torch
    import atvsnet_b200 as A
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        A.prob2depth(torch.zeros(1, 4, 2, 2), 4, torch.zeros(1), torch.ones(1))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        A.get_homographies(torch.zeros(1, 2, 4, 4), torch.zeros(1, 2, 4, 4), 4, torch.zeros(1), torch.ones(1))
