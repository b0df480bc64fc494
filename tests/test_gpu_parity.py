"""GPU parity tests (-m gpu): every CUDA entry point, called through the C ABI via the Python
operator layer, against the CPU oracle on the same seeded inputs and against the golden
fixtures generated from the reference's own sources.

Tolerances: geometry (homographies, warps, fp32 cost volumes) bit-exact; fp32 network path
<= 2e-4 of max|.| (different fp32 summation order through 31 conv+BN layers); bf16
tensor-core path: final depth MAE <= 0.1 % of the depth range (BASELINE.json north_star).
"""

import numpy as np
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu

# the two 16-bit operand formats of the tensor-core path (fp16 is the default, FLAGS.precision = 'fp16')
HALF = pytest.mark.parametrize('half', [torch.float16, torch.bfloat16], ids=['f16', 'bf16'])
HALF_EPS = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}
PREC = {torch.float16: 'fp16', torch.bfloat16: 'bf16'}
MAXB_CRM = 0.04     # bf16 (k = 1): max elementwise CRM error / range (measured 1.1e-2); fp16 is held to an 8th of it (measured 2.3e-3)


@pytest.fixture(scope='module')
def A():
    import atvsnet_b200 as A
    assert torch.cuda.is_available()
    A._lib.load()
    return A


def cu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def npy(t):
    return t.detach().float().cpu().numpy()


# ------------------------------------------------------------------ geometry
def test_get_homographies_bit_exact(A, golden):
    from oracle import homography_warping as ohw
    cams, ds, di = golden['ex0_cams'], golden['ds'], golden['di']
    for l, r, D in ((0, 1, 128), (0, 4, 128), (3, 0, 16)):
        H = npy(A.get_homographies(cu(cams[l:l + 1]), cu(cams[r:r + 1]), D, cu(ds), cu(di)))
        Ho = ohw.get_homographies(cams[l:l + 1], cams[r:r + 1], D, ds, di)
        assert np.array_equal(H, Ho)
    assert rel_err(H, golden['ex0_H_3_0']) < 5e-6
    A.FLAGS.inverse_depth = False
    try:
        H = npy(A.get_homographies(cu(cams[0:1]), cu(cams[2:3]), 8, cu(np.float32([2.0])), cu(np.float32([0.5]))))
    finally:
        A.FLAGS.inverse_depth = True
    assert np.array_equal(H, ohw.get_homographies(cams[0:1], cams[2:3], 8, np.float32([2.0]), np.float32([0.5]),
                                                  inverse_depth=False))
    # batch of 3 pairs in one call
    Hb = npy(A.get_homographies(cu(cams[0:3]), cu(cams[1:4]), 5, cu(np.repeat(ds, 3)), cu(np.repeat(di, 3))))
    assert np.array_equal(Hb, ohw.get_homographies(cams[0:3], cams[1:4], 5, np.repeat(ds, 3), np.repeat(di, 3)))


def test_homography_warping_golden_and_oracle(A, golden):
    img, Hs = golden['warp_img'], golden['warp_H']
    for d in (0, 3, 7):
        out, mask = A.homography_warping(cu(img), cu(Hs[:, d]), output_mask=True)
        assert np.array_equal(npy(out), golden['warp_bilinear_%d' % d])
        assert np.array_equal(mask.cpu().numpy(), golden['warp_mask_%d' % d])
    out, mask = A.homography_warping(cu(img[..., :1]), cu(Hs[:, 3]), method='nearest', output_mask=True)
    assert np.array_equal(npy(out), golden['warp_nearest_3'])
    assert np.array_equal(mask.cpu().numpy(), golden['warp_nearest_mask_3'])
    # identity homography: interior copied, last row / column zero (strict x < W-1 rule)
    eye = np.eye(3, dtype=np.float32)[None]
    out = npy(A.homography_warping(cu(img), cu(eye)))
    assert np.array_equal(out[:, :-1, :-1], img[:, :-1, :-1])
    assert not out[:, -1].any() and not out[:, :, -1].any()


def test_homography_warping_edge_cases(A):
    from oracle import homography_warping as ohw
    rng = np.random.default_rng(5)
    img = rng.standard_normal((2, 9, 11, 4)).astype(np.float32)
    H = np.stack([np.float32([[1, 0, 0.5], [0, 1, -0.25], [0, 0, 1]]),        # sub-pixel shift
                  np.float32([[0, 0, 0], [0, 0, 0], [0, 0, 0]])])             # degenerate: z == 0 -> +1e-7
    out, mask = A.homography_warping(cu(img), cu(H), output_mask=True)
    oo, om_ = ohw.homography_warping(img, H, output_mask=True)
    assert np.array_equal(npy(out), oo) and np.array_equal(mask.cpu().numpy(), om_)
    # single-channel (depth map) path, nearest + bilinear
    d1 = rng.standard_normal((2, 9, 11, 1)).astype(np.float32)
    for m in ('bilinear', 'nearest'):
        assert np.array_equal(npy(A.homography_warping(cu(d1), cu(H), method=m)), ohw.homography_warping(d1, H, method=m))
    # far-away homography: everything invalid -> exact zeros
    Hf = np.float32([[[1, 0, 1e4], [0, 1, 1e4], [0, 0, 1]]] * 2)
    out, mask = A.homography_warping(cu(img), cu(Hf), output_mask=True)
    assert not npy(out).any() and not mask.any()
    with pytest.raises(RuntimeError):
        A.homography_warping(torch.zeros(1, 4, 4, 4), torch.zeros(1, 3, 3))      # CPU tensors: no fallback


def test_homography_warping_by_depth(A, golden):
    from oracle import homography_warping as ohw
    c = golden['warp_cams']
    for m in ('bilinear', 'nearest'):
        out, mask = A.homography_warping_by_depth(cu(golden['warp_img']), cu(c[0:1]), cu(c[1:2]),
                                                  cu(golden['bydepth_depth']), output_mask=True, method=m)
        oo, om_ = ohw.homography_warping_by_depth(golden['warp_img'], c[0:1], c[1:2], golden['bydepth_depth'],
                                                  output_mask=True, method=m)
        assert np.array_equal(npy(out), oo) and np.array_equal(mask.cpu().numpy(), om_)


def test_build_cost_volume(A, golden):
    from oracle import model as om
    c = golden['warp_cams'][None, :2]
    ds, di = golden['ds'], golden['di'] * 32
    ref, view = golden['cv_ref'], golden['warp_img']
    cv = npy(A.build_cost_volume(cu(ref), cu(view), cu(c), 4, cu(ds), cu(di), 0, 1))
    assert np.array_equal(cv, om.build_cost_volume(ref, view, c, 4, ds, di, 0, 1))
    bad = np.abs(cv - golden['cv_concat']).max(axis=-1) > 2e-4 * np.abs(cv).max()
    assert bad.mean() < 1e-3
    # WHICH voxels differ from the reference-code golden: only samples that land within 2e-3 px of the validity boundary
    # (x = 0 | W-1, y = 0 | H-1, homography_warping.py:39-43), where the golden's LAPACK matrix inverse and the cofactor
    # inverse used here (homographies equal to 5e-6) put the sample on different sides of the strict mask
    from oracle import homography_warping as ohw_
    Hs = ohw_.get_homographies(c[:, 0], c[:, 1], 4, ds, di).astype(np.float64)
    hh, ww = view.shape[1:3]
    ys, xs = np.mgrid[0:hh, 0:ww]
    pix = np.stack([xs + 0.5, ys + 0.5, np.ones_like(xs, dtype=np.float64)], 0).reshape(3, -1)
    for d in range(4):
        q = Hs[0, d] @ pix
        x, y = q[0] / q[2] - 0.5, q[1] / q[2] - 0.5
        edge = (np.abs(x) < 2e-3) | (np.abs(y) < 2e-3) | (np.abs(x - (ww - 1)) < 2e-3) | (np.abs(y - (hh - 1)) < 2e-3)
        assert not (bad[0, d].reshape(-1) & ~edge).any(), (d, int((bad[0, d].reshape(-1) & ~edge).sum()))
    cv, H = A.build_cost_volume(cu(view), cu(ref), cu(c), 4, cu(ds), cu(di), 1, 0, output_homo=True)
    assert np.array_equal(npy(cv), om.build_cost_volume(view, ref, c, 4, ds, di, 1, 0))
    assert H.shape == (1, 4, 3, 3)
    cv = npy(A.build_cost_volume(cu(ref), cu(view), cu(c), 2, cu(ds), cu(di), 0, 1, warp_ref=True))
    assert np.array_equal(cv, om.build_cost_volume(ref, view, c, 2, ds, di, 0, 1, warp_ref=True))
    # bf16 output: the reference half is the fp32 value rounded once; the warped half is blended from
    # the bf16-rounded source features (test_build_cost_volume_bf16_source), i.e. within one more rounding
    cvb = A.build_cost_volume(cu(ref), cu(view), cu(c), 4, cu(ds), cu(di), 0, 1, out_dtype=torch.bfloat16)
    cvf = A.build_cost_volume(cu(ref), cu(view), cu(c), 4, cu(ds), cu(di), 0, 1)
    assert torch.equal(cvb[..., :8], cvf[..., :8].to(torch.bfloat16))
    assert float((cvb.float() - cvf).abs().max()) <= 2 ** -7 * float(cvf.abs().max())
    # warped-only and masked-L1 modes (model.py:272-280)
    wo = npy(A.build_cost_volume(cu(ref), cu(view), cu(c), 4, cu(ds), cu(di), 0, 1, mode='warped_only'))
    assert np.array_equal(wo, npy(cvf)[..., 8:])
    l1 = npy(A.build_cost_volume(cu(ref), cu(view), cu(c), 4, cu(ds), cu(di), 0, 1, mode='l1_masked'))
    from oracle import homography_warping as ohw
    Hs = ohw.get_homographies(c[:, 0], c[:, 1], 4, ds, di)
    for d in range(4):
        w_, m_ = ohw.homography_warping(view, Hs[:, d], output_mask=True)
        assert np.array_equal(l1[:, d], np.abs(w_ - ref) * m_.astype(np.float32))


def test_build_cost_volume_full_size_properties(A):
    """cfg2 size (D=128, 128x160, F=32): properties that need no oracle run."""
    D, h, w = 128, 128, 160
    cams = A.synthetic.orbit_cams(5, h, w, D)[None]
    f = A.synthetic.smooth_features(2, h, w, 32, seed=1)[None]
    tc, tf = cu(cams), cu(f)
    ds, di = tc[:, 0, 1, 3, 0], tc[:, 0, 1, 3, 1]
    cv = A.build_cost_volume(tf[:, 0], tf[:, 1], tc, D, ds, di, 0, 1)
    assert cv.shape == (1, D, h, w, 64)
    assert torch.equal(cv[0, :, :, :, :32], tf[0, 0].expand(D, h, w, 32))           # tiled reference half
    # linearity in the source feature
    cv2 = A.build_cost_volume(tf[:, 0], 2.0 * tf[:, 1], tc, D, ds, di, 0, 1)
    assert torch.equal(cv2[..., 32:], 2.0 * cv[..., 32:])
    # identical cameras => identity warp on the interior for every plane
    cvi = A.build_cost_volume(tf[:, 0], tf[:, 1], tc, D, ds, di, 0, 0)
    assert torch.equal(cvi[0, :, :-1, :-1, 32:], tf[0, 1, :-1, :-1].expand(D, h - 1, w - 1, 32))
    valid = (cv[..., 32:] != 0).any(dim=-1).float().mean().item()
    assert 0.7 < valid <= 1.0


# ------------------------------------------------------------------ conv primitives
LAYER_KINDS = [(64, 8, 1, 0), (64, 16, 2, 0), (16, 32, 2, 0), (32, 64, 2, 0), (16, 16, 1, 0), (32, 32, 1, 0),
               (64, 64, 1, 0), (8, 16, 2, 0), (8, 8, 1, 0), (8, 1, 1, 0), (8, 16, 1, 0),
               (64, 32, 2, 1), (32, 16, 2, 1), (16, 8, 2, 1)]


def _conv_case(cin, cout, stride, transposed, seed, shape=(2, 4, 6, 10)):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal(shape + (cin,)).astype(np.float32)
    wshape = (3, 3, 3, cout, cin) if transposed else (3, 3, 3, cin, cout)
    w = (rng.standard_normal(wshape) / np.sqrt(27 * cin)).astype(np.float32)
    return x, w


@pytest.mark.parametrize('cin,cout,stride,transposed', LAYER_KINDS)
def test_conv3d_fp32(A, cin, cout, stride, transposed):
    from oracle import network as onet
    from atvsnet_b200.network import conv3d_raw
    x, w = _conv_case(cin, cout, stride, transposed, 1)
    raw, stats = conv3d_raw(cu(x), 't', cu(w), cout, stride, bool(transposed), True)
    ref = onet.deconv3d(x, w) if transposed else onet.conv3d(x, w, stride)
    assert raw.shape == ref.shape
    assert rel_err(npy(raw), ref) < 2e-5
    s = stats.cpu().numpy()
    flat = ref.reshape(-1, cout).astype(np.float64)
    assert np.allclose(s[:cout], flat.sum(0), rtol=1e-4, atol=1e-3)
    assert np.allclose(s[cout:], (flat ** 2).sum(0), rtol=1e-4, atol=1e-3)


@HALF
@pytest.mark.parametrize('cin,cout,stride,transposed', LAYER_KINDS)
def test_conv3d_bf16_tensor_core(A, cin, cout, stride, transposed, half):
    """tcgen05 implicit GEMM vs the oracle conv on bf16-rounded operands (so only the fp32
    accumulation order differs)."""
    from oracle import network as onet
    from atvsnet_b200.network import conv3d_raw
    x, w = _conv_case(cin, cout, stride, transposed, 2, shape=(1, 8, 12, 20))
    xb = torch.from_numpy(x).to(half)
    wb = torch.from_numpy(w).to(half).float()
    A.variables.packed_cache().clear()
    raw, stats = conv3d_raw(xb.cuda(), 'tc_test_%d_%d_%d_%d' % (cin, cout, stride, transposed), wb.cuda(), cout,
                            stride, bool(transposed), True)
    torch.cuda.synchronize()
    xr = xb.float().numpy()
    ref = onet.deconv3d(xr, wb.numpy()) if transposed else onet.conv3d(xr, wb.numpy(), stride)
    assert raw.shape == ref.shape
    assert rel_err(npy(raw), ref) < 1e-4
    s = stats.cpu().numpy()
    flat = ref.reshape(-1, cout).astype(np.float64)
    assert np.allclose(s[:cout], flat.sum(0), rtol=1e-3, atol=1e-2)
    assert np.allclose(s[cout:], (flat ** 2).sum(0), rtol=1e-3, atol=1e-2)


@HALF
def test_conv3d_bf16_ragged_and_batched(A, half):
    """brick tiles hanging over every border, odd extents (stride 1 / deconv), batch > 1."""
    from oracle import network as onet
    from atvsnet_b200.network import conv3d_raw
    for (cin, cout, stride, tr, shape) in ((16, 16, 1, 0, (2, 3, 5, 7)), (32, 16, 2, 1, (2, 3, 5, 7)),
                                           (8, 8, 1, 0, (1, 1, 9, 33)), (64, 16, 2, 0, (2, 2, 6, 10)),
                                           (8, 16, 2, 0, (1, 10, 2, 18))):
        x, w = _conv_case(cin, cout, stride, tr, 3, shape=shape)
        xb = torch.from_numpy(x).to(half)
        wb = torch.from_numpy(w).to(half).float()
        A.variables.packed_cache().clear()
        raw, _ = conv3d_raw(xb.cuda(), 'rag', wb.cuda(), cout, stride, bool(tr), True)
        xr = xb.float().numpy()
        ref = onet.deconv3d(xr, wb.numpy()) if tr else onet.conv3d(xr, wb.numpy(), stride)
        assert rel_err(npy(raw), ref) < 1e-4, (cin, cout, stride, tr, shape)


RING_CASES = [(64, 8, (1, 8, 40, 104)), (8, 8, (1, 8, 40, 104)), (8, 1, (1, 9, 37, 101)), (8, 16, (2, 10, 40, 88)),
              (16, 16, (1, 33, 37, 29)), (32, 32, (1, 8, 64, 64)), (64, 64, (1, 8, 64, 64)), (32, 64, (1, 6, 80, 72)),
              (64, 16, (1, 40, 32, 32))]


@HALF
@pytest.mark.parametrize('cin,cout,shape', RING_CASES)
def test_conv3d_bf16_halo_ring(A, cin, cout, shape, half):
    """large stride-1 volumes take the halo-ring kernel (every input plane staged once in smem)."""
    from oracle import network as onet
    from atvsnet_b200.network import conv3d_raw
    assert shape[1] * shape[2] * shape[3] >= 32768
    x, w = _conv_case(cin, cout, 1, 0, 7, shape=shape)
    xb = torch.from_numpy(x).to(half)
    wb = torch.from_numpy(w).to(half).float()
    A.variables.packed_cache().clear()
    raw, stats = conv3d_raw(xb.cuda(), 'ring_%d_%d' % (cin, cout), wb.cuda(), cout, 1, False, True)
    torch.cuda.synchronize()
    ref = onet.conv3d(xb.float().numpy(), wb.numpy(), 1)
    assert rel_err(npy(raw), ref) < 1e-4
    s = stats.cpu().numpy()
    flat = ref.reshape(-1, cout).astype(np.float64)
    assert np.allclose(s[:cout], flat.sum(0), rtol=1e-3, atol=5e-2)
    assert np.allclose(s[cout:], (flat ** 2).sum(0), rtol=1e-3, atol=5e-2)


RAW16_CASES = [(8, 8, 1, 0, (1, 16, 64, 80)), (32, 8, 1, 0, (1, 16, 64, 80)), (8, 16, 1, 0, (1, 16, 64, 80)),
               (16, 16, 1, 0, (1, 12, 24, 40)), (8, 16, 2, 0, (1, 64, 128, 160)), (32, 16, 2, 0, (1, 16, 64, 80)),
               (16, 8, 2, 1, (1, 8, 32, 40)), (64, 32, 2, 1, (1, 4, 8, 12)), (64, 64, 1, 0, (1, 4, 8, 12)),
               (8, 1, 1, 0, (1, 16, 64, 80))]


@HALF
@pytest.mark.parametrize('cin,cout,stride,transposed,shape', RAW16_CASES)
def test_conv3d_bf16_raw_fp16(A, cin, cout, stride, transposed, shape, half):
    """raw outputs stored as saturated fp16 (layers that only feed the BN pass): every tensor kernel (ring, stride-2
    ring, per-tap TMA, fused deconv) against its own fp32 raw output; moments unchanged (fp32 accumulators); the BN
    pass on the fp16 tensor equals the BN pass on the fp32 one to bf16 output rounding."""
    from atvsnet_b200.network import conv3d_raw, bn_relu_add
    x, w = _conv_case(cin, cout, stride, transposed, 11, shape=shape)
    xb = torch.from_numpy(x).to(half).cuda()
    wb = torch.from_numpy(w).to(half).float().cuda()
    A.variables.packed_cache().clear()
    r32, s32 = conv3d_raw(xb, 'r16_%d_%d' % (cin, cout), wb, cout, stride, bool(transposed), True)
    r16, s16 = conv3d_raw(xb, 'r16_%d_%d' % (cin, cout), wb, cout, stride, bool(transposed), True, raw_dtype=torch.float16)
    torch.cuda.synchronize()
    assert r16.dtype == torch.float16 and r16.shape == r32.shape
    a, b = r32.cpu().numpy(), r16.float().cpu().numpy()
    assert np.abs(a - b).max() <= 2.0 ** -11 * np.abs(a).max() + 1e-7         # one fp16 rounding
    assert np.array_equal(a.astype(np.float16), r16.cpu().numpy())            # exactly round-to-nearest of the fp32 result
    assert np.allclose(s32.cpu().numpy(), s16.cpu().numpy(), rtol=1e-6, atol=1e-3)
    if cout % 4 == 0:
        p32, _ = bn_relu_add(r32, s32, True, [], True, False, half)
        p16, _ = bn_relu_add(r16, s16, True, [], True, False, half)
        d = (p32.float() - p16.float()).abs()
        assert float(d.max()) <= 2 * HALF_EPS[half] * max(1.0, float(p32.float().abs().max()))
        assert float((d > 0).float().mean()) < 0.25


@HALF
def test_raw_fp16_saturates(A, half):
    """values beyond the fp16 range are clamped to +-65504 (never inf), NaN stays NaN."""
    from atvsnet_b200.network import conv3d_raw
    x = torch.full((1, 8, 16, 16, 8), 300.0).to(half).cuda()
    w = torch.full((3, 3, 3, 8, 8), 2.0).cuda()      # 27 * 8 * 300 * 2 = 129 600 > 65 504
    w[..., 1] = -2.0
    A.variables.packed_cache().clear()
    A.pipeline.check_saturation(action='count')
    r16, _ = conv3d_raw(x, 'sat16', w, 8, 1, False, True, raw_dtype=torch.float16)
    v = r16.float()
    assert bool(torch.isfinite(v).all()) and float(v.max()) == 65504.0 and float(v.min()) == -65504.0
    # ... and is never silent: the epilogue counts every clamped row
    with pytest.raises(RuntimeError, match='clamped'):
        A.pipeline.check_saturation()
    assert A.pipeline.check_saturation(action='count') == 0          # the failed check reset the counter
    ok16, _ = conv3d_raw((x * 0.01).to(half), 'sat16', w, 8, 1, False, True, raw_dtype=torch.float16)
    assert A.pipeline.check_saturation(action='count') == 0


S2_RING_CASES = [(8, 16, (1, 32, 128, 160)), (16, 32, (2, 20, 144, 112)), (8, 8, (1, 12, 260, 196)), (16, 16, (1, 68, 132, 68))]


@HALF
@pytest.mark.parametrize('cin,cout,shape', S2_RING_CASES)
def test_conv3d_bf16_stride2_ring(A, cin, cout, shape, half):
    """large stride-2 volumes with 8 or 16 input channels take the de-interleaving ring kernel (conv_ring_s2.cu); the
    32-channel stride-2 layers run on the per-tap kernel (RAW16_CASES)."""
    from oracle import network as onet
    from atvsnet_b200.network import conv3d_raw
    assert (shape[1] // 2) * (shape[2] // 2) * (shape[3] // 2) >= 32768
    x, w = _conv_case(cin, cout, 2, 0, 9, shape=shape)
    xb = torch.from_numpy(x).to(half)
    wb = torch.from_numpy(w).to(half).float()
    A.variables.packed_cache().clear()
    raw, stats = conv3d_raw(xb.cuda(), 's2ring_%d_%d' % (cin, cout), wb.cuda(), cout, 2, False, True)
    torch.cuda.synchronize()
    ref = onet.conv3d(xb.float().numpy(), wb.numpy(), 2)
    assert raw.shape == ref.shape
    assert rel_err(npy(raw), ref) < 1e-4
    s = stats.cpu().numpy()
    flat = ref.reshape(-1, cout).astype(np.float64)
    assert np.allclose(s[:cout], flat.sum(0), rtol=1e-3, atol=5e-2)
    assert np.allclose(s[cout:], (flat ** 2).sum(0), rtol=1e-3, atol=5e-2)


# every case has >= 16384 input voxels (the plane ring's dispatch threshold); (1, 16, 40, 48) runs on 16 CTAs of 18 planes
# over columns of 16, so that most units start mid-column with a halo plane
DECONV_RING_CASES = [(16, 8, (1, 16, 40, 48)), (32, 16, (1, 10, 36, 52)), (16, 8, (2, 9, 33, 29)), (32, 16, (1, 5, 17, 193)),
                     (16, 8, (1, 64, 64, 80)), (16, 8, (1, 3, 2, 2736)), (16, 8, (1, 1, 16, 1032)), (32, 16, (1, 20, 32, 40))]


@HALF
@pytest.mark.parametrize('cin,cout,shape', DECONV_RING_CASES)
def test_deconv3d_plane_ring(A, cin, cout, shape, half):
    """transposed convolution as a plane ring (conv_deconv_ring.cu: 4 shifted MMAs per input plane into [3 output
    planes][4 parity classes][Cout] columns): against the oracle conv3d_transpose on 16-bit-rounded operands, ragged
    tiles, batches, H = 2, D = 1, units with and without the halo plane, fp32 and fp16 raw outputs, moments."""
    from oracle import network as onet
    from atvsnet_b200.network import conv3d_raw
    assert shape[0] * shape[1] * shape[2] * shape[3] >= 16384
    x, w = _conv_case(cin, cout, 2, 1, 13, shape=shape)
    xb = torch.from_numpy(x).to(half)
    wb = torch.from_numpy(w).to(half).float()
    A.variables.packed_cache().clear()
    raw, stats = conv3d_raw(xb.cuda(), 'dring_%d_%d' % (cin, cout), wb.cuda(), cout, 2, True, True)
    raw16, _ = conv3d_raw(xb.cuda(), 'dring_%d_%d' % (cin, cout), wb.cuda(), cout, 2, True, True, raw_dtype=torch.float16)
    torch.cuda.synchronize()
    ref = onet.deconv3d(xb.float().numpy(), wb.numpy())
    assert raw.shape == ref.shape
    assert rel_err(npy(raw), ref) < 2e-5
    assert np.array_equal(npy(raw).astype(np.float16), raw16.cpu().numpy())
    s = stats.cpu().numpy()
    flat = ref.reshape(-1, cout).astype(np.float64)
    assert np.allclose(s[:cout], flat.sum(0), rtol=1e-3, atol=5e-2)
    assert np.allclose(s[cout:], (flat ** 2).sum(0), rtol=1e-3, atol=5e-2)


@HALF
@pytest.mark.parametrize('stride,shape', [(1, (1, 8, 40, 104)), (2, (1, 8, 40, 104)), (1, (2, 4, 10, 12)), (2, (2, 4, 12, 10)),
                                          (2, (1, 8, 128, 160))])
def test_conv3d_split_cost_volume(A, stride, shape, half):
    """conv over [tile(ref, D) | warped] == conv(warped) + per-plane-class bias from ref (ring and TMA kernels)."""
    from oracle import network as onet
    from atvsnet_b200.network import SplitCostVolume, conv3d_split, conv3d_raw
    rng = np.random.default_rng(11)
    B, D, H, W = shape
    F, cout = 32, 8 if stride == 1 else 16
    ref = torch.from_numpy(rng.standard_normal((B, H, W, F)).astype(np.float32)).to(half)
    warped = torch.from_numpy(rng.standard_normal((B, D, H, W, F)).astype(np.float32)).to(half)
    w = torch.from_numpy((rng.standard_normal((3, 3, 3, 2 * F, cout)) / np.sqrt(27 * 2 * F)).astype(np.float32))
    w = w.to(half).float()
    A.variables.packed_cache().clear()
    stats = torch.zeros(128, dtype=torch.float64, device='cuda')
    A.FLAGS.first_raw_dtype = 'f32'
    try:
        raw, st = conv3d_split(SplitCostVolume(ref.float().cuda(), warped.cuda()), 'split_t', w.cuda(), cout, stride, stats)
    finally:
        A.FLAGS.first_raw_dtype = 'f16'
    assert raw.dtype == torch.float32
    # default storage: saturated fp16 (guarded by the saturation counter) = one rounding of the fp32 result
    raw16, _ = conv3d_split(SplitCostVolume(ref.float().cuda(), warped.cuda()), 'split_t', w.cuda(), cout, stride,
                            torch.zeros(128, dtype=torch.float64, device='cuda'))
    assert raw16.dtype == torch.float16 and np.array_equal(npy(raw).astype(np.float16), raw16.cpu().numpy())
    full = np.concatenate([np.tile(ref.float().numpy()[:, None], (1, D, 1, 1, 1)), warped.float().numpy()], axis=-1)
    refo = onet.conv3d(full, w.numpy(), stride)
    assert raw.shape == refo.shape
    assert rel_err(npy(raw), refo) < 1e-4
    flat = refo.reshape(-1, cout).astype(np.float64)
    assert np.allclose(st.cpu().numpy()[:cout], flat.sum(0), rtol=1e-3, atol=5e-2)
    # and equals the plain kernel on the materialised concatenation
    raw2, _ = conv3d_raw(torch.from_numpy(full).to(half).cuda(), 'split_full', w.cuda(), cout, stride, False, True)
    assert rel_err(npy(raw), npy(raw2)) < 1e-5


def test_bn_relu_add_pair(A):
    """add of two freshly convolved layers, each with its own batch statistics, in one pass."""
    from oracle import network as onet
    from atvsnet_b200.network import bn_relu_add_pair, _PendingRaw
    rng = np.random.default_rng(5)
    for C, shape in ((8, (1, 4, 6, 10)), (16, (1, 3, 5, 7)), (12, (1, 2, 3, 5))):
        ra = (rng.standard_normal(shape + (C,)) * 2 + 0.5).astype(np.float32)
        rb = (rng.standard_normal(shape + (C,)) * 0.7 - 1).astype(np.float32)
        sk = rng.standard_normal(ra.shape).astype(np.float32)

        def moments(r):
            f = r.reshape(-1, C).astype(np.float64)
            return torch.from_numpy(np.concatenate([f.sum(0), (f ** 2).sum(0)])).cuda()
        ref_a, ref_b = onet.relu(onet.batch_norm_train(ra)), onet.relu(onet.batch_norm_train(rb))
        plain, summ = bn_relu_add_pair(cu(ra), moments(ra), _PendingRaw(cu(rb), moments(rb), True), True, cu(sk), True,
                                       torch.float32)
        assert rel_err(npy(plain), ref_a) < 1e-5
        assert rel_err(npy(summ), ref_a + ref_b + sk) < 1e-5
        _, sb = bn_relu_add_pair(cu(ra), moments(ra), _PendingRaw(cu(rb), moments(rb), True), True, None, False,
                                 torch.bfloat16)
        assert rel_err(npy(sb), ref_a + ref_b) < 1e-2


@HALF
def test_build_cost_volume_bf16_source(A, half):
    """bf16 volumes gather from a bf16 copy of the source features: equals the fp32-source kernel up to
    the bf16 rounding of its inputs, and exactly the oracle run on bf16-rounded source features."""
    from oracle import model as om
    h, w, D, F = 24, 40, 20, 32
    cams = A.synthetic.orbit_cams(3, h, w, D)[None]
    feats = A.synthetic.smooth_features(3, h, w, F, seed=5)[None]
    ds, di = cams[:, 0, 1, 3, 0], cams[:, 0, 1, 3, 1]
    fr = torch.from_numpy(feats).to(half).float().numpy()
    for mode in ('warped_only', 'concat', 'l1_masked'):
        out = A.build_cost_volume(cu(feats[:, 0]), cu(feats[:, 2]), cu(cams), D, cu(ds), cu(di), 0, 2, mode=mode,
                                  out_dtype=half)
        full = om.build_cost_volume(feats[:, 0], fr[:, 2], cams, D, ds, di, 0, 2)
        if mode == 'warped_only':
            ref = full[..., F:]
        elif mode == 'concat':
            ref = full
        else:       # fp32 CUDA path of the same mode (itself checked against the oracle elsewhere)
            ref = npy(A.build_cost_volume(cu(feats[:, 0]), cu(fr[:, 2]), cu(cams), D, cu(ds), cu(di), 0, 2, mode=mode))
        got = npy(out.float())
        # bf16: fp32 blend, one rounding.  fp16: the blend itself runs in packed-half arithmetic (4 products + 3 fused
        # adds on fp16-rounded weights), a few fp16 roundings of the largest term
        k = 1.0 if half == torch.bfloat16 or mode == 'l1_masked' else 4.0
        assert np.abs(got - ref).max() <= k * HALF_EPS[half] * np.abs(ref).max() + 1e-6, mode


@HALF
def test_build_cost_volume_src16_entry(A, half):
    """atvs_build_cost_volume_src16 (16-bit view feature map handed in, as pipeline.run_multiview does once per frame)
    is bit-identical to atvs_build_cost_volume converting the fp32 map itself, in all three modes; argument errors."""
    h, w, D, F = 24, 40, 20, 32
    cams = A.synthetic.orbit_cams(3, h, w, D)[None]
    feats = A.synthetic.smooth_features(3, h, w, F, seed=6)[None]
    ds, di = cams[:, 0, 1, 3, 0], cams[:, 0, 1, 3, 1]
    v16 = cu(feats[:, 2]).to(half)
    for mode in ('warped_only', 'concat', 'l1_masked'):
        a = A.build_cost_volume(cu(feats[:, 0]), cu(feats[:, 2]), cu(cams), D, cu(ds), cu(di), 0, 2, mode=mode, out_dtype=half)
        b = A.build_cost_volume(cu(feats[:, 0]), v16, cu(cams), D, cu(ds), cu(di), 0, 2, mode=mode, out_dtype=half)
        assert torch.equal(a, b), mode
    with pytest.raises(ValueError):
        A.build_cost_volume(cu(feats[:, 0]), v16, cu(cams), D, cu(ds), cu(di), 0, 2)      # fp32 volume from a 16-bit map
    other = torch.float16 if half == torch.bfloat16 else torch.bfloat16
    with pytest.raises(ValueError):
        A.build_cost_volume(cu(feats[:, 0]), v16, cu(cams), D, cu(ds), cu(di), 0, 2, out_dtype=other)
    f12 = cu(feats[:, 2, :, :, :12]).contiguous().to(half)
    with pytest.raises(RuntimeError):
        A.build_cost_volume(cu(feats[:, 0, :, :, :12]).contiguous(), f12, cu(cams), D, cu(ds), cu(di), 0, 2,
                            mode='warped_only', out_dtype=half)


def test_conv3d_argument_errors(A):
    from atvsnet_b200.network import conv3d_raw
    x = torch.zeros(1, 3, 4, 4, 16, dtype=torch.bfloat16, device='cuda')
    w = torch.zeros(3, 3, 3, 16, 32, device='cuda')
    A.variables.packed_cache().clear()
    with pytest.raises(RuntimeError, match='even'):
        conv3d_raw(x, 'err', w, 32, 2, False, False)          # odd D with stride 2 on the TMA path
    with pytest.raises(RuntimeError):
        conv3d_raw(torch.zeros(1, 2, 2, 2, 12, device='cuda'), 'e2', torch.zeros(3, 3, 3, 12, 5, device='cuda'), 5, 1,
                   False, False)                               # Cout=5 unsupported on the fp32 path


def test_bn_relu_add(A):
    from oracle import network as onet
    from atvsnet_b200.network import bn_relu_add
    rng = np.random.default_rng(4)
    raw = (rng.standard_normal((1, 4, 6, 10, 16)) * 3 + 1).astype(np.float32)
    s1 = rng.standard_normal(raw.shape).astype(np.float32)
    s2 = rng.standard_normal(raw.shape).astype(np.float32)
    flat = raw.reshape(-1, 16).astype(np.float64)
    stats = torch.from_numpy(np.concatenate([flat.sum(0), (flat ** 2).sum(0)])).cuda()
    plain, summ = bn_relu_add(cu(raw), stats, True, [cu(s1), cu(s2)], True, True, torch.float32)
    ref = onet.relu(onet.batch_norm_train(raw))
    assert rel_err(npy(plain), ref) < 1e-5
    assert rel_err(npy(summ), ref + s1 + s2) < 1e-5
    pb, sb = bn_relu_add(cu(raw), stats, True, [cu(s1).bfloat16()], True, True, torch.bfloat16)
    assert rel_err(npy(pb), ref) < 1e-2 and rel_err(npy(sb), ref + s1) < 1e-2


# ------------------------------------------------------------------ networks
def test_cost_volume_reasoning_fp32_golden(A, golden, gweights):
    A.variables.load_weights(gweights)
    A.FLAGS.precision = 'fp32'
    try:
        prob, filt = A.cost_volume_reasoning(cu(golden['crm_in']), output_filtered_cost=True)
        assert rel_err(npy(filt), golden['crm_filtered']) < 5e-4
        assert rel_err(npy(prob), golden['crm_prob']) < 5e-4
        only = A.cost_volume_reasoning(cu(golden['crm_in']), output_prob=False)
        assert rel_err(npy(only), golden['crm_filtered_only']) < 5e-4
        tower = A.StackedUNet_prob({'data': cu(golden['crm_in'])}, is_training=True, reuse=None)
        for nm in ('conv_b0_1_0', 'conv_b0_0_1', 'conv_b0_3_1', 'conv_b0_4_0', 'conv_b0_6_0', 'conv_b1_0_0',
                   'conv_b1_5_0'):
            assert rel_err(npy(tower.get_output_by_name(nm)), golden['crm_' + nm]) < 5e-4, nm
    finally:
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION


@HALF
def test_cost_volume_reasoning_bf16(A, golden, gweights, half):
    A.variables.load_weights(gweights)
    A.FLAGS.precision = PREC[half]
    try:
        prob, filt = A.cost_volume_reasoning(cu(golden['crm_in']), output_filtered_cost=True)
    finally:
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION
    # 31 16-bit layers with batch-stat BN on tiny volumes: loose elementwise bound, tight on average (8x tighter for
    # the 11-bit format)
    k = HALF_EPS[half] / 2.0 ** -8
    e = np.abs(npy(filt) - golden['crm_filtered'])
    s_f = np.abs(golden['crm_filtered']).max()
    assert e.mean() < k * (0.03 * np.abs(golden['crm_filtered']).mean() + 0.03)
    e2 = np.abs(npy(prob) - golden['crm_prob'])
    s_p = np.abs(golden['crm_prob']).max()
    print("CRM %s vs reference-graph golden: filtered mean %.2e max %.2e of max|x|, logits mean %.2e max %.2e of max|x|"
          % (PREC[half], e.mean() / s_f, e.max() / s_f, e2.mean() / s_p, e2.max() / s_p))
    assert e2.mean() < k * 0.05 * np.abs(golden['crm_prob']).std()
    # elementwise: no voxel further than MAXB of the tensor's range from the reference-graph value
    assert e.max() < k * MAXB_CRM * s_f and e2.max() < k * MAXB_CRM * s_p


def test_attention_aggregation(A, golden, gweights):
    A.variables.load_weights(gweights)
    xs = golden['aam_in']
    A.FLAGS.precision = 'fp32'
    try:
        keep = A.cost_volume_aggregation(cu(xs), keepchannel=True)
        assert rel_err(npy(keep), golden['aam1_keep']) < 2e-5
        assert rel_err(npy(A.cost_volume_aggregation(cu(xs), keepchannel=False)), golden['aam1_prob']) < 2e-5
        assert rel_err(npy(A.cost_volume_aggregation_refine(cu(xs), keepchannel=True)), golden['aam2_keep']) < 2e-5
        assert rel_err(npy(A.output_conv(cu(golden['aam1_keep']))), golden['outconv']) < 2e-5
        assert rel_err(npy(A.output_conv_refine(cu(golden['aam1_keep']))), golden['outconv_refine']) < 2e-5
        # list-of-views input == stacked (B,D,H,W,C,N) input
        lst = [cu(xs[..., i]) for i in range(xs.shape[-1])]
        assert torch.equal(A.cost_volume_aggregation(lst, keepchannel=True), keep)
        # single view: softmax over one view is 1 -> output == input
        one = A.cost_volume_aggregation(cu(xs[..., :1]), keepchannel=True)
        assert rel_err(npy(one), xs[..., 0]) < 1e-6
    finally:
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION
    keepb = A.cost_volume_aggregation(cu(xs), keepchannel=True)
    assert rel_err(npy(keepb), golden['aam1_keep']) < 2e-2


@HALF
@pytest.mark.parametrize('nv,B,D,H,W', [(2, 1, 5, 11, 13), (3, 1, 8, 16, 24), (4, 2, 6, 20, 9), (4, 1, 16, 32, 40),
                                         (5, 1, 4, 17, 8), (8, 1, 3, 8, 12)])
def test_attention_fused(A, half, nv, B, D, H, W):
    """atvs_attention_fused (one kernel: attention convolutions of all views in TMEM + softmax over views + weighted sum,
    network.py:282-351, 379-408) against the oracle module on the SAME 16-bit-rounded views and weights (fp32 everywhere
    else: only the summation order and exp2f differ), on ragged tiles, several view counts (kernels built for 2 / 4 / 8)
    and batches; and against the two-kernel path, whose only difference is its fp16 storage of the logits."""
    from oracle import network as onet
    rng = np.random.default_rng(nv * 100 + D)
    w = A.variables.synthetic_weights(seed=3)
    ku, ks = 'attention_aggregate/attention_activation/weight_unique', 'attention_aggregate/attention_activation/weight_shared'
    # logits of a few units, like a trained module's: scale the He-normal kernels up
    w[ku] = (w[ku] * 3).astype(np.float32)
    w[ks] = (w[ks] * 3).astype(np.float32)
    A.variables.load_weights(w)
    rnd = lambda a: torch.from_numpy(a).to(half).float().numpy()
    xs = rnd(np.maximum(rng.standard_normal((B, D, H, W, 8, nv)), -0.5).astype(np.float32))
    wo = dict(w)
    wo[ku], wo[ks] = rnd(w[ku]), rnd(w[ks])
    ref = onet.AttAggregation_keepchannel({'data': xs}, wo).get_output()
    views = [cu(xs[..., n]).to(half) for n in range(nv)]
    A.FLAGS.precision = PREC[half]
    try:
        assert A.network.attention_fused_ok(views)
        A.cost_volume_aggregation(views, keepchannel=True)           # packs the weight image
        n0 = A._lib.load().atvs_launch_count()
        got = A.cost_volume_aggregation(views, keepchannel=True)
        assert A._lib.load().atvs_launch_count() - n0 == 1          # ONE kernel
        A.FLAGS.attention_fused = False
        two = A.cost_volume_aggregation(views, keepchannel=True)
    finally:
        A.FLAGS.attention_fused = True
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION
    assert got.shape == (B, D, H, W, 8) and got.dtype == torch.float32
    scale = np.abs(ref).max()
    assert np.abs(npy(got) - ref).max() < 2e-5 * scale, np.abs(npy(got) - ref).max() / scale
    d2 = np.abs(npy(two) - npy(got)).max() / scale
    print("attention fused vs two-kernel path (fp16 logits): max diff / scale %.2e" % d2)
    assert d2 < 4 * HALF_EPS[torch.float16]          # measured 4-7e-4


def test_prob2depth(A, golden):
    from oracle import model as om
    vol, ds, di = golden['p2d_vol'], golden['p2d_start'], golden['p2d_interval']
    est, pm = A.prob2depth(cu(vol), 16, cu(ds), cu(di), out_prob_map=True)
    assert rel_err(npy(est), golden['p2d_est']) < 2e-6
    assert (np.abs(npy(pm) - golden['p2d_prob']) > 1e-5).mean() < 1e-3
    e, eu, p, pu = A.prob2depth_upsample(cu(vol), 16, cu(ds), cu(di), out_prob_map=True)
    assert eu.shape == (1, 40, 48, 1)
    assert rel_err(npy(eu), golden['p2d_est_up']) < 2e-6
    assert (np.abs(npy(pu) - golden['p2d_prob_up']) > 1e-5).mean() < 2e-3
    # peaked volume -> estimate = that plane's depth; uniform volume -> mid-range
    D = 32
    v = np.full((1, D, 4, 5), 30.0, np.float32)
    v[0, 7] = -30.0
    est = npy(A.prob2depth(cu(v), D, cu(np.float32([1.0])), cu(np.float32([0.5]))))
    assert np.allclose(est, 1.0 + 7 * 0.5, rtol=1e-6)
    est = npy(A.prob2depth(cu(np.zeros((1, D, 4, 5), np.float32)), D, cu(np.float32([1.0])), cu(np.float32([0.5]))))
    assert np.allclose(est, 1.0 + 0.5 * (D - 1) / 2, rtol=1e-5)
    # batch of 2 with different ranges
    rng = np.random.default_rng(0)
    vb = rng.standard_normal((2, 12, 6, 7)).astype(np.float32)
    dsb, dib = np.float32([0.5, 2.0]), np.float32([0.1, 0.3])
    assert rel_err(npy(A.prob2depth(cu(vb), 12, cu(dsb), cu(dib))), om.prob2depth(vb, 12, dsb, dib)) < 2e-6
    # large planes take the 4-pixels-per-lane kernel (16-byte plane reads); D not a multiple of the batch
    vl = (rng.standard_normal((2, 21, 384, 512)) * 3).astype(np.float32)
    el, pl = A.prob2depth(cu(vl), 21, cu(dsb), cu(dib), out_prob_map=True)
    rl, rpl = om.prob2depth(vl, 21, dsb, dib, out_prob_map=True)
    assert rel_err(npy(el), rl) < 2e-6
    assert (np.abs(npy(pl) - rpl) > 1e-5).mean() < 1e-3
    # fused x4 upsampling, sliced kernel: batch of 2, ragged output rows (4*7 = 28 < 32 lanes), D = 21 / 37 / 3
    for D_, hh, ww in ((21, 9, 7), (37, 12, 19), (3, 5, 40)):
        vu = (rng.standard_normal((2, D_, hh, ww)) * 3).astype(np.float32)
        e, eu, p, pu = A.prob2depth_upsample(cu(vu), D_, cu(dsb), cu(dib), out_prob_map=True)
        re_, reu, rp, rpu = om.prob2depth_upsample(vu, D_, dsb, dib, out_prob_map=True)
        assert eu.shape == (2, 4 * hh, 4 * ww, 1)
        assert rel_err(npy(eu), reu) < 2e-6 and rel_err(npy(e), re_) < 2e-6
        assert (np.abs(npy(pu) - rpu) > 1e-5).mean() < 2e-3


def test_full_size_properties_cfg2(A):
    """BASELINE.json configs[1] sizes (D=128, 128x160 features), where the CPU oracle is too slow: size-independent
    properties.  (a) impulse response of the halo-ring convolution = the (bf16) kernel, zero elsewhere; (b) the
    BN pass leaves zero mean / unit variance per channel; (c) soft-argmin is invariant to a logit offset, returns
    the plane depth for a one-hot volume, and the x4 variant agrees with the plain one at the shared corner pixels."""
    from atvsnet_b200.network import conv3d_raw, bn_relu_add
    D, H, W = 128, 128, 160
    rng = np.random.default_rng(3)
    # (a)
    w = torch.from_numpy((rng.standard_normal((3, 3, 3, 8, 8)) * 0.2).astype(np.float32)).to(torch.bfloat16).float().cuda()
    x = torch.zeros((1, D, H, W, 8), dtype=torch.bfloat16, device='cuda')
    pz, py, px, pc = 77, 63, 95, 5
    x[0, pz, py, px, pc] = 1.0
    A.variables.packed_cache().clear()
    raw, st = conv3d_raw(x, 'impulse', w, 8, 1, False, True)
    got = raw[0, pz - 1:pz + 2, py - 1:py + 2, px - 1:px + 2].cpu().numpy()            # out[p + 1 - k] = w[k]
    want = w[:, :, :, pc, :].cpu().numpy()[::-1, ::-1, ::-1]
    assert np.array_equal(got, want)
    assert abs(float(raw.double().sum()) - float(w[:, :, :, pc, :].double().sum())) < 1e-5
    assert int((raw != 0).sum()) <= 27 * 8
    assert np.allclose(st.cpu().numpy()[:8], w[:, :, :, pc, :].double().sum(dim=(0, 1, 2)).cpu().numpy(), atol=1e-6)
    # (b)
    xr = torch.randn((1, D, H, W, 8), device='cuda').to(torch.bfloat16)
    raw, st = conv3d_raw(xr, 'impulse', w, 8, 1, False, True, raw_dtype=torch.float16)
    y, _ = bn_relu_add(raw, st, False, [], True, False, torch.float32)
    m, v = y.double().mean(dim=(0, 1, 2, 3)), y.double().var(dim=(0, 1, 2, 3), unbiased=False)
    assert float(m.abs().max()) < 2e-3 and float((v - 1).abs().max()) < 5e-3
    # (c)
    vol = (torch.randn((1, D, H, W), device='cuda') * 3).contiguous()
    ds, di = torch.tensor([0.05], device='cuda'), torch.tensor([0.0033], device='cuda')
    e0, u0 = A.prob2depth_upsample(vol, D, ds, di)
    e1, u1 = A.prob2depth_upsample(vol + 7.5, D, ds, di)
    assert float((e0 - e1).abs().max()) < 1e-6 and float((u0 - u1).abs().max()) < 1e-6
    assert float(e0.min()) >= 0.05 and float(e0.max()) <= 0.05 + 127 * 0.0033 + 1e-6
    # align_corners x4: output corner pixels sit exactly on source corner pixels
    assert abs(float(u0[0, 0, 0, 0]) - float(e0[0, 0, 0, 0])) < 2e-6
    assert abs(float(u0[0, -1, -1, 0]) - float(e0[0, -1, -1, 0])) < 2e-5
    hot = torch.full((1, D, H, W), 40.0, device='cuda')
    hot[0, 31] = -40.0
    eh, uh = A.prob2depth_upsample(hot, D, ds, di)
    assert np.allclose(npy(eh), 0.05 + 31 * 0.0033, rtol=1e-6) and np.allclose(npy(uh), 0.05 + 31 * 0.0033, rtol=1e-6)


# ------------------------------------------------------------------ end to end (stage I + II)
# the weights bench.py times: variables.synthetic_weights() defaults (logit_gain = 4: peaked, trained-like soft-argmin)
BENCH_GAIN = 4.0


def _e2e_inputs(A, D=16, h=16, w=24, nv=3, seed=3, gain=BENCH_GAIN):
    cams = A.synthetic.orbit_cams(nv, h, w, D)[None]
    feats = A.synthetic.smooth_features(nv, h, w, 32, seed=seed)[None]
    weights = A.variables.synthetic_weights(seed=11, logit_gain=gain)
    return cams, feats, weights


def _mae_over_range(a, b, cams, D):
    return float(np.abs(a - b).mean()) / ((D - 1) * float(cams[0, 0, 1, 3, 1]))


def test_tvsnet_base_siamese_fp32(A):
    from oracle import model as om
    cams, feats, weights = _e2e_inputs(A, gain=2.0)
    A.variables.load_weights(weights)
    A.FLAGS.precision = 'fp32'
    try:
        ds, di = cams[:, 0, 1, 3, 0], cams[:, 0, 1, 3, 1]
        d, p, f, dv = A.TVSNet_base_siamese(cu(feats), cu(cams), 16, cu(ds), cu(di), view_i=2)
        do, po, fo, dvo = om.TVSNet_base_siamese(feats, cams, 16, ds, di, 2, weights)
        assert rel_err(npy(f), fo) < 5e-4 and rel_err(npy(p), po) < 5e-4
        rng_ = 15 * float(di[0])
        assert np.abs(npy(d) - do).max() < 1e-3 * rng_ and np.abs(npy(dv) - dvo).max() < 1e-3 * rng_
    finally:
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION


def test_multiview_pipeline_fp32_and_16bit(A):
    from oracle import model as om
    cams, feats, weights = _e2e_inputs(A, gain=2.0)
    A.variables.load_weights(weights)
    ref = om.run_multiview_stage12(feats, cams, 16, weights, siamese=True)
    rng_ = 15 * float(cams[0, 0, 1, 3, 1])
    A.FLAGS.precision = 'fp32'
    try:
        out = A.pipeline.run_multiview(cu(feats), cu(cams), 16, siamese=True)
    finally:
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION
    assert rel_err(npy(out['cost_volume_agg']), ref['cost_volume_agg']) < 1e-3
    assert np.abs(npy(out['depth']) - ref['depth_agg_init']).max() < 1e-3 * rng_
    assert np.abs(npy(out['depth_up']) - ref['depth_agg_init_up']).max() < 1e-3 * rng_
    for a, b in zip(out['depth_views'], ref['depth_views']):
        assert np.abs(npy(a) - b).max() < 1e-3 * rng_
    # split cost volume path (16-bit) runs too at this tiny size (8-voxel deepest level: BN statistics of 8 samples);
    # its accuracy is checked at realistic sizes below
    for prec in ('fp16', 'bf16'):
        A.FLAGS.precision = prec
        try:
            outb = A.pipeline.run_multiview(cu(feats), cu(cams), 16, siamese=True)
        finally:
            A.FLAGS.precision = A.flags.DEFAULT_PRECISION
        assert np.abs(npy(outb['depth_up']) - ref['depth_agg_init_up']).mean() / rng_ < 5e-3


def test_multiview_pipeline_16bit_depth_mae(A):
    """north_star tolerance: final depth map of the tensor-core path within a mean absolute error of 0.1 % of the depth
    range of the fp32 reference (CPU oracle), with THE WEIGHTS bench.py TIMES (logit gain 4: mean peak probability
    ~0.5), at a volume large enough (64x64x80) for the batch-norm statistics of the deepest level (8x8x10 voxels) to be
    meaningful.  fp16 storage (the default) meets it with a 3x margin; bf16 storage (8 significant bits) does not and
    is only bounded (tests/precision_emulation.py reproduces both numbers on the CPU: 0.025 % / 0.19 %)."""
    from oracle import model as om
    D, h, w = 64, 64, 80
    cams, feats, weights = _e2e_inputs(A, D=D, h=h, w=w, nv=3)
    A.variables.load_weights(weights)
    ref = om.run_multiview_stage12(feats, cams, D, weights, siamese=False)
    # the softmax over depth must be peaked enough for the bound to mean something
    p = torch.softmax(-torch.from_numpy(ref['prob_volume_agg']), dim=1)
    assert p.max(dim=1).values.mean() > 0.3
    assert A.FLAGS.precision == 'fp16'
    out16 = A.pipeline.run_multiview(cu(feats), cu(cams), D, siamese=False)
    mae = _mae_over_range(npy(out16['depth_up']), ref['depth_agg_init_up'], cams, D)
    assert mae < 1e-3, mae
    assert mae < 5e-4, mae          # measured 2.5e-4 in the CPU emulation of the storage roundings
    A.FLAGS.precision = 'bf16'
    try:
        outb = A.pipeline.run_multiview(cu(feats), cu(cams), D, siamese=False)
    finally:
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION
    maeb = _mae_over_range(npy(outb['depth_up']), ref['depth_agg_init_up'], cams, D)
    assert maeb < 4e-3, maeb
    print("depth MAE / range at 64x64x80, gain 4: fp16 %.3e  bf16 %.3e" % (mae, maeb))
    # fp32 CUDA path at the same size, against the oracle
    A.FLAGS.precision = 'fp32'
    try:
        outf = A.pipeline.run_multiview(cu(feats), cu(cams), D, siamese=False)
    finally:
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION
    assert np.abs(npy(outf['depth_up']) - ref['depth_agg_init_up']).max() < 1e-3 * (D - 1) * float(cams[0, 0, 1, 3, 1])


@pytest.mark.slow
def test_cfg2_full_size_against_oracle(A):
    """BASELINE.json configs[1] at FULL size (1 ref + 4 src, 640x512 -> 128x160x32 features, D = 128, siamese stage I +
    stage II + x4 soft-argmin), exactly bench.py's inputs and weights (make_inputs / synthetic_weights defaults): the
    fp16 tensor-core path against the CPU oracle (~1 minute of host time) within 0.1 % of the depth range."""
    from oracle import model as om
    nv, h, w, D = 5, 128, 160, 128
    cams = A.synthetic.orbit_cams(nv, h, w, D)[None]
    feats = A.synthetic.smooth_features(nv, h, w, 32, seed=0)[None]
    weights = A.variables.synthetic_weights()
    A.variables.load_weights(weights)
    assert A.FLAGS.precision == 'fp16'
    out = A.pipeline.run_multiview(cu(feats), cu(cams), D, siamese=True)
    torch.cuda.synchronize()
    ref = om.run_multiview_stage12(feats, cams, D, weights, siamese=True)
    mae = _mae_over_range(npy(out['depth_up']), ref['depth_agg_init_up'], cams, D)
    mae_lo = _mae_over_range(npy(out['depth']), ref['depth_agg_init'], cams, D)
    p = torch.softmax(-torch.from_numpy(ref['prob_volume_agg']), dim=1).max(dim=1).values.mean().item()
    print("cfg2 full size: depth_up MAE / range = %.3e (low-res %.3e), mean peak probability %.3f" % (mae, mae_lo, p))
    assert p > 0.2          # peaked, trained-like soft-argmin (a uniform softmax would be 1/128)
    assert mae < 1e-3 and mae_lo < 1e-3, (mae, mae_lo)
    for a, b in zip(out['depth_views'], ref['depth_views']):
        assert _mae_over_range(npy(a), b, cams, D) < 1e-3


def test_frame_stream_matches_run_multiview(A):
    """pipeline.FrameStream (graph replay + double-buffered H2D / D2H on side streams): every frame's depth map, in
    order, equals the plain eager call on that frame."""
    D, h, w, nv = 16, 16, 24, 3
    weights = A.variables.synthetic_weights(seed=11, logit_gain=2.0)
    A.variables.load_weights(weights)
    assert A.FLAGS.precision == A.flags.DEFAULT_PRECISION
    cams = torch.from_numpy(A.synthetic.orbit_cams(nv, h, w, D)[None])
    frames = [(torch.from_numpy(A.synthetic.smooth_features(nv, h, w, 32, seed=s)[None]).pin_memory(), cams.pin_memory())
              for s in range(5)]
    fs = A.pipeline.FrameStream(tuple(frames[0][0].shape), tuple(cams.shape), D, 'cuda:0', siamese=True)
    got = [dm.clone() for dm in fs.run(frames)]
    assert len(got) == 5
    for (fh, ch), dm in zip(frames, got):
        ref = A.pipeline.run_multiview(fh.cuda(), ch.cuda(), D, siamese=True)['depth_up']
        assert torch.equal(dm, ref.cpu())
    # a second pass through the same object reuses the captured graph
    again = [dm.clone() for dm in fs.run(frames[:2])]
    assert torch.equal(again[0], got[0]) and torch.equal(again[1], got[1])
