"""Refinement stage (stage III of /root/reference/atvsnet/example.py:160-172) on torch CUDA tensors:
/root/reference/atvsnet/homography_warping.py:275-326 (transform_depth), :329-387 (get_visual_hull),
/root/reference/atvsnet/model.py:143-154 (extract_feature_shallow), :227-339 (refinement), :428-441 (TVSNet_refine),
/root/reference/cnn_wrapper/atvsnet.py:245-251 (ResNetDS2SPP_shallow_f16), :295-336 (CostVolRefineNet).

Geometry through the C ABI (csrc/geom.cu: atvs_transform_depth, atvs_refine_geo_group, atvs_refine_photo_group,
atvs_visual_hull, plus the existing by-depth warps and the L1_MASKED mode of K1); the refinement U-Net
(CostVolRefineNet) runs on the tensor-core kernels when FLAGS.precision is 16-bit (its 48 / 19 / 1 / 1-channel input
groups zero-padded to 64 / 32 / 8 / 8) and on the fp32 CUDA-core primitives otherwise.  Checked against
oracle/refine.py and the reference-function golden vectors (tests/test_gpu_refine.py)."""
import torch

from . import _lib as L
from . import fem
from . import network as N
from . import variables as V
from .flags import FLAGS
from .homography_warping import get_homographies, homography_warping_by_depth
from .model import build_cost_volume


@L.on_input_device
def transform_depth(left_depth, left_cam, right_cam):
    """homography_warping.py:275-326: (B,H,W,1) -> (B,H,W,1)."""
    L.require_cuda(left_depth, left_cam, right_cam)
    d, lc, rc = L.f32c(left_depth), L.f32c(left_cam), L.f32c(right_cam)
    B, H, W = d.shape[0], d.shape[1], d.shape[2]
    out = torch.empty_like(d)
    L.call("atvs_transform_depth", L.ptr(d), L.ptr(lc), L.ptr(rc), B, H, W, 1 if FLAGS.inverse_depth else 0, L.ptr(out),
           L.stream())
    return out


@L.on_input_device
def get_visual_hull(depth_images, cams, depth_num, depth_start, depth_interval, ref_id=0, view_num=2):
    """homography_warping.py:329-387 for view_num = 2: depth_images (B,N,H,W), cams (B,*,2,4,4) -> (B,D,H,W,1).  As in
    the reference the second slot is paired with cams[:, 1] whatever view it came from."""
    if view_num != 2:
        raise NotImplementedError("get_visual_hull: the refinement stage calls it with view_num = 2")
    L.require_cuda(depth_images, cams)
    di_, cams = L.f32c(depth_images), L.f32c(cams)
    order = [0, 1]
    order[0], order[ref_id] = ref_id, 0
    v = order[1]
    ref_cam, view_cam = cams[:, ref_id].contiguous(), cams[:, v].contiguous()
    ds, dint = L.f32c(depth_start).reshape(-1), L.f32c(depth_interval).reshape(-1)
    hv = get_homographies(ref_cam, view_cam, depth_num, ds, dint)
    trans = transform_depth(di_[:, v].unsqueeze(-1).contiguous(), view_cam, ref_cam)
    ref_depth = di_[:, ref_id].contiguous()
    B, H, W = ref_depth.shape
    out = torch.empty((B, int(depth_num), H, W, 1), dtype=torch.float32, device=ref_depth.device)
    L.call("atvs_visual_hull", L.ptr(ref_depth), L.ptr(trans), L.ptr(hv), L.ptr(ds), L.ptr(dint), B, int(depth_num), H, W, 2,
           1 if FLAGS.inverse_depth else 0, L.ptr(out), L.stream())
    return out


@L.on_input_device
def shallow_features(image):
    """cnn_wrapper/atvsnet.py:245-251: res_block(3, 16, 3 blocks, stride 4) + 1x1 linear conv."""
    x = fem.res_block(L.f32c(image), 'global_refine_conv0_x', 16, 3, 4, 1)
    return fem.conv2d(x, V.get_variable('global_refine_shallow_feature/kernel'))


_SHALLOW_MEMO = None      # view id -> shallow feature map, while a schedule over ONE image tensor is running


class shallow_cache(object):
    """``with refine.shallow_cache():`` around a schedule that refines several source views of the same images: the
    shallow features of a view are computed once (the reference recomputes the reference view's for every source,
    model.py:143-154 inside model.py:248).  Same numbers, (N-2) towers less."""

    def __enter__(self):
        global _SHALLOW_MEMO
        self.prev, _SHALLOW_MEMO = _SHALLOW_MEMO, {}
        return self

    def __exit__(self, *exc):
        global _SHALLOW_MEMO
        _SHALLOW_MEMO = self.prev
        return False


@L.on_input_device
def extract_feature_shallow(images, ref_id=0, view_id=1):
    """model.py:143-154."""
    if _SHALLOW_MEMO is None:
        return shallow_features(images[:, ref_id]), shallow_features(images[:, view_id])
    key = (images.data_ptr(), tuple(images.shape))
    out = []
    for v in (ref_id, view_id):
        if (key, v) not in _SHALLOW_MEMO:
            _SHALLOW_MEMO[(key, v)] = shallow_features(images[:, v])
        out.append(_SHALLOW_MEMO[(key, v)])
    return tuple(out)


def _pad_channels(x, cpad, dt):
    """(B,D,h,w,C) fp32 -> (B,D,h,w,cpad) in the activation dtype, extra channels zero: the tensor-core kernels take
    8 / 16 / 32 / 64 input channels, the refinement groups have 48 / 19 / 1 / 1 (model.py:328-333)."""
    B, D, h, w, C = x.shape
    if C == cpad:
        return N.to_dtype(x.contiguous(), dt)
    x = L.f32c(x)
    out = torch.empty((B, D, h, w, cpad), dtype=dt, device=x.device)
    L.call("atvs_pad_cast", L.ptr(x), B * D * h * w, C, cpad, L.ptr(out), L.dtype_code(out), L.stream())
    return out


def _padded_kernel(key, cpad):
    """kernel [3,3,3,Cin,Cout] zero-padded on Cin to ``cpad`` (cached next to the packed weight images)."""
    w = V.get_variable(key)
    if w.shape[-2] == cpad:
        return key, w
    cache = V.packed_cache()
    k = key + '/cin%d' % cpad
    if k not in cache:
        wp = torch.zeros(tuple(w.shape[:3]) + (cpad, w.shape[-1]), dtype=w.dtype, device=w.device)
        wp[..., :w.shape[-2], :] = w
        cache[k] = wp
    return k, cache[k]


def _cin_pad(c):
    return 8 if c <= 8 else 16 if c <= 16 else 32 if c <= 32 else 64


def _conv_bn(x, name, stride=1, transposed=False, skips=()):
    """conv_bn / deconv_bn (network.py:173-215, 511-550) + the following `add` of ``skips`` (network.py:696), in the
    dtype of ``x``: fp32 -> CUDA-core parity path, fp16 / bf16 -> tcgen05 path (fp16 raw output, fused BN + ReLU + add)."""
    key = name + ('/conv3d_transpose/kernel' if transposed else '/conv3d/kernel')
    w = V.get_variable(key)
    cout = w.shape[-2] if transposed else w.shape[-1]
    if x.dtype in N.HALF_DTYPES and not transposed:
        key, w = _padded_kernel(key, x.shape[-1])
    raw, stats = N.conv3d_raw(x, key, w, cout, stride, transposed, True, raw_dtype=N.raw_dtype_for_bn(x))
    plain, summ = N.bn_relu_add(raw, stats, True, list(skips), not skips, bool(skips), x.dtype)
    return summ if skips else plain


@L.on_input_device
def CostVolRefineNet(photo_group, geo_group, prob_vol, vis_hull):
    """cnn_wrapper/atvsnet.py:295-336 -> (global_refine_3dconv6_1 (B,D,H,W,8), global_refined_cost_vol (B,D,H,W,1)), fp32
    at the interface.  With FLAGS.precision = 'fp16' | 'bf16' the U-Net runs on the tensor-core kernels (input groups
    zero-padded to 64 / 32 / 8 / 8 channels), with 'fp32' on the CUDA-core parity path."""
    p = 'global_refine_'
    if any(int(n) % 8 for n in photo_group.shape[1:4]):
        raise ValueError("CostVolRefineNet: D, h, w must be multiples of 8 (three stride-2 levels joined by `add`), got %s"
                         % (tuple(photo_group.shape[1:4]),))
    dt = N.act_dtype()
    if dt in N.HALF_DTYPES:
        groups = [_pad_channels(g, _cin_pad(g.shape[-1]), dt) for g in (photo_group, geo_group, prob_vol, vis_hull)]
    else:
        groups = [photo_group, geo_group, prob_vol, vis_hull]
    heads = [_conv_bn(g, p + n) for g, n in zip(groups, ('photo_3dconv', 'geo_3dconv', 'prob_3dconv', 'vishull_3dconv'))]
    cat = torch.cat(heads, dim=-1).contiguous()
    c10 = _conv_bn(cat, p + '3dconv1_0', 2)
    c20 = _conv_bn(c10, p + '3dconv2_0', 2)
    c30 = _conv_bn(c20, p + '3dconv3_0', 2)
    c01 = _conv_bn(cat, p + '3dconv0_1')
    c11 = _conv_bn(c10, p + '3dconv1_1')
    c21 = _conv_bn(c20, p + '3dconv2_1')
    c31 = _conv_bn(c30, p + '3dconv3_1')
    c41 = _conv_bn(c31, p + '3dconv4_0', 2, True, skips=(c21,))
    c51 = _conv_bn(c41, p + '3dconv5_0', 2, True, skips=(c11,))
    c61 = _conv_bn(c51, p + '3dconv6_0', 2, True, skips=(c01,))
    wk = V.get_variable('global_refined_cost_vol/kernel')
    res, _ = N.conv3d_raw(c61, 'global_refined_cost_vol/kernel', wk, 1, 1, False, False)
    return N.to_dtype(c61, torch.float32), res


@L.on_input_device
def refinement(init_depth_images, cams, depth_num, depth_start, depth_interval, images, prob_vol, ref_id, view_id,
               view_homographies=None, num_depths=None, depth_ref_id=None, depth_view_id=None):
    """model.py:227-339: init_depth_images (B,2,h,w,1), images (B,N,H,W,3), prob_vol (B,D,h,w) ->
    (cost residual (B,D,h,w,8), prob residual (B,D,h,w)), fp32."""
    depth_ref_id = ref_id if depth_ref_id is None else depth_ref_id
    depth_view_id = view_id if depth_view_id is None else depth_view_id
    num_depths = FLAGS.view_num if num_depths is None else num_depths
    L.require_cuda(init_depth_images, cams, images, prob_vol)
    init, cams = L.f32c(init_depth_images), L.f32c(cams)
    D = int(depth_num)
    ds, dint = L.f32c(depth_start).reshape(-1), L.f32c(depth_interval).reshape(-1)
    d_ref = init[:, depth_ref_id].contiguous()
    d_view = init[:, depth_view_id].contiguous()
    ref_cam, view_cam = cams[:, ref_id].contiguous(), cams[:, view_id].contiguous()
    d_view_t = transform_depth(d_view, view_cam, ref_cam)
    hv = view_homographies if view_homographies is not None else get_homographies(ref_cam, view_cam, D, ds, dint)
    ref_f, view_f = extract_feature_shallow(images, ref_id, view_id)
    B, h, w, C = ref_f.shape
    # photometric L1 cost volume (K1, L1_MASKED mode) + by-depth photo error + tiled reference feature
    cost_photo = build_cost_volume(ref_f, view_f, cams, D, ds, dint, ref_id, view_id, mode='l1_masked',
                                   out_dtype=torch.float32)
    wf, mp = homography_warping_by_depth(view_f, ref_cam, view_cam, d_ref, output_mask=True)
    photo_group = torch.empty((B, D, h, w, 3 * C), dtype=torch.float32, device=ref_f.device)
    L.call("atvs_refine_photo_group", L.ptr(cost_photo), L.ptr(wf), L.ptr(mp.to(torch.uint8).contiguous()), L.ptr(ref_f), B, D,
           h, w, C, L.ptr(photo_group), L.stream())
    # geometric volumes
    wg, mg = homography_warping_by_depth(d_view_t, ref_cam, view_cam, d_ref, output_mask=True, method='nearest')
    geo_group = torch.empty((B, D, h, w, C + 3), dtype=torch.float32, device=ref_f.device)
    L.call("atvs_refine_geo_group", L.ptr(d_ref), L.ptr(d_view_t), L.ptr(hv), L.ptr(wg), L.ptr(mg.to(torch.uint8).contiguous()),
           L.ptr(ds), L.ptr(dint), B, D, h, w, C, L.ptr(geo_group), L.stream())
    vis = get_visual_hull(init[..., 0], cams, D, ds, dint, ref_id=ref_id, view_num=num_depths)
    pv = L.f32c(prob_vol).unsqueeze(-1).contiguous()
    c61, res = CostVolRefineNet(photo_group, geo_group, pv, vis)
    return c61, res.squeeze(-1)


@L.on_input_device
def TVSNet_refine(depth_b2, depth_view, prob_vol_b2, filtered_cost_volume, images, cams, depth_num, depth_start,
                  depth_interval, view_i, ref_i=0):
    """model.py:428-441 -> (refined_prob_vol (B,D,h,w), refined_cost_volume (B,D,h,w,8))."""
    init = torch.stack([L.f32c(depth_b2), L.f32c(depth_view)], dim=1).contiguous()
    cost_res, prob_res = refinement(init, cams, depth_num, depth_start, depth_interval, images, prob_vol_b2, ref_i, view_i,
                                    num_depths=2, depth_ref_id=0, depth_view_id=1)
    pv, fc = L.f32c(prob_vol_b2), L.f32c(filtered_cost_volume)
    return fem.add(pv, prob_res.contiguous()), fem.add(fc, cost_res)
