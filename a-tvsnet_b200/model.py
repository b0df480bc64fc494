"""Drop-in for the hot-path functions of /root/reference/atvsnet/model.py on torch CUDA
tensors: get_propability_map :13, prob2depth :80, prob2depth_upsample :113, output_conv
:132, build_cost_volume :157, cost_volume_reasoning :204, TVSNet_base :380,
TVSNet :346, TVSNet_base :380, TVSNet_base_siamese :398, TVSNet_feature_extraction :420,
TVSNet_refine :428, cost_volume_aggregation(_refine) :445/:460.  Same names, positional
argument order, layouts and depth-plane conventions; ``reuse`` is accepted and ignored.
The TVSNet_* entry points take ``images`` (B,N,H,W,3) as the reference does and run the 2-D
feature extractor (fem.ResNetDS2SPP) on the two views they use; a tensor whose last
dimension is not 3 is taken to be the (B,N,h,w,32) FEATURE tensor (extension: lets a caller
that already holds the features skip the FEM, e.g. pipeline.run_multiview)."""
import torch

from . import _lib as L
from .atvsnet import (AttAggregation, AttAggregation_keepchannel, AttAggregation_refine,
                      AttAggregation_refine_keepchannel, OutputConv, OutputConv_refine, StackedUNet,
                      StackedUNet_prob)
from .flags import FLAGS
from .homography_warping import get_homographies
from .network import act_dtype

AUTO_REUSE = 'AUTO_REUSE'


def _vec(x, B, device):
    t = torch.as_tensor(x, dtype=torch.float32, device=device).reshape(-1)
    if t.numel() == 1 and B > 1:
        t = t.expand(B)
    return t.contiguous()


def _prob2depth(prob_volume, depth_start, depth_interval, up, out_prob_map):
    L.require_cuda(prob_volume)
    v = L.f32c(prob_volume)
    B, D, H, W = v.shape
    ds, di = _vec(depth_start, B, v.device), _vec(depth_interval, B, v.device)
    est = torch.empty((B, H * up, W * up, 1), dtype=torch.float32, device=v.device)
    pm = torch.empty_like(est) if out_prob_map else None
    L.call("atvs_prob2depth", L.ptr(v), B, D, H, W, L.ptr(ds), L.ptr(di), up, L.ptr(est), L.ptr(pm), L.stream())
    return est, pm


@L.on_input_device
def prob2depth(prob_volume, depth_num, depth_start, depth_interval, out_prob_map=False):
    """(B,D,H,W) logits -> (B,H,W,1) [, prob map (B,H,W,1)].  model.py:80-109 (+ :13-65)."""
    if int(depth_num) != prob_volume.shape[1]:
        raise ValueError("depth_num (%d) != prob_volume.shape[1] (%d)" % (depth_num, prob_volume.shape[1]))
    est, pm = _prob2depth(prob_volume, depth_start, depth_interval, 1, out_prob_map)
    return (est, pm) if out_prob_map else est


@L.on_input_device
def prob2depth_upsample(prob_volume, depth_num, depth_start, depth_interval, out_prob_map=False):
    """model.py:113-129: (est, est_up[, prob, prob_up]); the x4 bilinear logit upsample
    (:68-76) is fused into the soft-argmin kernel and never materialised."""
    if int(depth_num) != prob_volume.shape[1]:
        raise ValueError("depth_num != prob_volume.shape[1]")
    est_up, pm_up = _prob2depth(prob_volume, depth_start, depth_interval, 4, out_prob_map)
    est, pm = _prob2depth(prob_volume, depth_start, depth_interval, 1, out_prob_map)
    if out_prob_map:
        return est, est_up, pm, pm_up
    return est, est_up


@L.on_input_device
def output_conv(cost_volume, reuse=AUTO_REUSE):
    """model.py:132-135: (B,D,H,W,C) -> (B,D,H,W)."""
    return OutputConv({'data': cost_volume}, is_training=True, reuse=reuse).get_output().squeeze(-1)


@L.on_input_device
def output_conv_refine(cost_volume, reuse=AUTO_REUSE):
    """model.py:137-140."""
    return OutputConv_refine({'data': cost_volume}, is_training=True, reuse=reuse).get_output().squeeze(-1)


_MODES = {'concat': 0, 'warped_only': 1, 'l1_masked': 2}


@L.on_input_device
def build_cost_volume(ref_feature, view_feature, cams, depth_num, depth_start, depth_interval, ref_id, view_id,
                      output_homo=False, warp_ref=False, mode='concat', out_dtype=torch.float32):
    """model.py:157-200: (B,h,w,F) x2, cams (B,N,2,4,4) -> (B,D,h,w,2F) [, (B,D,3,3)].
    One fused kernel per call: per depth plane homography + bilinear sample + concat with the
    reference feature, streamed straight to the output volume (no warped stack/tile/concat
    intermediates).  ``mode``/``out_dtype`` are extensions (defaults = reference behaviour)."""
    L.require_cuda(ref_feature, view_feature, cams)
    # a 16-bit view feature map in the volume's own dtype (e.g. converted once per frame, pipeline.run_multiview) is
    # gathered from directly: one launch, no per-call conversion
    src16 = view_feature.dtype in (torch.float16, torch.bfloat16)
    if src16 and (view_feature.dtype != out_dtype or warp_ref):
        raise ValueError("build_cost_volume: a 16-bit view feature map needs out_dtype == its dtype and warp_ref=False")
    ref, cams = L.f32c(ref_feature), L.f32c(cams)
    view = view_feature.contiguous() if src16 else L.f32c(view_feature)
    B, h, w, F = ref.shape
    D = int(depth_num)
    ref_cam = cams[:, ref_id].contiguous()
    view_cam = cams[:, view_id].contiguous()
    hv = get_homographies(ref_cam, view_cam, depth_num=D, depth_start=depth_start, depth_interval=depth_interval)
    hr = get_homographies(ref_cam, ref_cam, depth_num=D, depth_start=depth_start,
                          depth_interval=depth_interval) if warp_ref else None
    m = _MODES[mode]
    cout = 2 * F if m == 0 else F
    out = torch.empty((B, D, h, w, cout), dtype=out_dtype, device=ref.device)
    if src16:
        L.call("atvs_build_cost_volume_src16", L.ptr(ref), L.ptr(view), L.ptr(hv), B, D, h, w, F, m, L.dtype_code(out),
               L.ptr(out), L.stream())
    else:
        L.call("atvs_build_cost_volume", L.ptr(ref), L.ptr(view), L.ptr(hv), L.ptr(hr), B, D, h, w, F, m,
               L.dtype_code(out), L.ptr(out), L.stream())
    return (out, hv) if output_homo else out


@L.on_input_device
def cost_volume_reasoning(cost_volume, output_prob=True, output_filtered_cost=False, reuse=AUTO_REUSE):
    """model.py:204-223 (CRM): (B,D,h,w,2F) -> (B,D,h,w) and/or (B,D,h,w,C) fp32."""
    if output_prob:
        outs = ('conv_b2_6_2', 'conv_b2_6_1') if output_filtered_cost else ('conv_b2_6_2',)
        tower = StackedUNet_prob({'data': cost_volume}, is_training=True, reuse=reuse, outputs=outs)
        prob = tower.get_output().squeeze(-1)
        if output_filtered_cost:
            return prob, tower.get_output_by_name('conv_b2_6_1').float()
        return prob
    tower = StackedUNet({'data': cost_volume}, is_training=True, reuse=reuse, outputs=('conv_b2_6_1',))
    return tower.get_output_by_name('conv_b2_6_1').float()


@L.on_input_device
def cost_volume_aggregation(cost_volumes, reuse=AUTO_REUSE, keepchannel=False):
    """model.py:445-456 (AAM1): (B,D,h,w,C,N-1) -> (B,D,h,w,C) | (B,D,h,w).  A list of N-1
    (B,D,h,w,C) tensors is accepted too (avoids the host-side np.stack of example.py:150)."""
    if keepchannel:
        return AttAggregation_keepchannel({'data': cost_volumes}, is_training=True, reuse=reuse).get_output()
    return AttAggregation({'data': cost_volumes}, is_training=True, reuse=reuse).get_output().squeeze(-1)


@L.on_input_device
def cost_volume_aggregation_refine(cost_volumes, reuse=AUTO_REUSE, keepchannel=False):
    """model.py:460-468 (AAM2)."""
    if keepchannel:
        return AttAggregation_refine_keepchannel({'data': cost_volumes}, is_training=True, reuse=reuse).get_output()
    return AttAggregation_refine({'data': cost_volumes}, is_training=True, reuse=reuse).get_output().squeeze(-1)


def _cost_dtype():
    return act_dtype()


@L.on_input_device
def TVSNet_feature_extraction(images, view_i):
    """model.py:420-425: images (B,N,H,W,3) -> FEM feature of view ``view_i`` (B,H/4,W/4,32)."""
    from . import fem
    L.require_cuda(images)
    if images.shape[-1] != 3:
        raise ValueError("TVSNet_feature_extraction expects images (B,N,H,W,3), got %s" % (tuple(images.shape),))
    return fem.ResNetDS2SPP(images[:, view_i])


def _pair_features(images, ref_i, view_i):
    """(ref_feature, view_feature) of an image tensor (B,N,H,W,3) through the FEM, or slices of a feature tensor
    (B,N,h,w,F) when the caller already holds features."""
    if images.shape[-1] == 3:
        return TVSNet_feature_extraction(images, ref_i), TVSNet_feature_extraction(images, view_i)
    return images[:, ref_i], images[:, view_i]


def _tvsnet_base(ref, view, cams, depth_num, depth_start, depth_interval, view_i):
    cost_vol = build_cost_volume(ref, view, cams, depth_num, depth_start, depth_interval, ref_id=0, view_id=view_i,
                                 out_dtype=_cost_dtype())
    prob_vol_b2, filtered = cost_volume_reasoning(cost_vol, output_filtered_cost=True)
    depth_b2 = prob2depth(prob_vol_b2, depth_num, depth_start, depth_interval, out_prob_map=False)
    return depth_b2, prob_vol_b2, filtered


def _tvsnet_reverse(ref, view, cams, depth_num, depth_start, depth_interval, view_i):
    cost_vol_view = build_cost_volume(view, ref, cams, depth_num, depth_start, depth_interval, ref_id=view_i, view_id=0,
                                      out_dtype=_cost_dtype())
    prob_vol_view = cost_volume_reasoning(cost_vol_view, output_filtered_cost=False, reuse=AUTO_REUSE)
    return prob2depth(prob_vol_view, depth_num, depth_start, depth_interval, out_prob_map=False)


@L.on_input_device
def TVSNet_base(images, cams, depth_num, depth_start, depth_interval, view_i, ref_i=0):
    """model.py:380-395: images (B,N,H,W,3), cams (B,N,2,4,4) -> (depth_b2 (B,h,w,1), prob_vol_b2 (B,D,h,w),
    filtered_cost_volume (B,D,h,w,8))."""
    ref, view = _pair_features(images, ref_i, view_i)
    return _tvsnet_base(ref, view, cams, depth_num, depth_start, depth_interval, view_i)


@L.on_input_device
def TVSNet_base_siamese(images, cams, depth_num, depth_start, depth_interval, view_i, ref_i=0):
    """model.py:398-417: forward volume (ref <- view_i) and the reverse one (view_i as reference) for
    ``depth_view``; -> (depth_b2, prob_vol_b2, filtered_cost_volume, depth_view)."""
    ref, view = _pair_features(images, ref_i, view_i)
    depth_b2, prob_vol_b2, filtered = _tvsnet_base(ref, view, cams, depth_num, depth_start, depth_interval, view_i)
    depth_view = _tvsnet_reverse(ref, view, cams, depth_num, depth_start, depth_interval, view_i)
    return depth_b2, prob_vol_b2, filtered, depth_view


@L.on_input_device
def TVSNet(images, cams, depth_num, depth_start, depth_interval, view_i, ref_i=0):
    """model.py:346-377, the two-view network: FEM on both images, both directions of the cost volume + CRM, then the
    refinement stage on (depth_b2, depth_view) -> refined_prob_vol (B,D,h,w) = prob_vol_b2 + residual."""
    from . import refine
    if images.shape[-1] != 3:
        raise ValueError("TVSNet (two-view, with refinement) needs the images (B,N,H,W,3), got %s" % (tuple(images.shape),))
    ref, view = _pair_features(images, ref_i, view_i)
    depth_view = _tvsnet_reverse(ref, view, cams, depth_num, depth_start, depth_interval, view_i)
    depth_b2, prob_vol_b2, _ = _tvsnet_base(ref, view, cams, depth_num, depth_start, depth_interval, view_i)
    init = torch.stack([L.f32c(depth_b2), L.f32c(depth_view)], dim=1).contiguous()
    _, prob_residual = refine.refinement(init, cams, depth_num, depth_start, depth_interval, images, prob_vol_b2,
                                         ref_id=ref_i, view_id=view_i, view_homographies=None, num_depths=2,
                                         depth_ref_id=0, depth_view_id=1)
    return refine.fem.add(L.f32c(prob_vol_b2), prob_residual.contiguous())


@L.on_input_device
def TVSNet_refine(depth_b2, depth_view, prob_vol_b2, filtered_cost_volume, images, cams, depth_num, depth_start,
                  depth_interval, view_i, ref_i=0):
    """model.py:428-441 -> (refined_prob_vol (B,D,h,w), refined_cost_volume (B,D,h,w,8))."""
    from . import refine
    return refine.TVSNet_refine(depth_b2, depth_view, prob_vol_b2, filtered_cost_volume, images, cams, depth_num,
                                depth_start, depth_interval, view_i, ref_i)
