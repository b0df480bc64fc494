"""Drop-in for /root/reference/atvsnet/homography_warping.py on torch CUDA tensors.

Same function names, positional argument order and tensor layouts as the reference
(get_homographies :179, homography_warping :230, homography_warping_by_depth :108);
every op is one call into libatvs.so (include/atvs.h).  ``FLAGS.inverse_depth`` is read
exactly where the reference reads it (:149, :215)."""
import torch

from . import _lib as L
from .flags import FLAGS


@L.on_input_device
def get_homographies(left_cam, right_cam, depth_num, depth_start, depth_interval):
    """(B,2,4,4) x2, int, (B,), (B,) -> (B,D,3,3) fp32.  homography_warping.py:179-227."""
    L.require_cuda(left_cam, right_cam)
    lc, rc = L.f32c(left_cam), L.f32c(right_cam)
    B = lc.shape[0]
    ds = L.f32c(torch.as_tensor(depth_start, device=lc.device).reshape(-1))
    di = L.f32c(torch.as_tensor(depth_interval, device=lc.device).reshape(-1))
    if ds.numel() != B or di.numel() != B or lc.shape[1:] != (2, 4, 4) or rc.shape != lc.shape:
        raise ValueError("get_homographies: cams must be (B,2,4,4) and depth_start/interval (B,)")
    out = torch.empty((B, int(depth_num), 3, 3), dtype=torch.float32, device=lc.device)
    L.call("atvs_get_homographies", L.ptr(lc), L.ptr(rc), B, int(depth_num), L.ptr(ds), L.ptr(di),
           1 if FLAGS.inverse_depth else 0, L.ptr(out), L.stream())
    return out


def _method_code(method):
    if method == 'bilinear':
        return 0
    if method == 'nearest':
        return 1
    raise ValueError("method must be 'bilinear' or 'nearest'")


@L.on_input_device
def homography_warping(input_image, homography, method='bilinear', output_mask=False):
    """(B,H,W,C), (B,3,3) -> (B,H,W,C) [, bool (B,H,W,1)].  homography_warping.py:230-271."""
    L.require_cuda(input_image, homography)
    img, hm = L.f32c(input_image), L.f32c(homography)
    B, H, W, Cc = img.shape
    if hm.shape != (B, 3, 3):
        raise ValueError("homography must be (B,3,3)")
    out = torch.empty_like(img)
    mask = torch.empty((B, H, W, 1), dtype=torch.uint8, device=img.device) if output_mask else None
    L.call("atvs_homography_warping", L.ptr(img), L.ptr(hm), B, H, W, Cc, _method_code(method), L.ptr(out),
           L.ptr(mask), L.stream())
    return (out, mask.bool()) if output_mask else out


@L.on_input_device
def homography_warping_by_depth(input_image, left_cam, right_cam, depth_image, output_mask=False,
                                method='bilinear'):
    """homography_warping.py:108-176.  depth_image (B,H,W,1)."""
    L.require_cuda(input_image, left_cam, right_cam, depth_image)
    img, lc, rc, dep = L.f32c(input_image), L.f32c(left_cam), L.f32c(right_cam), L.f32c(depth_image)
    B, H, W, Cc = img.shape
    if dep.numel() != B * H * W:
        raise ValueError("depth_image must be (B,H,W,1)")
    out = torch.empty_like(img)
    mask = torch.empty((B, H, W, 1), dtype=torch.uint8, device=img.device) if output_mask else None
    L.call("atvs_homography_warping_by_depth", L.ptr(img), L.ptr(lc), L.ptr(rc), L.ptr(dep), B, H, W, Cc,
           _method_code(method), 1 if FLAGS.inverse_depth else 0, L.ptr(out), L.ptr(mask), L.stream())
    return (out, mask.bool()) if output_mask else out
