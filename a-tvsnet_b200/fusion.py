"""Depth-map fusion (SURVEY.md 8(f) row N4): what /root/reference/atvsnet/depth_fusion.py does by converting the depth
maps to Gipuma files and shelling out to the `fusibile` executable (fusibile/fusibile.cu:138-277 + main.cpp), as one call
on device tensors: probability filter (depth_fusion.py:183-202), fake normals (:93-112), camera set-up (:69-91 and
fusibile/cameraGeometryUtils.h:388-444), consistency kernel for ALL reference views in one launch and device-side
compaction of the point cloud (csrc/fusion.cu).  PLY writing is host-side NumPy as in the reference's displayUtils."""
import numpy as np
import torch

from . import _lib as L


def probability_filter(depth, prob, prob_threshold=0.8):
    """depth_fusion.py:183-202: depth[prob < threshold] = 0 (tensors, any shape)."""
    return torch.where(prob < prob_threshold, torch.zeros_like(depth), depth)


def fake_normals(depth):
    """depth_fusion.py:93-112: (1,1,1)/1.732050808 where depth > 0, zero elsewhere: (...,) -> (...,3)."""
    n = (depth > 0).to(torch.float32).unsqueeze(-1) * (1.0 / 1.732050808)
    return n.expand(depth.shape + (3,)).contiguous()


def cameras_from_krt(K, R, t):
    """K (N,3,3), R (N,3,3), t (N,3) (host arrays) -> device tensors P (N,3,4), M_inv (N,3,3), C (N,3), f (N)
    (P = (K E)[0:3]: depth_fusion.py:69-91; M_inv, C, f: cameraGeometryUtils.h:388, 434, 405)."""
    K, R, t = np.asarray(K, np.float64), np.asarray(R, np.float64), np.asarray(t, np.float64).reshape(-1, 3)
    P = np.einsum('nij,njk->nik', K, np.concatenate([R, t[:, :, None]], axis=2))
    Minv = np.linalg.inv(P[:, :, :3])
    C = -np.einsum('nji,nj->ni', R, t)
    f = K[:, 0, 0]
    return tuple(torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda() for a in (P, Minv, C, f))


@L.on_input_device
def fuse_depth_maps(depths, cams, images=None, normals=None, disp_thresh=0.01, num_consistent=2, normal_thresh_deg=360.0,
                    capacity=None):
    """depths (N,H,W) fp32 cuda (0 = no measurement), cams = cameras_from_krt(...), images (N,H,W,3|4) fp32 or None,
    normals (N,H,W,3) or None (-> fake normals) -> dict(points (M,3), normals (M,3), colors (M,4) | None, count)."""
    L.require_cuda(depths)
    d = L.f32c(depths)
    N, H, W = d.shape
    nrm = L.f32c(normals) if normals is not None else fake_normals(d)
    nd = torch.cat([nrm, d.unsqueeze(-1)], dim=-1).contiguous()
    img = None
    if images is not None:
        img = L.f32c(images)
        if img.shape[-1] == 3:
            img = torch.cat([img, torch.zeros_like(img[..., :1])], dim=-1).contiguous()
    P, Minv, C, f = cams
    cap = int(capacity if capacity is not None else N * H * W)
    ws = torch.empty(L.load().atvs_fuse_workspace_bytes(N, H, W), dtype=torch.uint8, device=d.device)
    pts = torch.empty((cap, 3), dtype=torch.float32, device=d.device)
    nout = torch.empty((cap, 3), dtype=torch.float32, device=d.device)
    tex = torch.empty((cap, 4), dtype=torch.float32, device=d.device) if img is not None else None
    count = torch.zeros(1, dtype=torch.int64, device=d.device)
    L.call("atvs_fuse_depth_maps", L.ptr(nd), L.ptr(img), L.ptr(P), L.ptr(Minv), L.ptr(C), L.ptr(f), N, H, W, float(disp_thresh),
           float(np.deg2rad(normal_thresh_deg)), int(num_consistent), 1 if img is not None else 0, L.ptr(ws), cap, L.ptr(pts),
           L.ptr(nout), L.ptr(tex), L.ptr(count), L.stream())
    m = min(int(count.item()), cap)
    return dict(points=pts[:m], normals=nout[:m], colors=tex[:m] if tex is not None else None, count=int(count.item()))


def write_ply(path, points, normals=None, colors=None):
    """binary little-endian PLY of the fused cloud (fusibile/displayUtils.h:80 storePlyFileBinaryPointCloud: x y z nx ny nz
    r g b per vertex)."""
    pts = points.detach().cpu().numpy().astype('<f4')
    n = pts.shape[0]
    nr = normals.detach().cpu().numpy().astype('<f4') if normals is not None else np.zeros((n, 3), '<f4')
    if colors is not None:
        c = colors.detach().cpu().numpy()[:, :3]
        rgb = np.clip(c[:, ::-1], 0, 255).astype(np.uint8)          # stored BGR (cv2), written as r g b
    else:
        rgb = np.zeros((n, 3), np.uint8)
    rec = np.empty(n, dtype=[('p', '<f4', 3), ('n', '<f4', 3), ('c', 'u1', 3)])
    rec['p'], rec['n'], rec['c'] = pts, nr, rgb
    with open(path, 'wb') as fh:
        fh.write(("ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n"
                  "property float nx\nproperty float ny\nproperty float nz\nproperty uchar red\nproperty uchar green\n"
                  "property uchar blue\nend_header\n" % n).encode('ascii'))
        fh.write(rec.tobytes())
