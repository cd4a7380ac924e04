"""CUDA drop-ins for every public function of the reference's network/render_ops.py (same names, argument
order, returned shapes and dtypes -- SURVEY.md section 8a rows a1-a7, a13, a15), each a thin launcher over the
C-ABI in include/neuray_b200.h.  The renderer itself (neuray_b200/renderer.py) does not call these: it uses the
fused point/ray kernels; these keep stand-alone callers working (e.g. reference network/init_net.py:10 imports
project_points_ref_views).

All tensors are contiguous fp32 CUDA tensors; there is no CPU path (calling with CPU tensors raises).

Autograd: the reference differentiates through exactly one of these functions -- `interpolate_feats` /
`interpolate_feature_map` with respect to the MAP (predict_mean_for_depth_loss, renderer.py:293; predict_self_hit_prob,
renderer.py:151) -- and that gradient is implemented (nr_interpolate_feats_bwd).  Every other input reaches these functions
detached in the reference (coordinates, poses, depths); if one of them requires grad while gradients are being recorded
the call raises instead of silently cutting the graph.
"""
import ctypes as C

import torch

from . import _lib
from .weights import camera_blocks

__all__ = [
    "coords2rays", "depth2points", "depth2dists", "depth2inv_dists", "interpolate_feats", "interpolate_feature_map",
    "alpha_values2hit_prob", "project_points_coords", "project_points_directions", "project_points_ref_views",
    "project_points_dict", "sample_depth", "sample_fine_depth",
]


def _no_grad_inputs(what, **tensors):
    """These launchers have no backward: refuse inputs that would need one (see the module docstring)."""
    if torch.is_grad_enabled():
        for name, t in tensors.items():
            if torch.is_tensor(t) and t.requires_grad:
                raise _lib.NeurayB200Error(
                    f"{what}: `{name}` requires grad but this CUDA drop-in has no backward for it (the reference never "
                    "differentiates this input); detach it or run under torch.no_grad()")


def _cam_of(poses, Ks, i):
    return camera_blocks({"poses": poses[i:i + 1], "Ks": Ks[i:i + 1]}, None)[0]


def coords2rays(coords, poses, Ks):
    """reference render_ops.py:4-25.  coords [n,rn,2], poses [n,3,4], Ks [n,3,3] -> centers, directions [n,rn,3]."""
    _no_grad_inputs("coords2rays", coords=coords, poses=poses, Ks=Ks)
    n, rn, _ = coords.shape
    coords = _lib.f32(coords)
    centers = torch.empty(n, rn, 3, dtype=torch.float32, device=coords.device)
    dirs = torch.empty_like(centers)
    for i in range(n):
        cam = _cam_of(poses, Ks, i)
        _lib.call("nr_coords2rays", _lib.ptr(coords[i]), _lib.ptr(cam), rn, _lib.ptr(centers[i]), _lib.ptr(dirs[i]), on=coords)
    return centers, dirs


def depth2points(que_imgs_info, que_depth):
    """reference render_ops.py:27-39 -> que_pts, que_dir [qn,rn,dn,3]."""
    _no_grad_inputs("depth2points", coords=que_imgs_info["coords"], que_depth=que_depth, poses=que_imgs_info["poses"])
    coords = _lib.f32(que_imgs_info["coords"])
    que_depth = _lib.f32(que_depth)
    qn, rn, dn = que_depth.shape
    pts = torch.empty(qn, rn, dn, 3, dtype=torch.float32, device=coords.device)
    dirs = torch.empty_like(pts)
    for i in range(qn):
        cam = _cam_of(que_imgs_info["poses"], que_imgs_info["Ks"], i)
        _lib.call("nr_depth2points", _lib.ptr(coords[i]), _lib.ptr(cam), _lib.ptr(que_depth[i]), rn, dn, _lib.ptr(pts[i]), _lib.ptr(dirs[i]),
                  on=coords)
    return pts, dirs


def depth2dists(depth):
    """reference render_ops.py:41-44."""
    _no_grad_inputs("depth2dists", depth=depth)
    depth = _lib.f32(depth)
    out = torch.empty_like(depth)
    dn = depth.shape[-1]
    _lib.call("nr_depth2dists", _lib.ptr(depth), depth.numel() // dn, dn, _lib.ptr(out), on=depth)
    return out


def depth2inv_dists(depth, depth_range):
    """reference render_ops.py:46-52.  depth [qn,rn,dn], depth_range [qn,2]."""
    _no_grad_inputs("depth2inv_dists", depth=depth)
    depth = _lib.f32(depth)
    out = torch.empty_like(depth)
    qn, rn, dn = depth.shape
    dr = _lib.f32(depth_range)
    for i in range(qn):
        _lib.call("nr_depth2inv_dists", _lib.ptr(depth[i]), _lib.ptr(dr[i]), rn, dn, _lib.ptr(out[i]), on=depth)
    return out


class _InterpFn(torch.autograd.Function):
    """Bilinear sampling of an NCHW map with the gradient with respect to the map (atomic scatter of the taps)."""

    @staticmethod
    def forward(ctx, feats, points, mask, h, w, border, align):
        f, pts = _lib.f32(feats), _lib.f32(points)
        m = _lib.f32(mask) if mask is not None else None
        b, c, ch, cw = f.shape
        n = pts.shape[1]
        out = torch.empty(b, n, c, dtype=torch.float32, device=f.device)
        _lib.call("nr_interpolate_feats", _lib.ptr(f), _lib.ptr(pts), _lib.ptr(m), b, c, ch, cw, n, float(h), float(w), border, align,
                  _lib.ptr(out), on=f)
        ctx.save_for_backward(pts, m)
        ctx.geom = (b, c, ch, cw, n, float(h), float(w), border, align)
        return out

    @staticmethod
    def backward(ctx, g):
        pts, m = ctx.saved_tensors
        b, c, ch, cw, n, h, w, border, align = ctx.geom
        g = _lib.f32(g)
        d_feats = torch.zeros(b, c, ch, cw, dtype=torch.float32, device=g.device)
        _lib.call("nr_interpolate_feats_bwd", _lib.ptr(g), _lib.ptr(pts), _lib.ptr(m), b, c, ch, cw, n, h, w, border, align, _lib.ptr(d_feats), on=g)
        return d_feats, None, None, None, None, None, None


def _interp(feats, points, mask, h, w, border, align, what):
    _no_grad_inputs(what, points=points, mask=mask)
    return _InterpFn.apply(feats, points, mask, h, w, border, align)


def interpolate_feats(feats, points, h=None, w=None, padding_mode="zeros", align_corners=False, inter_mode="bilinear"):
    """reference network/ops.py:14-34.  feats [b,f,ch,cw], points [b,n,2] -> [b,n,f].  Bilinear is the only mode any
    caller in the reference uses; 'nearest' / 'bicubic' would need their own kernels and raise."""
    if inter_mode != "bilinear":
        raise NotImplementedError(f"interpolate_feats: inter_mode={inter_mode!r} (every caller of the reference uses 'bilinear')")
    b, f, ch, cw = feats.shape
    if h is None and w is None:
        h, w = ch, cw
    return _interp(feats, points, None, h, w, 1 if padding_mode == "border" else 0, 1 if align_corners else 0, "interpolate_feats")


def interpolate_feature_map(ray_feats, coords, mask, h, w, border_type="border"):
    """reference render_ops.py:54-70.  ray_feats [rfn,f,fh,fw], coords [rfn,pn,2], mask [rfn,pn] -> [rfn,pn,f]."""
    rfn, f, fh, fw = ray_feats.shape
    align = 1 if (fh == h and fw == w) else 0
    return _interp(ray_feats, coords, mask.float(), h, w, 1 if border_type == "border" else 0, align, "interpolate_feature_map")


def alpha_values2hit_prob(alpha_values):
    """reference render_ops.py:72-80."""
    _no_grad_inputs("alpha_values2hit_prob", alpha_values=alpha_values)
    a = _lib.f32(alpha_values)
    out = torch.empty_like(a)
    dn = a.shape[-1]
    _lib.call("nr_alpha_values2hit_prob", _lib.ptr(a), a.numel() // dn, dn, _lib.ptr(out), on=a)
    return out


def _project(pts, poses, Ks, h, w, want_dir):
    _no_grad_inputs("project_points", pts=pts, poses=poses, Ks=Ks)
    pts = _lib.f32(pts)
    pn = pts.shape[0]
    rfn = poses.shape[0]
    _, vp = camera_blocks(None, {"poses": poses, "Ks": Ks})
    dev = pts.device
    pix = torch.empty(rfn, pn, 2, dtype=torch.float32, device=dev)
    depth = torch.empty(rfn, pn, 1, dtype=torch.float32, device=dev)
    mask = torch.empty(rfn, pn, dtype=torch.float32, device=dev)
    valid = torch.empty(rfn, pn, dtype=torch.float32, device=dev)
    d = torch.empty(rfn, pn, 3, dtype=torch.float32, device=dev) if want_dir else None
    _lib.call("nr_project_points", _lib.ptr(pts), pn, _lib.ptr(vp), rfn, int(h), int(w), _lib.ptr(d), _lib.ptr(pix), _lib.ptr(depth),
              _lib.ptr(mask), _lib.ptr(valid), on=pts)
    return d, pix, depth, mask, valid


def project_points_coords(pts, Rt, K):
    """reference render_ops.py:82-104 -> pts_2d [rfn,pn,2], valid [rfn,pn] bool, depth [rfn,pn,1]."""
    _, pix, depth, _, valid = _project(pts, Rt, K, 1 << 20, 1 << 20, False)
    return pix, valid > 0.5, depth


def project_points_directions(poses, points):
    """reference render_ops.py:106-115 -> [rfn,pn,3]."""
    eye = torch.eye(3, dtype=torch.float32, device=points.device)[None].expand(poses.shape[0], 3, 3)
    d, *_ = _project(points, poses, eye, 1 << 20, 1 << 20, True)
    return d


def project_points_ref_views(ref_imgs_info, que_points):
    """reference render_ops.py:117-130 -> prj_dir, prj_pts, prj_depth, valid_mask (bool)."""
    h, w = ref_imgs_info["imgs"].shape[-2:]
    d, pix, depth, mask, _ = _project(que_points, ref_imgs_info["poses"], ref_imgs_info["Ks"], h, w, True)
    return d, pix, depth, mask > 0.5


def project_points_dict(ref_imgs_info, que_pts):
    """reference render_ops.py:132-144 -> dict of [rfn,qn,rn,dn,*] tensors."""
    qn, rn, dn, _ = que_pts.shape
    prj_dir, prj_pts, prj_depth, prj_mask = project_points_ref_views(ref_imgs_info, que_pts.reshape(qn * rn * dn, 3))
    rfn, _, h, w = ref_imgs_info["imgs"].shape
    prj_ray_feats = interpolate_feature_map(ref_imgs_info["ray_feats"], prj_pts, prj_mask, h, w)
    prj_rgb = interpolate_feature_map(ref_imgs_info["imgs"], prj_pts, prj_mask, h, w)
    prj_dict = {"dir": prj_dir, "pts": prj_pts, "depth": prj_depth, "mask": prj_mask.float(),
                "ray_feats": prj_ray_feats, "rgb": prj_rgb}
    return {k: v.reshape(rfn, qn, rn, dn, -1) for k, v in prj_dict.items()}


def sample_depth(depth_range, coords, sample_num, random_sample):
    """reference render_ops.py:146-170 -> que_depth, que_dists [qn,rn,dn]."""
    qn, rn, _ = coords.shape
    dn = int(sample_num)
    assert dn > 2
    dev = coords.device
    depth = torch.empty(qn, rn, dn, dtype=torch.float32, device=dev)
    dists = torch.empty_like(depth)
    dr = _lib.f32(depth_range)
    # the uniforms come from torch's generator exactly like the reference's torch.rand(..., device=device)
    jitter = torch.rand(qn, rn, dn - 2, dtype=torch.float32, device=dev) if random_sample else None
    for i in range(qn):
        _lib.call("nr_sample_depth", _lib.ptr(dr[i]), rn, dn, _lib.ptr(jitter[i]) if jitter is not None else None, _lib.ptr(depth[i]),
                  _lib.ptr(dists[i]), on=coords)
    return depth, dists


def fine_sample_u(fdn, device):
    """Deterministic quantiles of reference render_ops.py:199-202 (same torch expression, so the same rounding)."""
    interval = 1 / fdn
    return (0.5 * interval + torch.arange(fdn) * interval).to(device).contiguous()


def sample_fine_depth(depth, hit_prob, depth_range, sample_num, random_sample, inv_mode=True):
    """reference render_ops.py:172-229 -> [qn,rn,sample_num] (unsorted)."""
    _no_grad_inputs("sample_fine_depth", depth=depth, hit_prob=hit_prob)
    depth, hit_prob = _lib.f32(depth), _lib.f32(hit_prob)
    qn, rn, dn = depth.shape
    fdn = int(sample_num)
    dev = depth.device
    out = torch.empty(qn, rn, fdn, dtype=torch.float32, device=dev)
    # the reference uses depth_range[0] for every query (render_ops.py:183)
    dr = _lib.f32(depth_range[0]) if inv_mode else None
    if random_sample:
        u = torch.rand([qn, rn, fdn]).to(dev).contiguous()      # CPU generator, like render_ops.py:205
        stride = fdn
    else:
        u = fine_sample_u(fdn, dev)
        stride = 0
    for i in range(qn):
        ui = u[i] if random_sample else u
        _lib.call("nr_sample_fine_depth", _lib.ptr(depth[i]), _lib.ptr(hit_prob[i]), _lib.ptr(dr), rn, dn, fdn, _lib.ptr(ui), stride, 0, 0,
                  _lib.ptr(out[i]), on=depth)
    return out
