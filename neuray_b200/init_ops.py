"""CUDA drop-in for the per-frame geometric consistency features of the reference's DepthInitNet
(network/init_net.py:29-61, SURVEY.md section 8f row 2): `get_diff_feats(ref_imgs_info, depth_in)`.

Same name, arguments and result ([rfn,8,h,w]) as the reference function; one fused launch (nr_diff_feats) instead of the
reference's chain of [rfn, rfn*h*w, *] intermediates.  Inputs carry no gradient in the reference (images, depth maps and
cameras come from the data loader), so there is no backward; an input that requires grad raises.
"""
import torch

from . import _lib
from .render_ops import _no_grad_inputs
from .weights import camera_blocks

__all__ = ["get_diff_feats"]


def get_diff_feats(ref_imgs_info, depth_in):
    imgs = ref_imgs_info["imgs"]
    _no_grad_inputs("get_diff_feats", imgs=imgs, depth_in=depth_in, poses=ref_imgs_info["poses"], Ks=ref_imgs_info["Ks"])
    rfn, _, h, w = imgs.shape
    if depth_in.shape != (rfn, 1, h, w):
        raise _lib.NeurayB200Error(f"depth_in {tuple(depth_in.shape)} must be [rfn,1,h,w] = {(rfn, 1, h, w)}")
    imgs_c, depth_c, poses_c, ks_c = (_lib.f32(t) for t in (imgs, depth_in, ref_imgs_info["poses"], ref_imgs_info["Ks"]))
    _, vp = camera_blocks(None, ref_imgs_info)
    out = torch.empty(rfn, 8, h, w, dtype=torch.float32, device=imgs.device)
    _lib.call("nr_diff_feats", _lib.ptr(imgs_c), _lib.ptr(depth_c), _lib.ptr(poses_c), _lib.ptr(ks_c), _lib.ptr(vp), rfn, h, w, _lib.ptr(out),
              on=imgs)
    return out
