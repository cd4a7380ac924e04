"""Host side of the encoders upstream of the ray path (SURVEY.md section 8f row 1), forward / inference.

    image_encoder = ResUNetLight(3, [1,2,6,4], 32, inplanes=16)   reference network/ops.py:150-230 (renderer.py:59)
    vis_encoder   = DefaultVisEncoder                              reference network/vis_encoder.py:6-21

The arithmetic runs in libneuray_b200.so (csrc/nr_encoder.cu: tensor-core implicit-GEMM convolutions with fused
InstanceNorm statistics, channel-last throughout).  This module holds
  * `ImageEncoder` / `VisEncoder`: parameter containers under the reference's state-dict names (a reference checkpoint's
    `image_encoder.*` / `vis_encoder.*` entries load unchanged) whose forward is the native path;
  * `encode_frame(owner, ref_imgs_info)`: what `NeuralRayBaseRenderer.render` does before its chunk loop
    (renderer.py:229-231), writing the results straight into the channel-last frame pack the point kernel reads.

Training: the encoders have no native backward.  With autograd enabled and parameters that require grad, `usable(owner)`
is False and `renderer.render` keeps calling the owner's own torch modules (the reference's, upstream of the boundary).
There is no CPU path: CUDA tensors only.
"""
import ctypes as C
import functools

import torch
import torch.nn as nn

from . import _lib, weights


def unet_param_names(blocks):
    """state_dict() order of the U-shaped residual encoder (ResUNetLight / ResEncoder, ops.py:150-312) with `blocks` BasicBlocks
    per stage: the first block of a stage carries the 1x1 downsample branch."""
    names = ["conv1.weight", "bn1.weight", "bn1.bias"]
    for layer, nb in enumerate(blocks, 1):
        for b in range(nb):
            p = f"layer{layer}.{b}"
            names += [f"{p}.conv1.weight", f"{p}.bn1.weight", f"{p}.bn1.bias", f"{p}.conv2.weight", f"{p}.bn2.weight", f"{p}.bn2.bias"]
            if b == 0:
                names += [f"{p}.downsample.0.weight", f"{p}.downsample.1.weight", f"{p}.downsample.1.bias"]
    for p in ("upconv3.conv", "iconv3", "upconv2.conv", "iconv2"):
        names += [f"{p}.conv.weight", f"{p}.conv.bias", f"{p}.bn.weight", f"{p}.bn.bias"]
    return names + ["out_conv.weight", "out_conv.bias"]


def unet_param_shapes(conv1_shape, blocks):
    inplanes = conv1_shape[0]
    shapes = {"conv1.weight": tuple(conv1_shape), "bn1.weight": (inplanes,), "bn1.bias": (inplanes,)}
    cin = inplanes
    for layer, (nb, cout) in enumerate(zip(blocks, (32, 64, 128)), 1):
        for b in range(nb):
            p = f"layer{layer}.{b}"
            shapes[f"{p}.conv1.weight"] = (cout, cin, 3, 3)
            shapes[f"{p}.conv2.weight"] = (cout, cout, 3, 3)
            for n in ("bn1", "bn2"):
                shapes[f"{p}.{n}.weight"] = shapes[f"{p}.{n}.bias"] = (cout,)
            if b == 0:
                shapes[f"{p}.downsample.0.weight"] = (cout, cin, 1, 1)
                shapes[f"{p}.downsample.1.weight"] = shapes[f"{p}.downsample.1.bias"] = (cout,)
            cin = cout
    for p, ci, co in (("upconv3.conv", 128, 64), ("iconv3", 128, 64), ("upconv2.conv", 64, 32), ("iconv2", 64, 32)):
        shapes[f"{p}.conv.weight"] = (co, ci, 3, 3)
        shapes[f"{p}.conv.bias"] = shapes[f"{p}.bn.weight"] = shapes[f"{p}.bn.bias"] = (co,)
    shapes["out_conv.weight"] = (32, 32, 1, 1)
    shapes["out_conv.bias"] = (32,)
    return {n: shapes[n] for n in unet_param_names(blocks)}


def image_param_names():
    """state_dict() order of ResUNetLight(3, [1,2,6,4], 32, inplanes=16) = the order nr_image_encoder_pack expects."""
    return unet_param_names((1, 2, 6))


def vis_param_names():
    """state_dict() order of DefaultVisEncoder = the order nr_vis_encoder_pack expects."""
    names = ["out_conv.0.weight"]
    for i in (1, 2):
        p = f"out_conv.{i}.conv"
        names += [f"{p}.0.weight", f"{p}.0.bias", f"{p}.2.weight", f"{p}.3.weight", f"{p}.3.bias", f"{p}.5.weight"]
    return names + ["out_conv.3.weight"]


def _image_shapes():
    return unet_param_shapes((16, 3, 7, 7), (1, 2, 6))


def _vis_shapes():
    shapes = {"out_conv.0.weight": (32, 64, 3, 3), "out_conv.3.weight": (32, 32, 1, 1)}
    for i in (1, 2):
        p = f"out_conv.{i}.conv"
        for n in ("0", "3"):
            shapes[f"{p}.{n}.weight"] = shapes[f"{p}.{n}.bias"] = (32,)
        shapes[f"{p}.2.weight"] = shapes[f"{p}.5.weight"] = (32, 32, 3, 3)
    return {n: shapes[n] for n in vis_param_names()}


class _Node(nn.Module):
    """Inner node of a parameter tree (gives the dotted state-dict names)."""


def _plant(root, shapes):
    # biases that sit next to a 4-D weight of the same module belong to a convolution
    conv_biases = {}
    for dotted, shape in shapes.items():
        if dotted.endswith(".weight") and len(shape) == 4 and dotted[:-6] + "bias" in shapes:
            conv_biases[dotted[:-6] + "bias"] = 1.0 / (shape[1] * shape[2] * shape[3]) ** 0.5
    for dotted, shape in shapes.items():
        node = root
        *path, leaf = dotted.split(".")
        for part in path:
            if not hasattr(node, part):
                node.add_module(part, _Node())
            node = getattr(node, part)
        if len(shape) == 4:        # nn.Conv2d default init (kaiming_uniform, a = sqrt(5)) bound = 1 / sqrt(fan_in)
            t = torch.empty(shape)
            bound = 1.0 / (shape[1] * shape[2] * shape[3]) ** 0.5
            nn.init.uniform_(t, -bound, bound)
        elif leaf == "weight":     # InstanceNorm2d(affine=True)
            t = torch.ones(shape)
        elif dotted in conv_biases:        # nn.Conv2d default bias init: U(-1/sqrt(fan_in), 1/sqrt(fan_in))
            t = torch.empty(shape)
            nn.init.uniform_(t, -conv_biases[dotted], conv_biases[dotted])
        else:
            t = torch.zeros(shape)
        node.register_parameter(leaf, nn.Parameter(t))


# kernels per forward: first layer 2, 3 blocks with a downsample branch x 5, 6 plain blocks x 4, 2 upsamplings, 4 conv+norm
# pairs, 2 skip copies, out_conv; vis encoder: conv0, 2 x (norm, conv, norm, conv), conv_out
IMAGE_LAUNCHES = 2 + 15 + 24 + 2 + 8 + 2 + 1
VIS_LAUNCHES = 10

# Convolution arithmetic: "fp32" = 3xTF32 tensor-core products (fp32 accuracy: parity with the fp32 reference; the default),
# "tf32" = one TF32 pass per product -- what the reference's cuDNN convolutions do on a GPU under torch's default
# torch.backends.cudnn.allow_tf32 = True (~1e-3 relative error), roughly three times fewer MMAs.
PRECISION = "fp32"


def set_precision(mode):
    global PRECISION
    if mode not in ("fp32", "tf32"):
        raise ValueError(f"encoder precision {mode!r}: 'fp32' or 'tf32'")
    PRECISION = mode


@functools.cache
def layout():
    """nr_encoder_layout: tensor counts and packed sizes of the image encoder, the vis encoder and DepthInitNet."""
    lay = _lib.NrEncoderLayout()
    _lib.check(_lib.lib().nr_encoder_layout(C.byref(lay)), "nr_encoder_layout")
    return lay


def image_dims(h, w):
    fh, fw = C.c_int(), C.c_int()
    _lib.check(_lib.lib().nr_image_encoder_dims(h, w, C.byref(fh), C.byref(fw)), "nr_image_encoder_dims")
    return fh.value, fw.value


def image_encoder_into(module, imgs, out, out_off):
    """imgs [n,3,h,w] -> channels [out_off, out_off + 32) of the channel-last buffer out [n,fh,fw,C]."""
    if not imgs.is_cuda:
        raise _lib.NeurayB200Error("the encoders need CUDA tensors (no CPU fallback)")
    n, c, h, w = imgs.shape
    if c != 3:
        raise _lib.NeurayB200Error(f"image_encoder expects [n,3,h,w] images, got {tuple(imgs.shape)}")
    dev = imgs.device
    packed = weights.packed(module, "image", image_param_names(), "nr_image_encoder_pack", layout().image_packed_floats, dev)
    nbytes = _lib.lib().nr_image_encoder_workspace(n, h, w)
    ws = _lib.workspace("image", nbytes, dev, torch.uint8)
    x = _lib.f32(imgs)
    _lib.call("nr_image_encoder_fwd", _lib.ptr(packed), _lib.ptr(x), n, h, w, _lib.ptr(out), out.shape[-1], out_off, int(PRECISION == "tf32"),
              ws.data_ptr(), nbytes, on=imgs, kernels=IMAGE_LAUNCHES)
    return out


def vis_encoder_inplace(module, feat):
    """feat [n,fh,fw,64] (ray_feats 0..31 | img_feats 32..63): channels 0..31 <- vis_encoder(ray_feats, img_feats)."""
    n, fh, fw, c = feat.shape
    if c != 64 or not feat.is_contiguous():
        raise _lib.NeurayB200Error("vis_encoder works on the contiguous [n,fh,fw,64] frame pack")
    dev = feat.device
    packed = weights.packed(module, "vis", vis_param_names(), "nr_vis_encoder_pack", layout().vis_packed_floats, dev)
    nbytes = _lib.lib().nr_vis_encoder_workspace(n, fh, fw)
    ws = _lib.workspace("vis", nbytes, dev, torch.uint8)
    _lib.call("nr_vis_encoder_fwd", _lib.ptr(packed), _lib.ptr(feat), n, fh, fw, int(PRECISION == "tf32"), ws.data_ptr(), nbytes,
              on=feat, kernels=VIS_LAUNCHES)
    return feat


def to_channel_last(x, out, out_off):
    """[n,c,h,w] -> channels [out_off, out_off + c) of out [n,h,w,C]."""
    n, c, h, w = x.shape
    xx = _lib.f32(x)
    _lib.call("nr_nchw_to_nhwc", _lib.ptr(xx), n, c, h, w, _lib.ptr(out), out.shape[-1], out_off, on=x)


def from_channel_last(buf, off, c):
    """channels [off, off + c) of buf [n,h,w,C] -> a new [n,c,h,w] tensor (the layout the reference's callers expect)."""
    n, h, w, C_ = buf.shape
    out = torch.empty(n, c, h, w, dtype=torch.float32, device=buf.device)
    _lib.call("nr_nhwc_to_nchw", _lib.ptr(buf), n, c, h, w, C_, off, _lib.ptr(out), on=buf)
    return out


class ImageEncoder(nn.Module):
    """ResUNetLight(3, [1,2,6,4], 32, inplanes=16) with the reference's parameter names; forward = the native path."""

    def __init__(self):
        super().__init__()
        _plant(self, _image_shapes())

    def forward(self, imgs):
        _refuse_training(self)
        n, _, h, w = imgs.shape
        fh, fw = image_dims(h, w)
        buf = torch.empty(n, fh, fw, 32, dtype=torch.float32, device=imgs.device)
        image_encoder_into(self, imgs, buf, 0)
        return from_channel_last(buf, 0, 32)


class VisEncoder(nn.Module):
    """DefaultVisEncoder with the reference's parameter names; forward(ray_feats, imgs_feats) = the native path."""
    default_cfg = {}

    def __init__(self, cfg=None):
        super().__init__()
        self.cfg = {**self.default_cfg, **(cfg or {})}
        _plant(self, _vis_shapes())

    def forward(self, ray_feats, imgs_feats):
        _refuse_training(self)
        n, _, fh, fw = ray_feats.shape
        feat = torch.empty(n, fh, fw, 64, dtype=torch.float32, device=ray_feats.device)
        to_channel_last(ray_feats, feat, 0)
        to_channel_last(imgs_feats, feat, 32)
        vis_encoder_inplace(self, feat)
        return from_channel_last(feat, 0, 32)


def _refuse_training(module):
    if weights.wants_grad(module):
        raise _lib.NeurayB200Error(f"{type(module).__name__}: the native encoders are forward-only; run them under torch.no_grad() "
                                   "(training keeps the torch encoders upstream of the boundary)")


def usable(owner, ref_imgs_info):
    """True when render() can run the owner's encoders natively: modules with the reference's parameter names, CUDA inputs,
    and no gradient wanted through them."""
    ie, ve = getattr(owner, "image_encoder", None), getattr(owner, "vis_encoder", None)
    if ie is None or ve is None or not ref_imgs_info["imgs"].is_cuda:
        return False
    rf = ref_imgs_info.get("ray_feats")
    if rf is None:
        from . import init_nets
        if getattr(owner, "init_net", None) is None or not init_nets.init_usable(owner.init_net, ref_imgs_info):
            return False
    if weights.wants_grad(ie, ve) or (torch.is_grad_enabled() and rf is not None and rf.requires_grad):
        return False
    return weights.has_names(ie, image_param_names()) and weights.has_names(ve, vis_param_names())


def encode_frame(owner, ref_imgs_info, feat):
    """renderer.py:229-231 on the frame pack: feat [rfn,fh,fw,64] <- (vis_encoder(ray_feats, img_feats) | img_feats).
    Also leaves NCHW 'img_feats' / 'ray_feats' in ref_imgs_info, which later callers of the reference read
    (predict_mean_for_depth_loss, renderer.py:281)."""
    imgs = ref_imgs_info["imgs"]
    if ref_imgs_info.get("ray_feats") is not None:
        to_channel_last(ref_imgs_info["ray_feats"], feat, 0)
    else:                                  # renderer.py:269 -- the owner's init net, channel-last in place
        from . import init_nets
        init_nets.init_forward_into(owner.init_net, ref_imgs_info, feat, 0)
    image_encoder_into(owner.image_encoder, imgs, feat, 32)
    vis_encoder_inplace(owner.vis_encoder, feat)
    ref_imgs_info["img_feats"] = from_channel_last(feat, 32, 32)
    ref_imgs_info["ray_feats"] = from_channel_last(feat, 0, 32)
    return feat
