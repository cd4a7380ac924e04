"""Host side of DepthInitNet, the init net of the neuray_gen_depth model (reference network/init_net.py:63-101), forward /
inference:

    depth      = extract_depth_for_init(ref_imgs_info)                       nr_extract_depth
    diff_feats = get_diff_feats(ref_imgs_info, depth)                        nr_diff_feats (neuray_b200.init_ops)
    feats      = res_net(cat([imgs, depth, diff_feats]))                     ResEncoder (ops.py:232-312) on the tensor cores
    ray_feats  = conv_out(cat([depth_skip(depth), feats]))                   nr_depth_init_fwd

`DepthInitNet` is a parameter container under the reference's state-dict names whose forward is the native path (it returns
the reference's NCHW [rfn,32,h/4,w/4] tensor); `forward_into` writes channel-last straight into the frame pack, where the
vis encoder expects the init net's ray_feats.  `patch.install()` puts `forward_or_reference` over the reference class'
forward: with a gradient wanted through the net (training) the reference's own torch code runs.  CUDA tensors only.
"""
import ctypes as C
import functools

import torch
import torch.nn as nn

from . import _lib, encoders, init_ops, weights

BLOCKS = (2, 2, 2)
LAUNCHES = 3 + 2 + 3 * (5 + 4) + 2 + 8 + 2 + 1 + 1 + 1       # input assembly, first layer, 3 stages, decoder, out_conv, depth_skip, conv_out


def param_names():
    """state_dict() order of DepthInitNet = the order nr_depth_init_pack expects (72 tensors)."""
    return (["res_net." + n for n in encoders.unet_param_names(BLOCKS)] +
            ["depth_skip.0.weight", "depth_skip.0.bias", "depth_skip.2.weight", "depth_skip.2.bias", "conv_out.weight", "conv_out.bias"])


def _shapes():
    shapes = {"res_net." + k: v for k, v in encoders.unet_param_shapes((32, 12, 8, 8), BLOCKS).items()}
    shapes.update({"depth_skip.0.weight": (8, 1, 2, 2), "depth_skip.0.bias": (8,), "depth_skip.2.weight": (16, 8, 2, 2), "depth_skip.2.bias": (16,),
                   "conv_out.weight": (32, 48, 1, 1), "conv_out.bias": (32,)})
    return {n: shapes[n] for n in param_names()}


def dims(h, w):
    fh, fw = C.c_int(), C.c_int()
    _lib.check(_lib.lib().nr_depth_init_dims(h, w, C.byref(fh), C.byref(fw)), "nr_depth_init_dims")
    return fh.value, fw.value


def usable(module, ref_imgs_info):
    return ref_imgs_info["imgs"].is_cuda and weights.has_names(module, param_names()) and not weights.wants_grad(module)


def extract_depth_for_init(ref_imgs_info):
    """init_net.py:76-79 -> [rfn,1,h,w] normalised inverse depth."""
    depth, rng = ref_imgs_info["depth"], ref_imgs_info["depth_range"]
    rfn, _, h, w = depth.shape
    d, r = _lib.f32(depth), _lib.f32(rng)
    out = torch.empty_like(d)
    _lib.call("nr_extract_depth", _lib.ptr(d), _lib.ptr(r), rfn, h, w, _lib.ptr(out), on=depth)
    return out


def forward_into(module, ref_imgs_info, out, out_off):
    """DepthInitNet.forward (init_net.py:93-101) into channels [out_off, out_off + 32) of the channel-last buffer out."""
    imgs = ref_imgs_info["imgs"]
    if not imgs.is_cuda:
        raise _lib.NeurayB200Error("DepthInitNet needs CUDA tensors (no CPU fallback)")
    rfn, _, h, w = imgs.shape
    dev = imgs.device
    depth = extract_depth_for_init(ref_imgs_info)
    diff = init_ops.get_diff_feats(ref_imgs_info, depth)
    packed = weights.packed(module, "depth_init", param_names(), "nr_depth_init_pack", encoders.layout().depth_init_packed_floats, dev)
    nbytes = _lib.lib().nr_depth_init_workspace(rfn, h, w)
    ws = _lib.workspace("depth_init", nbytes, dev, torch.uint8)
    x = _lib.f32(imgs)
    _lib.call("nr_depth_init_fwd", _lib.ptr(packed), _lib.ptr(x), _lib.ptr(depth), _lib.ptr(diff.contiguous()), rfn, h, w, _lib.ptr(out),
              out.shape[-1], out_off, int(encoders.PRECISION == "tf32"), ws.data_ptr(), nbytes, on=imgs, kernels=LAUNCHES)
    return out


def forward_nchw(module, ref_imgs_info):
    imgs = ref_imgs_info["imgs"]
    rfn, _, h, w = imgs.shape
    fh, fw = dims(h, w)
    buf = torch.empty(rfn, fh, fw, 32, dtype=torch.float32, device=imgs.device)
    forward_into(module, ref_imgs_info, buf, 0)
    return encoders.from_channel_last(buf, 0, 32)


class DepthInitNet(nn.Module):
    """reference init_net.py:76-101 with the reference's parameter names; forward(ref_imgs_info, src_imgs_info, is_train)."""
    default_cfg = {}

    def __init__(self, cfg=None):
        super().__init__()
        self.cfg = {**self.default_cfg, **(cfg or {})}
        encoders._plant(self, _shapes())

    def forward(self, ref_imgs_info, src_imgs_info=None, is_train=False):
        if not usable(self, ref_imgs_info):
            raise _lib.NeurayB200Error("DepthInitNet: the native init net is forward-only and CUDA-only; run it under torch.no_grad() "
                                       "(training keeps the torch module upstream of the boundary)")
        return forward_nchw(self, ref_imgs_info)


def forward_or_reference(reference_forward):
    """The forward patch.install() puts over the reference's DepthInitNet: native when no gradient is wanted through the net."""
    def forward(self, ref_imgs_info, src_imgs_info, is_train):
        if usable(self, ref_imgs_info):
            return forward_nchw(self, ref_imgs_info)
        return reference_forward(self, ref_imgs_info, src_imgs_info, is_train)
    return forward


# ---- CostVolumeInitNet (reference network/init_net.py:205-254; SURVEY.md 8f row 4) ---------------------------------------------------

def mvsnet_tensor_names():
    """MVSNet.state_dict() order (network/mvsnet/mvsnet.py:7-66) = the order nr_mvsnet_pack expects (89 tensors)."""
    bn = lambda p: [f"{p}.weight", f"{p}.bias", f"{p}.running_mean", f"{p}.running_var"]
    names = []
    for i in range(7):
        names += [f"feature.conv{i}.conv.weight"] + bn(f"feature.conv{i}.bn")
    names += ["feature.feature.weight", "feature.feature.bias"]
    for i in range(7):
        names += [f"cost_regularization.conv{i}.conv.weight"] + bn(f"cost_regularization.conv{i}.bn")
    for i in (7, 9, 11):
        names += [f"cost_regularization.conv{i}.0.weight"] + bn(f"cost_regularization.conv{i}.1")
    return names + ["cost_regularization.prob.weight", "cost_regularization.prob.bias"]


def _mvsnet_shapes():
    s = {}
    for name, (ci, co, k) in zip([f"feature.conv{i}" for i in range(7)], [(3, 8, 3), (8, 8, 3), (8, 16, 5), (16, 16, 3), (16, 16, 3), (16, 32, 5), (32, 32, 3)]):
        s[f"{name}.conv.weight"] = (co, ci, k, k)
        for n in ("weight", "bias", "running_mean", "running_var"):
            s[f"{name}.bn.{n}"] = (co,)
    s["feature.feature.weight"], s["feature.feature.bias"] = (32, 32, 3, 3), (32,)
    for i, (ci, co) in enumerate([(32, 8), (8, 16), (16, 16), (16, 32), (32, 32), (32, 64), (64, 64)]):
        s[f"cost_regularization.conv{i}.conv.weight"] = (co, ci, 3, 3, 3)
        for n in ("weight", "bias", "running_mean", "running_var"):
            s[f"cost_regularization.conv{i}.bn.{n}"] = (co,)
    for i, (ci, co) in zip((7, 9, 11), [(64, 32), (32, 16), (16, 8)]):
        s[f"cost_regularization.conv{i}.0.weight"] = (ci, co, 3, 3, 3)          # ConvTranspose3d: [in, out, k, k, k]
        for n in ("weight", "bias", "running_mean", "running_var"):
            s[f"cost_regularization.conv{i}.1.{n}"] = (co,)
    s["cost_regularization.prob.weight"], s["cost_regularization.prob.bias"] = (1, 8, 3, 3, 3), (1,)
    return {n: s[n] for n in mvsnet_tensor_names()}


def _stack_names(pre):
    p = f"{pre}.1.conv"
    return [f"{pre}.0.weight", f"{p}.0.weight", f"{p}.0.bias", f"{p}.2.weight", f"{p}.3.weight", f"{p}.3.bias", f"{p}.5.weight", f"{pre}.2.weight"]


def cost_volume_head_names():
    """CostVolumeInitNet's tensors after mvsnet.* in state_dict() order = the order nr_cost_volume_head_pack expects (120 tensors)."""
    return (["res_net." + n for n in encoders.unet_param_names((2, 3, 6))] + _stack_names("volume_conv2d") + _stack_names("depth_conv") +
            _stack_names("out_conv"))


def _cost_volume_head_shapes(sn):
    s = {"res_net." + k: v for k, v in encoders.unet_param_shapes((32, 3, 7, 7), (2, 3, 6)).items()}
    for pre, cin in (("volume_conv2d", sn), ("depth_conv", 1), ("out_conv", 96)):
        p = f"{pre}.1.conv"
        s[f"{pre}.0.weight"], s[f"{pre}.2.weight"] = (32, cin, 3, 3), (32, 32, 1, 1)
        s[f"{p}.2.weight"] = s[f"{p}.5.weight"] = (32, 32, 3, 3)
        for n in ("0", "3"):
            s[f"{p}.{n}.weight"] = s[f"{p}.{n}.bias"] = (32,)
    return {n: s[n] for n in cost_volume_head_names()}


@functools.cache
def _packed_floats(which, sn):
    """Size of the packed MVSNet ('mvsnet': BatchNorm folded, conv weights re-laid) or cost-volume head ('head') buffer."""
    n_t, n_f = C.c_int(), C.c_longlong()
    if which == "mvsnet":
        _lib.check(_lib.lib().nr_mvsnet_layout(C.byref(n_t), C.byref(n_f)), "nr_mvsnet_layout")
    else:
        _lib.check(_lib.lib().nr_cost_volume_head_layout(sn, C.byref(n_t), C.byref(n_f)), "nr_cost_volume_head_layout")
    return n_f.value


def cost_volume_usable(module, ref_imgs_info, src_imgs_info):
    if src_imgs_info is None or not ref_imgs_info["imgs"].is_cuda or "nn_ids" not in ref_imgs_info:
        return False
    return weights.has_names(module, ["mvsnet." + n for n in mvsnet_tensor_names()] + cost_volume_head_names()) and not weights.wants_grad(module)


def mvsnet_cost_volume(module, ref_imgs_info, src_imgs_info, is_train):
    """construct_cost_volume_with_src (init_net.py:113-160) natively: (prob [rfn,ho,wo,sn] channel-last, depth [rfn,ho,wo])."""
    imgs, simgs = ref_imgs_info["imgs"], src_imgs_info["imgs"]
    rfn, _, h, w = imgs.shape
    dev = imgs.device
    sn = int(module.cfg["cost_volume_sn"])
    packed = weights.packed(module, "mvsnet", ["mvsnet." + n for n in mvsnet_tensor_names()], "nr_mvsnet_pack", _packed_floats("mvsnet", sn), dev)
    keep = [_lib.f32(t) for t in (imgs, simgs, ref_imgs_info["Ks"], ref_imgs_info["poses"], src_imgs_info["Ks"], src_imgs_info["poses"],
                                  ref_imgs_info["depth_range"])] + [ref_imgs_info["nn_ids"].detach().to(torch.int32).contiguous()]
    a = _lib.NrMvsIn()
    (a.ref_imgs, a.src_imgs, a.ref_Ks, a.ref_poses, a.src_Ks, a.src_poses, a.depth_range, a.nn_ids) = [_lib.ptr(t) for t in keep[:7]] + [keep[7].data_ptr()]
    a.rfn, a.sn, a.nn, a.h, a.w, a.dn, a.is_train = rfn, simgs.shape[0], keep[7].shape[1], h, w, sn, int(bool(is_train))
    ho, wo = C.c_int(), C.c_int()
    _lib.check(_lib.lib().nr_mvsnet_dims(h, w, a.is_train, C.byref(ho), C.byref(wo)), "nr_mvsnet_dims")
    nbytes = _lib.lib().nr_mvsnet_workspace(C.byref(a))
    if nbytes <= 0:
        raise _lib.NeurayB200Error(f"MVSNet: unsupported shape (images {h}x{w}, {sn} depth planes: h/4, w/4 and the planes must be multiples of 8)")
    ws = _lib.workspace("mvsnet", nbytes, dev, torch.uint8)
    prob = torch.empty(rfn, ho.value, wo.value, sn, dtype=torch.float32, device=dev)
    depth = torch.empty(rfn, ho.value, wo.value, dtype=torch.float32, device=dev)
    _lib.call("nr_mvsnet_fwd", _lib.ptr(packed), C.byref(a), _lib.ptr(prob), _lib.ptr(depth), ws.data_ptr(), nbytes, on=imgs,
              kernels=2 + 8 * (rfn + simgs.shape[0]) + 1 + rfn * 13)
    return prob, depth


def cost_volume_forward_into(module, ref_imgs_info, src_imgs_info, is_train, out, out_off):
    """CostVolumeInitNet.forward (init_net.py:247-254) into channels [out_off, out_off + 32) of the channel-last buffer out."""
    imgs = ref_imgs_info["imgs"]
    rfn, _, h, w = imgs.shape
    dev = imgs.device
    sn = int(module.cfg["cost_volume_sn"])
    prob, depth = mvsnet_cost_volume(module, ref_imgs_info, src_imgs_info, is_train)
    depth_norm = extract_depth_for_init({"depth": depth[:, None], "depth_range": ref_imgs_info["depth_range"]})
    packed = weights.packed(module, "head", cost_volume_head_names(), "nr_cost_volume_head_pack", _packed_floats("head", sn), dev, sn)
    nbytes = _lib.lib().nr_cost_volume_head_workspace(sn, rfn, h, w)
    ws = _lib.workspace("cv_head", nbytes, dev, torch.uint8)
    x = _lib.f32(imgs)
    _lib.call("nr_cost_volume_head_fwd", sn, _lib.ptr(packed), _lib.ptr(x), _lib.ptr(prob), _lib.ptr(depth_norm), rfn, h, w, _lib.ptr(out),
              out.shape[-1], out_off, int(encoders.PRECISION == "tf32"), ws.data_ptr(), nbytes, on=imgs,
              kernels=1 + 2 + 5 + 7 * 4 + 5 + 2 + 8 + 2 + 1 + 3 * 6)
    return out


def cost_volume_forward_nchw(module, ref_imgs_info, src_imgs_info, is_train):
    rfn, _, h, w = ref_imgs_info["imgs"].shape
    fh, fw = encoders.image_dims(h, w)
    buf = torch.empty(rfn, fh, fw, 32, dtype=torch.float32, device=ref_imgs_info["imgs"].device)
    cost_volume_forward_into(module, ref_imgs_info, src_imgs_info, is_train, buf, 0)
    return encoders.from_channel_last(buf, 0, 32)


class CostVolumeInitNet(nn.Module):
    """reference init_net.py:205-254 with the reference's tensor names (mvsnet.* frozen, BatchNorm statistics as buffers)."""
    default_cfg = {"cost_volume_sn": 64}

    def __init__(self, cfg=None):
        super().__init__()
        self.cfg = {**self.default_cfg, **(cfg or {})}
        self.register_buffer("imagenet_mean", torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1))
        self.register_buffer("imagenet_std", torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1))
        mv = {"mvsnet." + k: v for k, v in _mvsnet_shapes().items()}
        encoders._plant(self, {k: v for k, v in mv.items() if "running_" not in k})
        for k, shape in mv.items():
            if "running_" in k:
                node = self
                *path, leaf = k.split(".")
                for part in path:
                    node = getattr(node, part)
                node.register_buffer(leaf, torch.ones(shape) if leaf == "running_var" else torch.zeros(shape))
        for p in self.mvsnet.parameters():          # init_net.py:214-216: MVSNet is not trained
            p.requires_grad = False
        encoders._plant(self, _cost_volume_head_shapes(int(self.cfg["cost_volume_sn"])))

    def forward(self, ref_imgs_info, src_imgs_info, is_train=False):
        if not cost_volume_usable(self, ref_imgs_info, src_imgs_info):
            raise _lib.NeurayB200Error("CostVolumeInitNet: the native init net is forward-only and CUDA-only and needs src_imgs_info and "
                                       "ref_imgs_info['nn_ids']; run it under torch.no_grad() (training keeps the torch module)")
        return cost_volume_forward_nchw(self, ref_imgs_info, src_imgs_info, is_train)


def cost_volume_forward_or_reference(reference_forward):
    """The forward patch.install() puts over the reference's CostVolumeInitNet."""
    def forward(self, ref_imgs_info, src_imgs_info, is_train):
        if cost_volume_usable(self, ref_imgs_info, src_imgs_info):
            return cost_volume_forward_nchw(self, ref_imgs_info, src_imgs_info, is_train)
        return reference_forward(self, ref_imgs_info, src_imgs_info, is_train)
    return forward


SRC_KEY = "_nr_src_imgs_info"      # ref_imgs_info: the source views of the frame being encoded (CostVolumeInitNet), set by the frame renderer


def is_cost_volume(module):
    """True for a CostVolumeInitNet, this package's or the reference's (which carries an `mvsnet`); else a DepthInitNet."""
    return isinstance(module, CostVolumeInitNet) or hasattr(module, "mvsnet")


def init_usable(module, ref_imgs_info):
    if is_cost_volume(module):
        return cost_volume_usable(module, ref_imgs_info, ref_imgs_info.get(SRC_KEY))
    return usable(module, ref_imgs_info)


def init_forward_into(module, ref_imgs_info, out, out_off, is_train=False):
    """The owner's init net (DepthInitNet or CostVolumeInitNet) into a slot of the frame pack."""
    if is_cost_volume(module):
        return cost_volume_forward_into(module, ref_imgs_info, ref_imgs_info[SRC_KEY], is_train, out, out_off)
    return forward_into(module, ref_imgs_info, out, out_off)
