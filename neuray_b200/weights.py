"""Host glue around the library's packers (csrc/nr_pack.cu): which parameter tensor goes into which field of NrPassWeights.

Source: any mapping {state-dict name -> tensor} with the reference's names (SURVEY.md section 8 row a18), e.g.
`dict(renderer.named_parameters())` of a reference NeuralRayBaseRenderer, or of neuray_b200.renderer.NeuralRayRenderPath.
The packing itself (transposes, K re-ordering, hi/lo tf32 split, 128-byte swizzle) is `nr_pack_weights`; the camera terms
(K^-1, K@Rt, camera centres) are `nr_camera_blocks`.  No arithmetic happens here.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

HEADS = ("mean_decoder", "var_decoder", "aw_decoder", "vis_decoder")
_AGG_FIELDS = (("ray_dir_fc", (0, 2)), ("neuray_fc", (0, 2)), ("base_fc", (0, 2)), ("vis_fc", (0, 2)), ("vis_fc2", (0, 2)),
               ("rgb_fc", (0, 2, 4)), ("geometry_fc", (0, 2)), ("out_geometry_fc", (0, 2)))


def posenc_table(n_samples, d_hid=16):
    """Sinusoid table of reference network/ibrnet.py:305-313 (built in float64 numpy, cast to fp32) -> [n,16]."""
    pos = np.arange(n_samples, dtype=np.float64)[:, None]
    j = np.arange(d_hid)[None, :]
    table = pos / np.power(10000, 2 * (j // 2) / d_hid)
    table[:, 0::2] = np.sin(table[:, 0::2])
    table[:, 1::2] = np.cos(table[:, 1::2])
    return torch.from_numpy(table).float()


def pass_weight_struct(params, dec, agg):
    """NrPassWeights of one pass + the list of tensors whose storage it points into (keep them alive while it is used).
    params: name -> contiguous fp32 CUDA tensor; dec: 'dist_decoder' | 'fine_dist_decoder'; agg: 'agg_net' | 'fine_agg_net'."""
    w = _lib.NrPassWeights()
    keep = []

    def ptr(name):
        t = params[name].detach()
        if t.dtype != torch.float32 or not t.is_contiguous():
            t = t.float().contiguous()
        keep.append(t)
        return _lib.ptr(t)

    def lin(dst, prefix):
        dst.w, dst.b = ptr(prefix + ".weight"), ptr(prefix + ".bias")

    for h, head in enumerate(HEADS):
        if f"{dec}.{head}.0.weight" not in params:
            continue
        for l, idx in enumerate((0, 2, 4)):
            lin(w.dist_decoder[h][l], f"{dec}.{head}.{idx}")
    lin(w.prob_embed[0], f"{agg}.prob_embed.0")
    lin(w.prob_embed[1], f"{agg}.prob_embed.2")
    ib = f"{agg}.agg_impl"
    for field, idxs in _AGG_FIELDS:
        arr = getattr(w, field)
        for l, idx in enumerate(idxs):
            lin(arr[l], f"{ib}.{field}.{idx}")
    at = f"{ib}.ray_attention"
    w.w_qs, w.w_ks, w.w_vs = ptr(f"{at}.w_qs.weight"), ptr(f"{at}.w_ks.weight"), ptr(f"{at}.w_vs.weight")
    w.attn_fc = ptr(f"{at}.fc.weight")
    w.layer_norm_w, w.layer_norm_b = ptr(f"{at}.layer_norm.weight"), ptr(f"{at}.layer_norm.bias")
    return w, keep


def pack_pass(params, dec, agg, out=None):
    """(w_point, w_ray, w_tc) of one pass through nr_pack_weights (one memset + one launch per buffer set, no host sync).
    `out`: optional previously returned triple to overwrite in place."""
    any_t = params[f"{dec}.mean_decoder.0.weight"]
    dev = any_t.device
    L, T = _lib.weight_layout(), _lib.tc_layout()
    if out is None:
        out = (torch.empty(L.total_point, dtype=torch.float32, device=dev), torch.empty(L.total_ray, dtype=torch.float32, device=dev),
               torch.empty(T.total, dtype=torch.float32, device=dev))
    w, keep = pass_weight_struct(params, dec, agg)
    _lib.call("nr_pack_weights", C.byref(w), _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.ptr(out[2]), on=any_t)
    del keep
    return out


def named_tensors(module):
    """The module's parameters and buffers by state-dict name."""
    return {**dict(module.named_parameters()), **dict(module.named_buffers())}


def has_names(module, names):
    """True when the module has every one of names (the reference's state-dict names) as a parameter or a buffer."""
    return set(names) <= named_tensors(module).keys()


def wants_grad(*modules):
    """True when autograd is recording and a parameter of the modules requires a gradient (the native front end is forward-only)."""
    return torch.is_grad_enabled() and any(p.requires_grad for m in modules for p in m.parameters())


def stamp(tensors, *extra):
    """Identity of tensors at their current contents: changes when one is replaced or updated in place (optimizer steps bump
    tensor._version)."""
    return tuple((t.data_ptr(), t._version) for t in tensors) + extra


def packed(module, key, names, entry, n_floats, dev, *lead):
    """Buffer of n_floats that the library packer `entry`(*lead, tensors, n, out, stream) fills from the module's tensors
    `names` (parameters or buffers), cached on the module under `key`.  A changed stamp re-packs into a fresh buffer, so a
    consumer of the old one is unaffected."""
    have = named_tensors(module)
    lost = [n for n in names if n not in have]
    if lost:
        raise _lib.NeurayB200Error(f"{type(module).__name__}: tensors {lost[:3]}... not found (expected the reference's state-dict names)")
    tensors = [have[n] for n in names]
    st = stamp(tensors, str(dev), *lead)
    cache = module.__dict__.setdefault("_nr_packed", {})
    hit = cache.get(key)
    if hit is None or hit[0] != st:
        if tensors[0].device != torch.device(dev):
            raise _lib.NeurayB200Error(f"{type(module).__name__}: parameters live on {tensors[0].device} but the inputs are on {dev}")
        keep = [_lib.f32(t) for t in tensors]
        ptrs = (C.c_void_p * len(keep))(*[t.data_ptr() for t in keep])
        out = torch.empty(n_floats, dtype=torch.float32, device=dev)
        _lib.call(entry, *lead, ptrs, len(keep), _lib.ptr(out), on=out)
        hit = cache[key] = (st, out)
    return hit[1]


def point_index_map(params, dec, agg):
    """For the packed-layout gradient of nr_self_hit_prob: position in w_point -> 1 + flat index into the concatenated
    parameters (0 = padding), derived by packing parameters whose elements are their own index (exact in fp32 < 2^24)."""
    names = list(params)
    coded, off = {}, 1
    dev = params[names[0]].device
    for k in names:
        n = params[k].numel()
        coded[k] = torch.arange(off, off + n, dtype=torch.float32, device=dev).reshape(params[k].shape)
        off += n
    assert off < 2 ** 24
    wp, _, _ = pack_pass(coded, dec, agg)
    return wp.long(), names, [params[k].numel() for k in names], [tuple(params[k].shape) for k in names]


def camera_blocks(que_imgs_info=None, ref_imgs_info=None):
    """que_cam [24] and/or view_params [rfn,20] through nr_camera_blocks (one launch, no host sync)."""
    src = que_imgs_info if que_imgs_info is not None else ref_imgs_info
    dev = src["poses"].device
    cam = vp = None
    args = [None] * 6
    rfn = 0
    keep = []
    if que_imgs_info is not None:
        keep += [_lib.f32(que_imgs_info["poses"][0]), _lib.f32(que_imgs_info["Ks"][0])]
        rng = que_imgs_info.get("depth_range")
        keep.append(_lib.f32(rng[0]) if rng is not None else None)
        args[0:3] = [_lib.ptr(t) for t in keep[-3:]]
        cam = torch.empty(24, dtype=torch.float32, device=dev)
    if ref_imgs_info is not None:
        keep += [_lib.f32(ref_imgs_info["poses"]), _lib.f32(ref_imgs_info["Ks"])]
        rng = ref_imgs_info.get("depth_range")
        keep.append(_lib.f32(rng) if rng is not None else None)
        args[3:6] = [_lib.ptr(t) for t in keep[-3:]]
        rfn = ref_imgs_info["poses"].shape[0]
        vp = torch.empty(rfn, 20, dtype=torch.float32, device=dev)
    _lib.call("nr_camera_blocks", *args, rfn, _lib.ptr(cam), _lib.ptr(vp), on=src["poses"])
    return cam, vp
