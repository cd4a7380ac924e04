"""Host side of the per-ray rendering path: the reference's NeuralRayBaseRenderer API over the fused CUDA kernels.

Mirrors reference network/renderer.py:24-254 for the hot path (SURVEY.md section 8a rows a8-a16):

    render_by_depth   :168-203      one point-kernel + one ray-kernel launch (nr_render_pass_fwd)
    fine_render_impl  :205-215      the resampling is fused into the coarse pass' ray kernel
    render_impl       :217-226
    render            :228-254      chunk loop; per-frame NCHW -> channel-last repack hoisted out of it

Two ways to use it:
  * `NeuralRayRenderPath` -- a self-contained nn.Module holding the hot path's parameters under the reference's
    state-dict names (loads a reference checkpoint with strict=False); `render()` takes encoder outputs.
  * `neuray_b200.patch.install()` -- rebinds the same functions onto the reference's own NeuralRayBaseRenderer so
    render.py / run_training.py run unchanged.

The functions below are written against "owner": any nn.Module that has `.cfg` (reference base_cfg keys) and the
sub-modules dist_decoder / agg_net (/ fine_dist_decoder / fine_agg_net) with the reference's parameter names.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib, encoders, init_nets, modules
from .render_ops import fine_sample_u, interpolate_feats, sample_depth
from .weights import camera_blocks, pack_pass, point_index_map, posenc_table, stamp

PACK_KEY = "_nr_frame_pack"        # ref_imgs_info: the FramePack of the frame being rendered (lives for one render() call)
CAM_KEY = "_nr_que_cam"            # que_imgs_info: que_cam block of the frame being rendered (same lifetime)

base_cfg = {
    "vis_encoder_type": "default", "vis_encoder_cfg": {},
    "dist_decoder_type": "mixture_logistics", "dist_decoder_cfg": {},
    "agg_net_type": "default", "agg_net_cfg": {},
    "use_hierarchical_sampling": False, "fine_agg_net_cfg": {}, "fine_dist_decoder_cfg": {},
    "fine_depth_sample_num": 64, "fine_depth_use_all": False,
    "ray_batch_num": 2048, "depth_sample_num": 64, "alpha_value_ground_state": -15,
    "use_dr_prediction": False, "use_nr_color_for_dr": False, "use_self_hit_prob": False,
    "use_ray_mask": True, "ray_mask_view_num": 2, "ray_mask_point_num": 8,
    "render_depth": False,
    # NeuralRayGenRenderer.default_cfg (renderer.py:256-261), read by predict_mean_for_depth_loss
    "use_depth_loss": False, "depth_loss_coords_num": 8192,
}


_PACK_POOL = {}      # (device, feat shape, rgb shape) -> [(feat, rgb)] of dropped FramePacks, at most two kept


_PACK_SOURCES = ("ray_feats", "img_feats", "imgs", "poses", "Ks", "depth_range")


class FramePack:
    """Per-frame device data shared by every chunk and both passes: channel-last maps + per-view parameters.

    A pack keeps strong references to the tensors it was built from and is valid only for exactly those tensor objects
    at exactly those versions (`matches`): a fresh encoder output that happens to get a recycled address is a different
    object, and an in-place edit bumps `_version`."""

    def __del__(self):
        try:
            pool = _PACK_POOL.setdefault(self._pool_key, [])
            if len(pool) < 2:
                pool.append((self.feat, self.rgb))
        except Exception:      # interpreter shutdown
            pass

    def __init__(self, ref_imgs_info, encoder_owner=None):
        """encoder_owner: a module with image_encoder / vis_encoder (reference parameter names).  The pack then takes the INIT
        net's ray_feats from ref_imgs_info, runs both encoders natively into the channel-last buffer (encoders.encode_frame,
        reference renderer.py:229-231) and leaves their NCHW results in ref_imgs_info['img_feats'] / ['ray_feats']."""
        imgs = ref_imgs_info["imgs"]
        if not imgs.is_cuda:
            raise _lib.NeurayB200Error("the rendering path needs CUDA tensors (no CPU fallback)")
        rfn, _, h, w = imgs.shape
        rf = ref_imgs_info.get("ray_feats")
        if encoder_owner is not None:
            fh, fw = encoders.image_dims(h, w)
            if rf is None:       # the owner's init net writes its ray_feats straight into the pack (encoders.encode_frame)
                if not init_nets.is_cost_volume(encoder_owner.init_net) and init_nets.dims(h, w) != (fh, fw):
                    raise _lib.NeurayB200Error(f"init net and image encoder disagree on the map size for {h}x{w} images")
            elif tuple(rf.shape[-2:]) != (fh, fw) or rf.shape[1] != 32:
                raise _lib.NeurayB200Error(f"ray_feats {tuple(rf.shape)} do not match the image encoder's output size {(fh, fw)} for {h}x{w} images")
        else:
            imf = ref_imgs_info.get("img_feats")
            if rf is None or imf is None:
                raise _lib.NeurayB200Error("ref_imgs_info needs the encoder outputs 'ray_feats' and 'img_feats' [rfn,32,fh,fw] "
                                           "(or render through an owner with native encoders: NeuralRayFrameRenderer)")
            if rf.shape != imf.shape or rf.shape[1] != 32:
                raise _lib.NeurayB200Error(f"ray_feats {tuple(rf.shape)} and img_feats {tuple(imf.shape)} must both be [rfn,32,fh,fw]")
            fh, fw = rf.shape[-2:]
        if rfn > _lib.NR_MAX_VIEWS:
            raise _lib.NeurayB200Error(f"at most {_lib.NR_MAX_VIEWS} reference views per call, got {rfn}")
        dev = imgs.device
        self.rfn, self.h, self.w, self.fh, self.fw = rfn, h, w, fh, fw
        self._pool_key = (str(dev), (rfn, fh, fw, 64), (rfn, h, w, 4))
        spare = _PACK_POOL.get(self._pool_key)
        if spare:
            self.feat, self.rgb = spare.pop()
        else:
            self.feat = torch.empty(rfn, fh, fw, 64, dtype=torch.float32, device=dev)
            self.rgb = torch.empty(rfn, h, w, 4, dtype=torch.float32, device=dev)
        if encoder_owner is not None:      # the encoders write the feature maps; only the images are repacked below
            encoders.encode_frame(encoder_owner, ref_imgs_info, self.feat)
            rf_c = imf_c = feat = None
        else:
            rf_c, imf_c, feat = _lib.f32(rf), _lib.f32(imf), self.feat
        imgs_c = _lib.f32(imgs)
        _lib.call("nr_pack_feature_maps", _lib.ptr(rf_c), _lib.ptr(imf_c), _lib.ptr(imgs_c), rfn, h, w, fh, fw, _lib.ptr(feat), _lib.ptr(self.rgb),
                  on=imgs, kernels=1 if feat is None else 2)
        _, self.view_params = camera_blocks(None, ref_imgs_info)
        self.src = tuple((ref_imgs_info[k], ref_imgs_info[k]._version) for k in _PACK_SOURCES)

    def matches(self, ref_imgs_info):
        return all(ref_imgs_info.get(k) is t and t._version == ver for k, (t, ver) in zip(_PACK_SOURCES, self.src))


def frame_pack(ref_imgs_info):
    """The pack of the frame in flight (installed by render_chunks for the duration of one render() call), or a fresh one
    for a direct render_by_depth / render_impl call.  A fresh pack is NOT left in the caller's dict."""
    pack = ref_imgs_info.get(PACK_KEY)
    if pack is None or not pack.matches(ref_imgs_info):
        pack = FramePack(ref_imgs_info)
    return pack


def pass_params(owner, is_fine):
    """(dec, agg, dec_name, agg_name, {state-dict name: parameter}) of the coarse or the fine pass, decoder parameters first."""
    dec, agg, dec_name, agg_name = (owner.fine_dist_decoder, owner.fine_agg_net, "fine_dist_decoder", "fine_agg_net") if is_fine else \
        (owner.dist_decoder, owner.agg_net, "dist_decoder", "agg_net")
    params = {f"{dec_name}.{k}": v for k, v in dec.named_parameters()}
    params.update({f"{agg_name}.{k}": v for k, v in agg.named_parameters()})
    return dec, agg, dec_name, agg_name, params


def pass_weights(owner, is_fine, dn, device):
    """Packed weights of one pass (nr_pack_weights), cached on the owner and re-packed when any parameter changed
    (optimizer steps bump tensor._version).  Every re-pack gets fresh buffers: an autograd graph recorded before the
    parameter update keeps reading the buffers it was recorded with."""
    _, agg, dec_name, agg_name, params = pass_params(owner, is_fine)
    st = stamp(params.values(), str(device))
    cache = owner.__dict__.setdefault("_nr_wcache", {})
    hit = cache.get(is_fine)
    if hit is None or hit[0] != st:
        first = next(iter(params.values()))
        if first.device != torch.device(device):
            raise _lib.NeurayB200Error(f"parameters live on {first.device} but the rays are on {device}")
        wp, wr, wt = pack_pass(params, dec_name, agg_name)
        hit = (st, wp, wr, hit[3] if hit is not None else {}, wt)
        cache[is_fine] = hit
    pe = hit[3].get(dn)
    if pe is None:
        n_samples = agg.agg_impl.n_samples
        if n_samples != dn:
            # the reference fails with a broadcast error here (ibrnet.py:356); keep that behaviour explicit
            raise _lib.NeurayB200Error(
                f"{agg_name}: pos_encoding was built for sample_num={n_samples} but the pass has {dn} samples per ray")
        pe = posenc_table(dn).to(device).contiguous()
        hit[3][dn] = pe
    return hit[1], hit[2], pe, hit[4]


def pass_index_map(owner, is_fine, dev):
    """weights.point_index_map of a pass (packed w_point position -> parameter element), cached on the owner."""
    _, _, dec_name, agg_name, allp = pass_params(owner, is_fine)
    maps = owner.__dict__.setdefault("_nr_index_maps", {})
    key = (is_fine, str(dev), tuple(allp))
    if key not in maps:
        maps[key] = point_index_map(allp, dec_name, agg_name)
    return maps[key]


def _check_supported(owner):
    cfg = owner.cfg
    if cfg.get("use_dr_prediction", False):
        raise NotImplementedError("use_dr_prediction (direct rendering / SH fit) is outside the B200 hot path (SURVEY.md 8f)")


def _launch_pass(owner, dec, que_depth, que_imgs_info, ref_imgs_info, is_fine, fine, want_hit):
    """Enqueues the two kernels of one pass (dec: its distance decoder); returns the raw output dict (ray_mask as uint8)."""
    cfg = owner.cfg
    coords = que_imgs_info["coords"]
    dev = coords.device
    pack = frame_pack(ref_imgs_info)
    _, rn, dn = que_depth.shape
    w_point, w_ray, pos_enc, w_tc = pass_weights(owner, is_fine, dn, dev)
    cam = que_imgs_info.get(CAM_KEY)
    if cam is None:
        cam, _ = camera_blocks(que_imgs_info, None)
    coords_c = _lib.f32(coords[0])

    out = {
        "pixel_colors": torch.empty(1, rn, 3, dtype=torch.float32, device=dev),
        "hit_prob": torch.empty(1, rn, dn, dtype=torch.float32, device=dev) if (want_hit or fine) else None,
        "render_depth": torch.empty(1, rn, dtype=torch.float32, device=dev),
        "ray_mask_u8": torch.empty(1, rn, dtype=torch.uint8, device=dev),
    }
    rec = _lib.workspace("point_rec", rn * dn * _lib.NR_POINT_REC, dev, torch.float32)
    p = _lib.NrPassParams()
    p.coords, p.que_depth, p.que_cam = _lib.ptr(coords_c), _lib.ptr(que_depth), _lib.ptr(cam)
    p.rn, p.dn = rn, dn
    p.feat, p.rgb, p.view_params = _lib.ptr(pack.feat), _lib.ptr(pack.rgb), _lib.ptr(pack.view_params)
    p.rfn, p.h, p.w, p.fh, p.fw = pack.rfn, pack.h, pack.w, pack.fh, pack.fw
    p.w_point, p.w_ray, p.pos_enc = _lib.ptr(w_point), _lib.ptr(w_ray), _lib.ptr(pos_enc)
    p.w_tc = _lib.ptr(w_tc)
    # compute_prob is always the COARSE decoder's method (reference renderer.py:75): its use_vis decides
    p.use_vis = 1 if owner.dist_decoder.cfg["use_vis"] else 0
    if p.use_vis and not dec.cfg["use_vis"]:
        raise _lib.NeurayB200Error("coarse dist_decoder has use_vis but the active decoder has no vis head (the reference fails too)")
    p.var_bias = float(dec.cfg["bias_val"])
    p.ray_mask_view_num, p.ray_mask_point_num = int(cfg["ray_mask_view_num"]), int(cfg["ray_mask_point_num"])
    p.point_rec = _lib.ptr(rec)
    p.pixel_colors, p.hit_prob = _lib.ptr(out["pixel_colors"]), _lib.ptr(out["hit_prob"])
    p.render_depth, p.ray_mask = _lib.ptr(out["render_depth"]), _lib.ptr(out["ray_mask_u8"])
    if fine:
        m = fine["dn"] + (dn if fine["use_all"] else 0)
        out["fine_depth"] = torch.empty(1, rn, m, dtype=torch.float32, device=dev)
        p.fine_dn, p.fine_use_all = int(fine["dn"]), 1 if fine["use_all"] else 0
        p.fine_u, p.fine_u_stride, p.fine_depth = _lib.ptr(fine["u"]), int(fine["u_stride"]), _lib.ptr(out["fine_depth"])
    stream = _lib.stream_of(coords)
    if rn == 0:          # nothing to render: the (empty) outputs are already in place
        out["_bwd"] = None
        return out
    if _lib.PROFILE is not None:
        # bench.py: time the dominant kernel alone, with CUDA events on the launching stream
        with _lib.on_device(coords):      # Event.record() records on the current device's stream
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            _lib.call("nr_point_kernel", C.byref(p), on=coords)
            e1.record()
            _lib.call("nr_ray_kernel", C.byref(p), on=coords)
            e2.record()
        _lib.PROFILE.append((e0, e1, rn * dn, e2))
    else:
        _lib.call("nr_render_pass_fwd", C.byref(p), on=coords, kernels=2)
    # what nr_render_pass_bwd needs to run on the same inputs (kept alive by the autograd node, dropped otherwise)
    out["_bwd"] = (p, (coords_c, que_depth, cam, pack, w_point, w_ray, pos_enc, w_tc), (pack.rfn, pack.fh, pack.fw, 64), stream)
    return out


def run_pass(owner, que_depth, que_imgs_info, ref_imgs_info, is_fine, fine=None, want_hit=True):
    """One fused pass.  que_depth [1,rn,dn].  `fine`: None or dict(dn=, use_all=, u=, u_stride=) to also emit the
    next pass' depths.  Returns dict with pixel_colors [1,rn,3], hit_prob [1,rn,dn], render_depth [1,rn],
    ray_mask [1,rn] (bool) and optionally fine_depth [1,rn,M].

    When gradients are being recorded and the reference feature maps or any parameter of the pass require them, the
    outputs are attached to autograd through backward.RenderPassFn (forward values still come from the kernels)."""
    _check_supported(owner)
    coords = que_imgs_info["coords"]
    if coords.shape[0] != 1:
        raise _lib.NeurayB200Error("one query view per call (qn == 1), like every call site of the reference")
    que_depth = _lib.f32(que_depth)
    _, rn, dn = que_depth.shape
    if dn > _lib.NR_MAX_SAMPLES:
        raise _lib.NeurayB200Error(f"at most {_lib.NR_MAX_SAMPLES} samples per ray per pass, got {dn}")
    dec, _, dec_name, agg_name, params = pass_params(owner, is_fine)
    rf, imf = ref_imgs_info["ray_feats"], ref_imgs_info["img_feats"]
    needs_grad = torch.is_grad_enabled() and (rf.requires_grad or imf.requires_grad or any(v.requires_grad for v in params.values()))
    launch = lambda: _launch_pass(owner, dec, que_depth, que_imgs_info, ref_imgs_info, is_fine, fine, want_hit)
    if not needs_grad:
        out = launch()
        out.pop("_bwd", None)
    else:
        from .backward import RenderPassFn
        meta = {"names": list(params), "dec": dec_name, "agg": agg_name}
        res = RenderPassFn.apply(launch, meta, rf, imf, *params.values())
        out = {"pixel_colors": res[0], "hit_prob": res[1], "render_depth": res[2], "ray_mask_u8": res[3]}
        if fine:
            out["fine_depth"] = res[4]
    out["ray_mask"] = out.pop("ray_mask_u8").bool()
    return out


def _finish_outputs(owner, res, que_depth, que_imgs_info):
    cfg = owner.cfg
    outputs = {"pixel_colors_nr": res["pixel_colors"], "hit_prob_nr": res["hit_prob"]}
    if "imgs" in que_imgs_info:
        outputs["pixel_colors_gt"] = interpolate_feats(que_imgs_info["imgs"], que_imgs_info["coords"], align_corners=True)
    if cfg["use_ray_mask"]:
        outputs["ray_mask"] = res["ray_mask"]
    if cfg["render_depth"]:
        outputs["render_depth"] = res["render_depth"]
    return outputs


def _self_hit_prob(self, que_depth, que_imgs_info, is_fine):
    """a17 predict_self_hit_prob (reference renderer.py:137-155): the query view's own ray_feats decoded along its rays
    (fine-tuning configs).  nr_self_hit_prob, forward and backward."""
    dec, _, dec_name, _, allp = pass_params(self, is_fine)
    feats = que_imgs_info["ray_feats"]
    coords = que_imgs_info["coords"]
    h, w = que_imgs_info["imgs"].shape[-2:]
    if feats.shape[0] != 1 or coords.shape[0] != 1:
        raise _lib.NeurayB200Error("one query view per call (qn == 1), like every call site of the reference")
    from .backward import SelfHitProbFn
    dev = coords.device
    _, rn, dn = que_depth.shape
    w_point = pass_weights(self, is_fine, dn, dev)[0]
    dec_params = {n: v for n, v in allp.items() if n.startswith(dec_name + ".")}
    index_map = pass_index_map(self, is_fine, dev)
    fmap = _lib.f32(feats[0])
    cc, qd = _lib.f32(coords[0]), _lib.f32(que_depth[0])
    rng = _lib.f32(que_imgs_info["depth_range"][0])
    use_vis, var_bias = 1 if dec.cfg["use_vis"] else 0, float(dec.cfg["bias_val"])

    def params():
        p = _lib.NrSelfParams()
        p.map, p.coords, p.que_depth, p.w_point = _lib.ptr(fmap), _lib.ptr(cc), _lib.ptr(qd), _lib.ptr(w_point)
        p.rn, p.dn, p.h, p.w, p.fh, p.fw, p.use_vis = rn, dn, int(h), int(w), fmap.shape[1], fmap.shape[2], use_vis
        p.depth_range, p.var_bias = _lib.ptr(rng), var_bias
        return p

    named = list(dec_params.items())
    meta = {"params": params, "index_map": index_map, "stream": _lib.stream_of(coords), "map_shape": tuple(fmap.shape),
            "dec_names": [n for n, _ in named], "keep": (fmap, cc, qd, w_point, rng)}
    return SelfHitProbFn.apply(meta, feats, *[v for _, v in named])


def render_by_depth(self, que_depth, que_imgs_info, ref_imgs_info, is_train, is_fine):
    """reference renderer.py:168-203."""
    res = run_pass(self, que_depth, que_imgs_info, ref_imgs_info, is_fine)
    outputs = _finish_outputs(self, res, que_depth, que_imgs_info)
    if is_train and self.cfg["use_self_hit_prob"]:
        outputs["hit_prob_self"] = _self_hit_prob(self, que_depth, que_imgs_info, is_fine)
    return outputs


def _fine_request(self, rn, is_train, device):
    fdn = int(self.cfg["fine_depth_sample_num"])
    if is_train:
        u = torch.rand([1, rn, fdn]).to(device).contiguous()       # CPU generator, as reference render_ops.py:205-209
        return {"dn": fdn, "use_all": bool(self.cfg["fine_depth_use_all"]), "u": u, "u_stride": fdn}
    return {"dn": fdn, "use_all": bool(self.cfg["fine_depth_use_all"]), "u": fine_sample_u(fdn, device), "u_stride": 0}


def fine_render_impl(self, coarse_render_info, que_imgs_info, ref_imgs_info, is_train):
    """reference renderer.py:205-215 (stand-alone form: resample with the CUDA sample_fine_depth, then a fine pass)."""
    from .render_ops import sample_fine_depth
    fine_depth = sample_fine_depth(coarse_render_info["depth"], coarse_render_info["hit_prob"].detach(),
                                   que_imgs_info["depth_range"], self.cfg["fine_depth_sample_num"], is_train)
    if self.cfg["fine_depth_use_all"]:
        que_depth = torch.sort(torch.cat([coarse_render_info["depth"], fine_depth], -1), -1)[0]
    else:
        que_depth = torch.sort(fine_depth, -1)[0]
    return render_by_depth(self, que_depth, que_imgs_info, ref_imgs_info, is_train, True)


def render_impl(self, que_imgs_info, ref_imgs_info, is_train):
    """reference renderer.py:217-226: coarse pass, fused resampling, fine pass."""
    que_depth, _ = sample_depth(que_imgs_info["depth_range"], que_imgs_info["coords"], self.cfg["depth_sample_num"], False)
    hier = bool(self.cfg["use_hierarchical_sampling"])
    rn = que_imgs_info["coords"].shape[1]
    fine = _fine_request(self, rn, is_train, que_depth.device) if hier else None
    res = run_pass(self, que_depth, que_imgs_info, ref_imgs_info, False, fine=fine)
    outputs = _finish_outputs(self, res, que_depth, que_imgs_info)
    self_hit = is_train and self.cfg["use_self_hit_prob"]
    if self_hit:
        outputs["hit_prob_self"] = _self_hit_prob(self, que_depth, que_imgs_info, False)
    if hier:
        res_f = run_pass(self, res["fine_depth"], que_imgs_info, ref_imgs_info, True)
        fine_out = _finish_outputs(self, res_f, res["fine_depth"], que_imgs_info)
        if self_hit:
            fine_out["hit_prob_self"] = _self_hit_prob(self, res["fine_depth"], que_imgs_info, True)
        for k, v in fine_out.items():
            outputs[k + "_fine"] = v
    return outputs


def render_chunks(self, que_imgs_info, ref_imgs_info, is_train, pack=None):
    """The chunk loop of reference renderer.py:236-254 (everything after the encoders).  The per-frame pack (channel-last
    maps, per-view parameters) and the query camera block are built once here and live exactly as long as this call: they
    are handed to the per-chunk functions through the two info dicts and removed again before returning."""
    ray_batch_num = self.cfg["ray_batch_num"]
    coords = que_imgs_info["coords"]
    ray_num = coords.shape[1]
    render_info_all = {}
    ref_imgs_info[PACK_KEY] = pack if pack is not None else FramePack(ref_imgs_info)
    que_imgs_info[CAM_KEY] = camera_blocks(que_imgs_info, None)[0]
    try:
        # an empty ray set still runs one (empty) chunk so that the caller gets every key with a zero-length ray axis
        for ray_id in range(0, max(ray_num, 1), ray_batch_num):
            que_imgs_info["coords"] = coords[:, ray_id:ray_id + ray_batch_num]
            render_info = render_impl(self, que_imgs_info, ref_imgs_info, is_train)
            for k, v in render_info.items():
                if is_train or (not k.startswith("hit_prob")):
                    render_info_all.setdefault(k, []).append(v)
    finally:
        que_imgs_info["coords"] = coords
        ref_imgs_info.pop(PACK_KEY, None)
        que_imgs_info.pop(CAM_KEY, None)
    return {k: (v[0] if len(v) == 1 else torch.cat(v, 1)) for k, v in render_info_all.items()}


def render(self, que_imgs_info, ref_imgs_info, is_train):
    """reference renderer.py:228-254, for an owner that has the reference's encoders.  Inference runs the two encoders
    natively, straight into the channel-last frame pack (encoders.encode_frame); when a gradient is wanted through them
    (training) the owner's own torch modules run, upstream of the boundary, exactly as in the reference."""
    pack = None
    if encoders.usable(self, ref_imgs_info):
        pack = FramePack(ref_imgs_info, encoder_owner=self)
    else:
        ref_img_feats = self.image_encoder(ref_imgs_info["imgs"])
        ref_imgs_info["img_feats"] = ref_img_feats
        ref_imgs_info["ray_feats"] = self.vis_encoder(ref_imgs_info["ray_feats"], ref_img_feats)
    if is_train and self.cfg["use_self_hit_prob"]:
        que_img_feats = self.image_encoder(que_imgs_info["imgs"])
        que_imgs_info["ray_feats"] = self.vis_encoder(que_imgs_info["ray_feats"], que_img_feats)
    return render_chunks(self, que_imgs_info, ref_imgs_info, is_train, pack)


class NeuralRayRenderPath(nn.Module):
    """The hot path as a stand-alone module: parameters under the reference's state-dict names, kernels for the math.

    `render(que_imgs_info, ref_imgs_info, is_train)` expects ref_imgs_info to already hold the encoder outputs
    'ray_feats' and 'img_feats' [rfn,32,H/4,W/4] (reference renderer.py:229-231 produces them; the CNN encoders are
    out of scope, SURVEY.md section 8f)."""
    base_cfg = base_cfg

    def __init__(self, cfg):
        super().__init__()
        self.cfg = {**self.base_cfg, **cfg}
        self.dist_decoder = modules.name2dist_decoder[self.cfg["dist_decoder_type"]](self.cfg["dist_decoder_cfg"])
        self.agg_net = modules.name2agg_net[self.cfg["agg_net_type"]](self.cfg["agg_net_cfg"])
        if self.cfg["use_hierarchical_sampling"]:
            self.fine_dist_decoder = modules.name2dist_decoder[self.cfg["dist_decoder_type"]](self.cfg["fine_dist_decoder_cfg"])
            self.fine_agg_net = modules.name2agg_net[self.cfg["agg_net_type"]](self.cfg["fine_agg_net_cfg"])

    render_by_depth = render_by_depth
    fine_render_impl = fine_render_impl
    render_impl = render_impl

    def predict_mean_for_depth_loss(self, ref_imgs_info):
        """NeuralRayGenRenderer.predict_mean_for_depth_loss (reference renderer.py:280-316); cfg 'depth_loss_coords_num'."""
        from . import losses
        return losses.predict_mean_for_depth_loss(self, ref_imgs_info)

    def render(self, que_imgs_info, ref_imgs_info, is_train):
        return render_chunks(self, dict(que_imgs_info), ref_imgs_info, is_train)

    def forward(self, data):
        is_train = "eval" not in data
        return self.render(data["que_imgs_info"].copy(), data["ref_imgs_info"].copy(), is_train)


class NeuralRayFrameRenderer(NeuralRayRenderPath):
    """NeuralRayRenderPath plus the two encoders of NeuralRayBaseRenderer (renderer.py:56-59), under the reference's
    state-dict names `image_encoder.*` / `vis_encoder.*`: `render()` is the reference's `render` (renderer.py:228-254) --
    ref_imgs_info carries the INIT net's 'ray_feats' [rfn,32,H/4,W/4]; both encoders run natively into the frame pack."""

    def __init__(self, cfg):
        super().__init__(cfg)
        self.image_encoder = encoders.ImageEncoder()
        self.vis_encoder = encoders.VisEncoder(self.cfg["vis_encoder_cfg"])

    def render(self, que_imgs_info, ref_imgs_info, is_train):
        return render(self, dict(que_imgs_info), ref_imgs_info, is_train)


class NeuralRayGenFrameRenderer(NeuralRayFrameRenderer):
    """The inference frame path of NeuralRayGenRenderer (reference renderer.py:255-327; init_net_type 'depth' = the neuray_gen_depth
    model, 'cost_volume' = neuray_gen_cost_volume with its MVSNet): init net -> image_encoder + vis_encoder -> chunk loop, every stage native, the three front
    stages writing the channel-last frame pack in place.  State-dict names are the reference's (`init_net.*`,
    `image_encoder.*`, `vis_encoder.*`, `dist_decoder.*`, ...), so a gen-model checkpoint loads unchanged.
    ref_imgs_info carries imgs, depth_range, poses, Ks and depth (DepthInitNet) or nn_ids + data['src_imgs_info'] (CostVolumeInitNet);
    forward(data) like the reference."""

    def __init__(self, cfg):
        super().__init__(cfg)
        kind = self.cfg.get("init_net_type", "depth")
        if kind not in ("depth", "cost_volume"):
            raise ValueError(f"init_net_type {kind!r}")
        self.init_net = (init_nets.DepthInitNet if kind == "depth" else init_nets.CostVolumeInitNet)(self.cfg.get("init_net_cfg", {}))

    def render_call(self, que_imgs_info, ref_imgs_info, is_train, src_imgs_info=None):
        """renderer.py:268-270: the init net's ray_feats go straight into the frame pack (no 'ray_feats' entry needed)."""
        ref_imgs_info.pop("ray_feats", None)
        ref_imgs_info[init_nets.SRC_KEY] = src_imgs_info
        if not encoders.usable(self, ref_imgs_info):
            raise _lib.NeurayB200Error("NeuralRayGenFrameRenderer is the INFERENCE frame path (CUDA tensors, torch.no_grad() or frozen front-end "
                                       "parameters); training goes through patch.install() on the reference's NeuralRayGenRenderer")
        return render(self, dict(que_imgs_info), ref_imgs_info, is_train)

    def forward(self, data):
        ref_imgs_info, que_imgs_info = data["ref_imgs_info"].copy(), data["que_imgs_info"].copy()
        is_train = "eval" not in data
        out = self.render_call(que_imgs_info, ref_imgs_info, is_train, data.get("src_imgs_info"))
        if (self.cfg["use_depth_loss"] and "true_depth" in ref_imgs_info) or (not is_train):
            out.update(self.predict_mean_for_depth_loss(ref_imgs_info))
        return out
