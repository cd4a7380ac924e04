"""Training extras next to the ray path (SURVEY.md section 8f row 3), native forward + backward:

    predict_mean_for_depth_loss   reference network/renderer.py:266-316 (NeuralRayGenRenderer)
    RenderLoss / DepthLoss / ConsistencyLoss, name2loss   reference network/loss.py:17-138

Same constructor cfg keys, call signature `loss(data_pr, data_gt, step)` and output dict keys as the reference, so
`train/trainer.py`'s loss loop reads them unchanged.  The arithmetic runs in libneuray_b200.so (csrc/nr_losses.cu); every
result is attached to the autograd graph through a Function whose backward is the matching native kernel.  CUDA tensors
only; there is no CPU path.
"""
import ctypes as C

import torch

from . import _lib
from .backward import unpack_point_grads


class _DepthMeanFn(torch.autograd.Function):
    """nr_depth_mean: ray_feats [rfn,32,fh,fw] + coords -> decoder means [rfn,pn,2] of the coarse (and fine) mean head."""

    @staticmethod
    def forward(ctx, meta, ray_feats, *params):
        p = _lib.NrDepthMeanParams()
        rfn, _, fh, fw = ray_feats.shape
        pn = meta["coords"].shape[1]
        dev = ray_feats.device
        feats = _lib.f32(ray_feats)
        outs = [torch.empty(rfn, pn, 2, dtype=torch.float32, device=dev) for _ in meta["w_point"]]
        p.map, p.coords = _lib.ptr(feats), _lib.ptr(meta["coords"])
        p.rfn, p.pn, p.h, p.w, p.fh, p.fw = rfn, pn, meta["h"], meta["w"], fh, fw
        for k, (wp, o) in enumerate(zip(meta["w_point"], outs)):
            p.w_point[k], p.mean[k] = _lib.ptr(wp), _lib.ptr(o)
        _lib.call("nr_depth_mean", C.byref(p), on=ray_feats)
        ctx.meta, ctx.feats = meta, feats
        ctx.need_feats = ray_feats.requires_grad
        ctx.need = [t.requires_grad for t in params]
        return tuple(outs)

    @staticmethod
    def backward(ctx, *g):
        meta, feats = ctx.meta, ctx.feats
        rfn, _, fh, fw = feats.shape
        dev = feats.device
        p = _lib.NrDepthMeanParams()
        p.map, p.coords = _lib.ptr(feats), _lib.ptr(meta["coords"])
        p.rfn, p.pn, p.h, p.w, p.fh, p.fw = rfn, meta["coords"].shape[1], meta["h"], meta["w"], fh, fw
        d_map = torch.zeros_like(feats) if ctx.need_feats else None
        keep, d_w = [], []
        for k, wp in enumerate(meta["w_point"]):
            gk = _lib.f32(g[k]) if g[k] is not None else torch.zeros(rfn, p.pn, 2, dtype=torch.float32, device=dev)
            dw = torch.zeros(wp.numel(), dtype=torch.float32, device=dev)
            keep.append(gk)
            d_w.append(dw)
            p.w_point[k], p.d_mean[k], p.d_w_point[k] = _lib.ptr(wp), _lib.ptr(gk), _lib.ptr(dw)
        p.d_map = _lib.ptr(d_map)
        _lib.call("nr_depth_mean", C.byref(p), on=feats, what="nr_depth_mean (backward)")
        grads = {}
        for k, (names, imap) in enumerate(zip(meta["names"], meta["index_maps"])):
            got = unpack_point_grads(imap, d_w[k])
            grads.update({n: got[n] for n in names})
        gp = [grads.get(n) if need else None for n, need in zip(meta["param_names"], ctx.need)]
        return (None, d_map, *gp)


def gen_depth_loss_coords(h, w, num, device):
    """reference renderer.py:272-278 (torch.randperm on the CPU generator, like the reference)."""
    coords = torch.stack(torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij"), -1).reshape(-1, 2).to(device)
    idxs = torch.randperm(coords.shape[0])[:num]
    return coords[idxs.to(device)]


def predict_mean_for_depth_loss(self, ref_imgs_info):
    """NeuralRayGenRenderer.predict_mean_for_depth_loss (renderer.py:280-316) for an owner with dist_decoder
    (/ fine_dist_decoder) under the reference's parameter names; returns the same dict."""
    from .renderer import pass_index_map, pass_params, pass_weights
    ray_feats, ref_imgs = ref_imgs_info["ray_feats"], ref_imgs_info["imgs"]
    if not ray_feats.is_cuda:
        raise _lib.NeurayB200Error("predict_mean_for_depth_loss needs CUDA tensors (no CPU fallback)")
    rfn, _, h, w = ref_imgs.shape
    coords = gen_depth_loss_coords(h, w, self.cfg["depth_loss_coords_num"], ref_imgs.device)
    coords = coords.unsqueeze(0).repeat(rfn, 1, 1)
    fine = bool(self.cfg["use_hierarchical_sampling"])
    w_point, names, index_maps, params, param_names = [], [], [], [], []
    for is_fine in (False, True) if fine else (False,):
        dn = self.cfg["fine_depth_sample_num" if is_fine else "depth_sample_num"]
        if is_fine and self.cfg["fine_depth_use_all"]:
            dn += self.cfg["depth_sample_num"]
        w_point.append(pass_weights(self, is_fine, dn, ray_feats.device)[0])
        _, _, dec_name, _, allp = pass_params(self, is_fine)
        own = {n: v for n, v in allp.items() if n.startswith(f"{dec_name}.mean_decoder.")}
        index_maps.append(pass_index_map(self, is_fine, ray_feats.device))     # covers the whole pass; only the mean head gets a gradient here
        names.append(list(own))
        params += list(own.values())
        param_names += list(own)
    meta = {"coords": coords.float().contiguous(), "h": h, "w": w, "w_point": w_point, "names": names, "index_maps": index_maps,
            "param_names": param_names}
    means = _DepthMeanFn.apply(meta, ray_feats, *params)
    outputs = {"depth_mean": means[0][..., 0], "depth_coords": coords, "depth_mean_2": means[0][..., 1]}
    if fine:
        outputs["depth_mean_fine"] = means[1][..., 0]
        outputs["depth_mean_fine_2"] = means[1][..., 1]
    return outputs


class _RenderLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pr, gt, mask):
        qn, rn, _ = pr.shape
        a, b = _lib.f32(pr), _lib.f32(gt)
        m = None if mask is None else mask.detach().contiguous().to(torch.uint8)
        loss = torch.empty(qn, dtype=torch.float32, device=pr.device)
        _lib.call("nr_render_loss", _lib.ptr(a), _lib.ptr(b), _lib.ptr(m), qn, rn, _lib.ptr(loss), None, None, on=pr)
        ctx.keep = (a, b, m)
        return loss

    @staticmethod
    def backward(ctx, g):
        a, b, m = ctx.keep
        qn, rn, _ = a.shape
        d = torch.empty_like(a)
        gg = _lib.f32(g)
        _lib.call("nr_render_loss", _lib.ptr(a), _lib.ptr(b), _lib.ptr(m), qn, rn, None, _lib.ptr(gg), _lib.ptr(d), on=a,
                  what="nr_render_loss (backward)")
        return d, (-d if ctx.needs_input_grad[1] else None), None


class _DepthLossFn(torch.autograd.Function):
    @staticmethod
    def _params(meta, depth_pr):
        p = _lib.NrDepthLossParams()
        rfn, pn = depth_pr.shape
        p.depth_pr, p.coords, p.true_depth, p.aug_depth, p.depth_range = (_lib.ptr(depth_pr), _lib.ptr(meta["coords"]), _lib.ptr(meta["true_depth"]),
                                                                          _lib.ptr(meta["aug_depth"]), _lib.ptr(meta["depth_range"]))
        p.rfn, p.pn, p.h, p.w, p.loss_type = rfn, pn, meta["h"], meta["w"], meta["loss_type"]
        p.beta, p.correct_thresh = meta["beta"], meta["thresh"]
        return p

    @staticmethod
    def forward(ctx, meta, depth_pr):
        x = _lib.f32(depth_pr)
        loss = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        p = _DepthLossFn._params(meta, x)
        p.loss = _lib.ptr(loss)
        _lib.call("nr_depth_loss", C.byref(p), on=x)
        ctx.meta, ctx.x = meta, x
        return loss

    @staticmethod
    def backward(ctx, g):
        x = ctx.x
        d = torch.empty_like(x)
        gg = _lib.f32(g)
        p = _DepthLossFn._params(ctx.meta, x)
        p.g, p.d_depth_pr = _lib.ptr(gg), _lib.ptr(d)
        _lib.call("nr_depth_loss", C.byref(p), on=x, what="nr_depth_loss (backward)")
        return None, d


class _ConsistencyFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, prob0, prob1):
        a, b = _lib.f32(prob0), _lib.f32(prob1)
        qn, rn, dn = b.shape
        loss = torch.empty(qn, dtype=torch.float32, device=b.device)
        _lib.call("nr_consistency_loss", _lib.ptr(a), _lib.ptr(b), qn, rn, dn, _lib.ptr(loss), None, None, on=b)
        ctx.keep = (a, b)
        return loss

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.keep
        qn, rn, dn = b.shape
        d = torch.empty_like(b)
        gg = _lib.f32(g)
        _lib.call("nr_consistency_loss", _lib.ptr(a), _lib.ptr(b), qn, rn, dn, None, _lib.ptr(gg), _lib.ptr(d), on=b,
                  what="nr_consistency_loss (backward)")
        return None, d


class Loss:
    def __init__(self, keys):
        self.keys = keys

    def __call__(self, data_pr, data_gt, step, **kwargs):
        pass


class ConsistencyLoss(Loss):
    """reference loss.py:17-44 (the ray mask it prepares is never applied there; neither here)."""
    default_cfg = {"use_ray_mask": False, "use_dr_loss": False, "use_dr_fine_loss": False, "use_nr_fine_loss": False}

    def __init__(self, cfg):
        self.cfg = {**self.default_cfg, **cfg}
        super().__init__(["loss_prob", "loss_prob_fine"])

    def __call__(self, data_pr, data_gt, step, **kwargs):
        if "hit_prob_self" not in data_pr:
            return {}
        outputs = {"loss_prob": _ConsistencyFn.apply(data_pr["hit_prob_nr"].detach(), data_pr["hit_prob_self"])}
        if "hit_prob_nr_fine" in data_pr:
            outputs["loss_prob_fine"] = _ConsistencyFn.apply(data_pr["hit_prob_nr_fine"].detach(), data_pr["hit_prob_self_fine"])
        return outputs


class RenderLoss(Loss):
    """reference loss.py:46-76."""
    default_cfg = {"use_ray_mask": True, "use_dr_loss": False, "use_dr_fine_loss": False, "use_nr_fine_loss": False}

    def __init__(self, cfg):
        self.cfg = {**self.default_cfg, **cfg}
        super().__init__(["loss_rgb"])

    def __call__(self, data_pr, data_gt, step, **kwargs):
        rgb_gt = data_pr["pixel_colors_gt"]
        mask = data_pr["ray_mask"] if self.cfg["use_ray_mask"] else None
        results = {"loss_rgb_nr": _RenderLossFn.apply(data_pr["pixel_colors_nr"], rgb_gt, mask)}
        if self.cfg["use_dr_loss"]:
            results["loss_rgb_dr"] = _RenderLossFn.apply(data_pr["pixel_colors_dr"], rgb_gt, mask)
        if self.cfg["use_dr_fine_loss"]:
            results["loss_rgb_dr_fine"] = _RenderLossFn.apply(data_pr["pixel_colors_dr_fine"], rgb_gt, mask)
        if self.cfg["use_nr_fine_loss"]:
            results["loss_rgb_nr_fine"] = _RenderLossFn.apply(data_pr["pixel_colors_nr_fine"], rgb_gt, mask)
        return results


class DepthLoss(Loss):
    """reference loss.py:78-132."""
    default_cfg = {"depth_correct_thresh": 0.02, "depth_loss_type": "l2", "depth_loss_l1_beta": 0.05}

    def __init__(self, cfg):
        super().__init__(["loss_depth"])
        self.cfg = {**self.default_cfg, **cfg}
        if self.cfg["depth_loss_type"] not in ("l2", "smooth_l1"):
            raise ValueError(f"depth_loss_type {self.cfg['depth_loss_type']!r}")

    def __call__(self, data_pr, data_gt, step, **kwargs):
        ref = data_gt["ref_imgs_info"]
        if "true_depth" not in ref:
            return {"loss_depth": torch.zeros([1], dtype=torch.float32, device=data_pr["pixel_colors_nr"].device)}
        depth_maps = ref["true_depth"]
        rfn, _, h, w = depth_maps.shape
        gso = data_gt["scene_name"].startswith("gso")
        meta = {"coords": _lib.f32(data_pr["depth_coords"]), "true_depth": _lib.f32(depth_maps), "aug_depth": _lib.f32(ref["depth"]) if gso else None,
                "depth_range": _lib.f32(ref["depth_range"]), "h": h, "w": w, "loss_type": 0 if self.cfg["depth_loss_type"] == "l2" else 1,
                "beta": float(self.cfg["depth_loss_l1_beta"]), "thresh": float(self.cfg["depth_correct_thresh"])}
        outputs = {"loss_depth": _DepthLossFn.apply(meta, data_pr["depth_mean"])}
        if "depth_mean_fine" in data_pr:
            outputs["loss_depth_fine"] = _DepthLossFn.apply(meta, data_pr["depth_mean_fine"])
        return outputs


name2loss = {"render": RenderLoss, "depth": DepthLoss, "consist": ConsistencyLoss}
