"""TEST INFRASTRUCTURE ONLY -- tests/golden/dropin_*.npz: what the UNMODIFIED reference's own NeuralRayGenRenderer, render_ops and
losses compute on small seeded inputs, run on the CPU through oracle/ref_import.py.  tests/test_reference_gpu.py and
tests/test_render_ops_gpu.py run the native path on the same inputs and parameters and compare with these files.

    python oracle/gen_golden_dropin.py

Inputs are rebuilt from seeds (make_data / cost_volume_data below, shared with the tests); parameters come from seeds too:
the hot-path modules from synthetic.make_weights, everything in front of them (image / vis encoder, init net, MVSNet) from
neuray_oracle.encoder_test_weights / mvs_test_weights over the state-dict shapes the goldens store.  Both pass through the CPU
generator, as do the random draws of a forward (training-mode fine quantiles, depth-loss coordinates), so a seed set before
a forward makes the same draws on the CPU and on the GPU.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import neuray_oracle as orc  # noqa: E402
from neuray_b200 import synthetic  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
HOT = ("dist_decoder.", "agg_net.", "fine_dist_decoder.", "fine_agg_net.")
DN = 24
CFG = {"init_net_type": "depth", "use_hierarchical_sampling": True, "use_depth_loss": True, "dist_decoder_cfg": {"use_vis": False},
       "depth_sample_num": DN, "fine_depth_sample_num": DN, "agg_net_cfg": {"sample_num": DN}, "fine_agg_net_cfg": {"sample_num": DN},
       "ray_batch_num": 192, "render_depth": True, "depth_loss_coords_num": 256}
FORWARD_SEED = 77          # set before every forward: randperm of the depth-loss coordinates, torch.rand of the fine quantiles


def _smooth(rs, shape, lo, hi, cells=8):
    """Low-frequency random field (bilinear upsampling of a coarse grid): images and depth maps of real scenes are smooth at
    the pixel scale; white noise would make every bilinear lookup hypersensitive to the last bit of its coordinates."""
    n, c, h, w = shape
    coarse = torch.from_numpy(rs.uniform(lo, hi, (n, c, max(2, h // cells), max(2, w // cells))).astype(np.float32))
    return torch.nn.functional.interpolate(coarse, size=(h, w), mode="bilinear", align_corners=True)


def make_data(rfn=6, rays=384, self_feats=False, seed=3):
    que, ref = synthetic.make_scene(64, 80, rfn, seed=seed, smooth=2)
    ref = dict(ref)
    ref.pop("ray_feats"), ref.pop("img_feats")
    rs = np.random.RandomState(seed)
    ref["imgs"] = _smooth(rs, tuple(ref["imgs"].shape), 0.0, 1.0)
    que = dict(que, imgs=_smooth(rs, tuple(que["imgs"].shape), 0.0, 1.0))
    ref["depth"] = _smooth(rs, (rfn, 1, 64, 80), 2.5, 5.0)
    ref["true_depth"] = ref["depth"]
    n = que["coords"].shape[1]
    idx = torch.from_numpy(rs.permutation(n)[:rays])
    que = dict(que, coords=que["coords"][:, idx].contiguous())
    if self_feats:
        que["ray_feats"] = torch.from_numpy(rs.standard_normal((1, 32, 16, 20)).astype(np.float32))
    return que, ref


def cost_volume_data():
    """The neuray_gen_cost_volume model's inputs: 4 reference views, 3 source views, 2 neighbours each, 384 query rays."""
    que, ref = synthetic.make_scene(64, 96, 4, seed=5, smooth=2)
    _, src = synthetic.make_scene(64, 96, 3, seed=6, smooth=2)
    ref = dict(ref)
    ref.pop("ray_feats"), ref.pop("img_feats")
    rs = np.random.RandomState(5)
    ref["imgs"] = _smooth(rs, tuple(ref["imgs"].shape), 0.0, 1.0)
    src = {"imgs": _smooth(rs, tuple(src["imgs"].shape), 0.0, 1.0), "poses": src["poses"], "Ks": src["Ks"]}
    ref["nn_ids"] = torch.from_numpy(np.stack([rs.permutation(3)[:2] for _ in range(4)]).astype(np.int64))
    que = dict(que, imgs=_smooth(rs, tuple(que["imgs"].shape), 0.0, 1.0),
               coords=que["coords"][:, torch.from_numpy(rs.permutation(que["coords"].shape[1])[:384])].contiguous())
    return que, ref, src


def weights(cfg, shapes, seed=0):
    """Parameters of the whole gen network: hot path from synthetic.make_weights (a density head that terminates rays
    gradually), the front end (`shapes`: {name: shape} of everything else) seeded; MVSNet with mvs_test_weights, whose
    softened depth-softmax logits keep the cost volume from being an argmax."""
    W = synthetic.make_weights(cfg, seed=seed, sigma_gain=1.0, sigma_bias=0.02)
    mvs = {k[len("init_net.mvsnet."):]: v for k, v in shapes.items() if k.startswith("init_net.mvsnet.")}
    W.update({"init_net.mvsnet." + k: v for k, v in orc.mvs_test_weights(mvs, 41).items()})
    W.update(orc.encoder_test_weights({k: v for k, v in shapes.items() if not k.startswith("init_net.mvsnet.")}, 42))
    return W


def front_shapes(net):
    """{name: shape} of the parameters and buffers in front of the hot path.  The constant imagenet normalisation is left out,
    and so is the reference's sph_fitter: only its use_dr_prediction branch reads it, which these models leave off."""
    return {k: list(v.shape) for k, v in net.state_dict().items()
            if not k.startswith(HOT + ("sph_fitter.",)) and "imagenet_" not in k}


def loss_of(out):
    """The shape of the reference's training loss (network/loss.py:46-132): render terms on both passes + a depth term on
    the decoder means + the self-hit-prob consistency term when present."""
    loss = ((out["pixel_colors_nr"] - out["pixel_colors_gt"]) ** 2).mean() + ((out["pixel_colors_nr_fine"] - out["pixel_colors_gt_fine"]) ** 2).mean()
    loss = loss + 0.1 * out["depth_mean"].abs().mean() + 0.1 * out["depth_mean_fine"].abs().mean()
    if "hit_prob_self" in out:
        loss = loss + ((out["hit_prob_self"] - out["hit_prob_nr"].detach()) ** 2).mean() + ((out["hit_prob_self_fine"] - out["hit_prob_nr_fine"].detach()) ** 2).mean()
    return loss


LOSS_READS = ("pixel_colors_nr", "pixel_colors_nr_fine", "depth_mean", "depth_mean_fine", "hit_prob_self", "hit_prob_self_fine")
LOSS_CFGS = {"render": {"use_nr_fine_loss": True}, "depth": {"depth_loss_type": "smooth_l1"}, "consist": {}}


def evaluate_losses(name2loss, out, ref_imgs_info):
    """The three losses train/trainer.py builds by name, on one forward's outputs: values, and the gradients of a weighted sum
    with respect to every output tensor they read."""
    data_pr = {k: (v.detach().clone().requires_grad_(True) if k in LOSS_READS else v) for k, v in out.items()}
    data_gt = {"ref_imgs_info": ref_imgs_info, "scene_name": "dtu_train/scan1"}
    res = {}
    for name, c in LOSS_CFGS.items():
        res.update(name2loss[name](c)(data_pr, data_gt, 0))
    total = sum((i + 1.0) * v.sum() for i, v in enumerate(res.values()))
    total.backward()
    return {k: v.detach() for k, v in res.items()}, {k: data_pr[k].grad for k in LOSS_READS}


def interpolation_inputs():
    g = torch.Generator().manual_seed(21)
    fm = torch.randn(2, 32, 12, 16, generator=g)
    pts = torch.rand(2, 50, 2, generator=g) * torch.tensor([60.0, 44.0])
    mask = (torch.rand(2, 50, generator=g) > 0.2).float()
    return fm, pts, mask


def resampling_inputs():
    """tests/test_render_ops_gpu.py::test_compositing_and_resampling's coarse depths and hit probabilities."""
    que, _ = synthetic.make_scene(40, 52, 5, que_h=20, que_w=24, seed=4, smooth=2)
    torch.manual_seed(0)
    torch.rand(3, 50, 24)
    depth, _ = orc.sample_depth(que["depth_range"], que["coords"][:, :200], 24, False)
    hit = orc.alpha_values2hit_prob(torch.rand(1, 200, 24) * 0.4)
    return depth, hit, que["depth_range"]


def _npz(path, **arrays):
    np.savez_compressed(path, **arrays)
    print(path, "%.1f KB" % (os.path.getsize(path) / 1024))


def _outs(prefix, out):
    return {f"{prefix}{k}": v.detach().numpy() for k, v in out.items()}


def _build(mod, cfg):
    torch.manual_seed(0)
    import ref_import
    cwd = os.getcwd()
    os.chdir(ref_import.REFERENCE_ROOT)          # CostVolumeInitNet opens network/mvsnet/mvsnet_pl.ckpt relative to the reference root
    try:
        net = mod.NeuralRayGenRenderer(cfg)
    finally:
        os.chdir(cwd)
    shapes = front_shapes(net)
    missing, unexpected = net.load_state_dict(weights(cfg, shapes), strict=False)
    assert not unexpected and all("imagenet_" in k or k.startswith("sph_fitter.") for k in missing), (missing, unexpected)
    return net, shapes


def _forward(net, que, ref, is_train, src=None):
    data = {"que_imgs_info": dict(que), "ref_imgs_info": dict(ref)}
    if src is not None:
        data["src_imgs_info"] = dict(src)
    if not is_train:
        data["eval"] = True
    torch.manual_seed(FORWARD_SEED)
    return net(data)


def eval_golden(mod):
    """dropin_eval.npz: the gen_depth and gen_cost_volume models in eval mode, the reference's interpolate_feature_map with its
    gradient, sample_fine_depth in both resampling modes, and the three training losses."""
    g = {}
    net, shapes = _build(mod, CFG)
    que, ref = make_data()
    with torch.no_grad():
        g.update(_outs("depth_out_", _forward(net.eval(), que, ref, False)))
    g["depth_shapes"] = json.dumps(shapes)

    cfg = dict(CFG, init_net_type="cost_volume")
    net, shapes = _build(mod, cfg)
    que, ref, src = cost_volume_data()
    with torch.no_grad():
        g.update(_outs("cv_out_", _forward(net.eval(), que, ref, False, src)))
    g["cv_shapes"] = json.dumps(shapes)

    import network.render_ops as ref_ops
    fm, pts, mask = interpolation_inputs()
    fm.requires_grad_(True)
    out = ref_ops.interpolate_feature_map(fm, pts, mask, 48, 64)
    out.square().sum().backward()
    g["interp_out"], g["interp_grad"] = out.detach().numpy(), fm.grad.numpy()

    depth, hit, rng = resampling_inputs()
    g["fine_depth_inv"] = ref_ops.sample_fine_depth(depth, hit, rng, 16, False).numpy()
    g["fine_depth_lin"] = ref_ops.sample_fine_depth(depth, hit, rng, 16, False, inv_mode=False).numpy()

    import network.loss as ref_loss
    cfg = dict(CFG, use_self_hit_prob=True)
    net, _ = _build(mod, cfg)
    que, ref = make_data(self_feats=True)
    with torch.no_grad():
        out = _forward(net.train(), que, ref, True)
    res, grads = evaluate_losses(ref_loss.name2loss, out, ref)
    g.update(_outs("loss_in_", out))
    g.update({f"loss_val_{k}": v.numpy() for k, v in res.items()})
    g.update({f"loss_grad_{k}": v.numpy() for k, v in grads.items()})
    _npz(os.path.join(GOLDEN, "dropin_eval.npz"), **g)


def train_golden(mod, self_hit):
    """dropin_train_self_hit_<0|1>[_inputs].npz: one training-mode forward + backward of loss_of.  _inputs: what the path
    receives from the encoders in front of it; the other file: every output, the gradient of every hot-path parameter, and
    d loss / d each of those inputs (what the path hands back to the encoders)."""
    cfg = dict(CFG, use_self_hit_prob=self_hit)
    net, _ = _build(mod, cfg)
    net.train()
    que, ref = make_data(self_feats=self_hit)
    feats = []

    def hook(name):
        def fn(module, inputs, output):
            output.retain_grad()
            feats.append((name, output))
        return fn
    handles = [getattr(net, n).register_forward_hook(hook(n)) for n in ("image_encoder", "vis_encoder")]
    # the vis encoder reads the image features too: detached there, d loss / d img_feats is what the path alone hands back
    handles.append(net.vis_encoder.register_forward_pre_hook(lambda module, args: (args[0], args[1].detach())))
    out = _forward(net, que, ref, True)
    loss_of(out).backward()
    for h in handles:
        h.remove()
    # the path reads the reference views' img_feats and ray_feats and, with the self-hit term, the query's ray_feats (call 3);
    # the query's image features (call 2) only feed the vis encoder in front of the path
    assert [n for n, _ in feats] == ["image_encoder", "vis_encoder"] * (2 if self_hit else 1)
    path_inputs = {"ref_img_feats": feats[0][1], "ref_ray_feats": feats[1][1]}
    if self_hit:
        path_inputs["que_ray_feats"] = feats[3][1]
    name = f"dropin_train_self_hit_{int(self_hit)}"
    _npz(os.path.join(GOLDEN, name + "_inputs.npz"), **{k: f.detach().numpy() for k, f in path_inputs.items()})
    g = _outs("out_", out)
    g.update({f"feat_grad_{k}": f.grad.numpy() for k, f in path_inputs.items()})
    g.update({f"grad_{k}": p.grad.numpy() for k, p in net.named_parameters() if k.startswith(HOT) and p.grad is not None})
    _npz(os.path.join(GOLDEN, name + ".npz"), **g)


def main():
    import ref_import
    mod = ref_import.load_reference()
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    eval_golden(mod)
    for self_hit in (False, True):
        train_golden(mod, self_hit)


if __name__ == "__main__":
    main()
