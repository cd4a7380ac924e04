"""GPU: the drop-in proof.  The UNMODIFIED reference's own NeuralRayGenRenderer, render_ops and losses were run on seeded inputs
(oracle/gen_golden_dropin.py -> tests/golden/dropin_*.npz); the native path runs on the same inputs and parameters, and
everything the reference's callers read is compared with what the reference computed: every output key of forward() in eval
mode (gen_depth and gen_cost_volume models, init net and encoders included), and in training mode every output key, the
gradient of every hot-path parameter and the gradients the path hands to the encoders in front of it, after backward() of the
reference's kind of loss (render + depth terms, self-hit-prob term).

The encoders and the init net have no native backward: in training patch.install() keeps the reference's own PyTorch modules
in front of the path.  So the training comparison feeds the path the reference's encoder outputs and checks what flows back
into them; the encoders' backward, the reference's code, is linear in that gradient.

This is the test of SURVEY.md section 8b: `render.py` / `run_training.py` construct the network by name, call
`network(data)` and `loss.backward()`; nothing else touches the renderer.
"""
import json
import os

import numpy as np
import pytest
import torch

import gen_golden_dropin as gd
from neuray_b200 import renderer, synthetic

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CFG = gd.CFG


def golden(name, prefix=""):
    z = np.load(os.path.join(GOLDEN, name))
    return {k[len(prefix):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix) and z[k].dtype.kind != "U"}


def gen_net(cfg, tag):
    """The native NeuralRayGenFrameRenderer with the parameters the reference ran with (same state-dict names and shapes)."""
    shapes = json.loads(str(np.load(os.path.join(GOLDEN, "dropin_eval.npz"))[f"{tag}_shapes"]))
    net = renderer.NeuralRayGenFrameRenderer(cfg)
    assert gd.front_shapes(net) == shapes
    missing, unexpected = net.load_state_dict(gd.weights(cfg, shapes), strict=False)
    assert not unexpected and all("imagenet_" in k for k in missing), (missing, unexpected)
    return net.cuda().eval()


def run(net, que, ref, is_train, src=None):
    data = {"que_imgs_info": synthetic.to_device(que, "cuda"), "ref_imgs_info": synthetic.to_device(ref, "cuda")}
    if src is not None:
        data["src_imgs_info"] = synthetic.to_device(src, "cuda")
    if not is_train:
        data["eval"] = True
    torch.manual_seed(gd.FORWARD_SEED)            # randperm of the depth-loss coordinates, torch.rand of the fine quantiles
    return net(data)


def compare_outputs(a, b, fine_bad_frac):
    assert set(a) == set(b), set(a) ^ set(b)
    for k in a:
        x, y = a[k].detach().float().cpu(), b[k].detach().float().cpu()
        assert x.shape == y.shape, k
        if a[k].dtype == torch.bool:
            assert (x != y).float().mean().item() <= (fine_bad_frac if k.endswith("_fine") else 0.0), k
            continue
        bad = ((x - y).abs() > 1e-4 + 1e-3 * y.abs()).float().mean().item()
        # fine-pass quantities sit behind searchsorted (SURVEY.md section 7): isolated samples may move by a bin
        allowed = fine_bad_frac if ("fine" in k) else 0.0
        assert bad <= allowed, (k, bad, float((x - y).abs().max()))


def test_eval_forward_patched_equals_unpatched():
    que, ref = gd.make_data()
    net = gen_net(CFG, "depth")
    with torch.no_grad():
        got = run(net, que, ref, False)
    torch.cuda.synchronize()
    assert "hit_prob_nr" not in got and "depth_mean_fine" in got
    compare_outputs(got, golden("dropin_eval.npz", "depth_out_"), fine_bad_frac=0.01)


@pytest.mark.parametrize("self_hit", [False, True])
def test_training_forward_and_every_gradient(self_hit):
    """forward() in training mode + backward() of the reference's kind of loss, native path against the reference:
      * every output key;
      * every parameter of the hot-path modules (dist_decoder, agg_net and their fine twins);
      * the gradients the path hands to the encoders in front of it (d img_feats, d ray_feats of the reference views and, with
        the self-hit term, d ray_feats of the query)."""
    cfg = dict(CFG, use_self_hit_prob=self_hit)
    name = f"dropin_train_self_hit_{int(self_hit)}"
    que, ref = gd.make_data(self_feats=self_hit)
    net = renderer.NeuralRayRenderPath(cfg)
    net.load_state_dict(gd.weights(cfg, {}), strict=True)
    net.cuda().train()
    feats = {k: v.cuda().requires_grad_(True) for k, v in golden(name + "_inputs.npz").items()}
    dq, dr = synthetic.to_device(que, "cuda"), synthetic.to_device(ref, "cuda")
    dr["img_feats"], dr["ray_feats"] = feats["ref_img_feats"], feats["ref_ray_feats"]
    if self_hit:
        dq["ray_feats"] = feats["que_ray_feats"]
    torch.manual_seed(gd.FORWARD_SEED)
    out = net.render(dq, dr, True)
    out.update(net.predict_mean_for_depth_loss(dr))      # NeuralRayGenRenderer.forward with use_depth_loss and a true depth
    gd.loss_of(out).backward()
    torch.cuda.synchronize()
    compare_outputs(out, golden(name + ".npz", "out_"), fine_bad_frac=0.01)
    # what the path hands upstream
    for k, g_ref in golden(name + ".npz", "feat_grad_").items():
        g = feats[k].grad.cpu()
        rel = float((g - g_ref).abs().max()) / float(g_ref.abs().max())
        print(f"d loss / d {k}: relative difference {rel:.2e}")
        assert rel <= 2e-3, (k, rel)
    grads = golden(name + ".npz", "grad_")
    params = dict(net.named_parameters())
    assert set(grads) <= set(params), set(grads) - set(params)
    for k, p in params.items():           # no gradient in the reference (the fine vis decoder without the self-hit term)
        if k not in grads:
            assert p.grad is None or float(p.grad.abs().max()) < 1e-7, k
    module_scale = {}
    for k, g_ref in grads.items():
        m = k.split(".")[0]
        module_scale[m] = max(module_scale.get(m, 0.0), float(g_ref.abs().max()))
    checked, worst = 0, (0.0, "")
    for k, g_ref in grads.items():
        assert params[k].grad is not None, f"{k}: the native path sends no gradient here"
        g = params[k].grad.cpu()
        scale = float(g_ref.abs().max())
        if scale == 0.0:
            assert float(g.abs().max()) < 1e-7, k
            continue
        # parameters whose true gradient is zero (the bias in front of a softmax) hold rounding noise only, in the reference
        # too: measured against the module's largest gradient entry
        noise = 1e-4 * module_scale[k.split(".")[0]]
        err = float((g - g_ref).abs().max())
        # 5e-3: the fine pass runs on resampled depths that differ in the last bits between the two implementations
        assert err <= 5e-3 * scale + noise, (k, err, scale, noise)
        if scale > noise:
            worst = max(worst, (err / scale, k))
        checked += 1
    print(f"worst relative gradient difference {worst[0]:.2e} ({worst[1]}), {checked} parameters")
    assert checked > 100, checked


def test_render_ops_refuse_to_cut_a_graph():
    """A drop-in without a backward raises when handed an input that requires grad (instead of silently detaching)."""
    from neuray_b200 import _lib, render_ops
    d = torch.rand(1, 8, 16, device="cuda", requires_grad=True)
    with pytest.raises(_lib.NeurayB200Error):
        render_ops.depth2dists(d)
    with torch.no_grad():
        render_ops.depth2dists(d)
    fm, pts, mask = (t.cuda() for t in gd.interpolation_inputs())
    fm.requires_grad_(True)
    out = render_ops.interpolate_feature_map(fm, pts, mask, 48, 64)
    out.square().sum().backward()
    want = golden("dropin_eval.npz")                     # the reference's own torch implementation
    assert torch.allclose(out.cpu(), want["interp_out"], atol=1e-5)
    assert torch.allclose(fm.grad.cpu(), want["interp_grad"], atol=1e-4, rtol=1e-4)


def test_losses_patched_equal_unpatched():
    """network.loss.name2loss (what train/trainer.py builds its losses from) against the native losses that patch.install()
    puts in its place: the three losses on the outputs of one training-mode forward of the reference network, values and the
    gradients with respect to every output tensor they read."""
    from neuray_b200 import losses
    _, ref = gd.make_data(self_feats=True)
    out = {k: v.cuda() for k, v in golden("dropin_eval.npz", "loss_in_").items()}
    got, ggot = gd.evaluate_losses(losses.name2loss, out, synthetic.to_device(ref, "cuda"))
    want, gwant = golden("dropin_eval.npz", "loss_val_"), golden("dropin_eval.npz", "loss_grad_")
    assert set(got) == set(want) == {"loss_rgb_nr", "loss_rgb_nr_fine", "loss_depth", "loss_depth_fine", "loss_prob", "loss_prob_fine"}
    for k in want:
        assert torch.allclose(got[k].cpu(), want[k], rtol=2e-5, atol=1e-6), (k, got[k], want[k])
    for k in gd.LOSS_READS:
        assert gwant[k] is not None and ggot[k] is not None, k
        err, scale = float((ggot[k].cpu() - gwant[k]).abs().max()), float(gwant[k].abs().max())
        assert err <= 1e-4 * scale + 1e-9, (k, err, scale)


def test_cost_volume_model_eval_forward_patched_equals_unpatched():
    """The neuray_gen_cost_volume model (init_net_type 'cost_volume': CostVolumeInitNet with its MVSNet, seeded here) in eval
    mode: the native run goes through nr_mvsnet_fwd + nr_cost_volume_head_fwd, the native encoders and the render kernels."""
    cfg = dict(CFG, init_net_type="cost_volume")
    que, ref, src = gd.cost_volume_data()
    net = gen_net(cfg, "cv")
    with torch.no_grad():
        got = run(net, que, ref, False, src)
    torch.cuda.synchronize()
    compare_outputs(got, golden("dropin_eval.npz", "cv_out_"), fine_bad_frac=0.01)
