"""CPU: the oracle (oracle/neuray_oracle.py) run and differentiated in float64, against the gradients the UNMODIFIED
reference's autograd produced in float32 (tests/golden/grads_*.npz, oracle/gen_golden_grads.py).  The GPU backward tests
(tests/test_backward_gpu.py) judge the CUDA backward against this float64 oracle, so the oracle itself is pinned here:
every dist_decoder / agg_net / fine_* parameter gradient, the gradients of ref ray_feats / img_feats, and
predict_self_hit_prob's values and gradients."""
import os

import numpy as np
import pytest
import torch

import neuray_oracle as orc
from golden_io import GOLDEN_DIR, GoldenCase


def f64(d):
    return {k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in d.items()}


def load(name):
    z = np.load(os.path.join(GOLDEN_DIR, f"grads_{name}.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def within(got, gold, what):
    """The bound of the host-build tests (tests/test_backward_cpu.py)."""
    err, scale = float((got - gold.double()).abs().max()), float(gold.abs().max())
    assert err <= 3e-4 * max(scale, 1e-3) + 3e-6, (what, err, scale)
    return err / max(scale, 1e-3)


@pytest.mark.parametrize("name", ["train8", "views10"])
def test_fp64_oracle_matches_the_reference_gradients(name):
    g, z = GoldenCase(name), load(name)
    sel = g.stage_sel
    W = {k: v.double().requires_grad_(True) for k, v in g.W.items()}
    ref = f64(g.ref)
    ref["ray_feats"].requires_grad_(True)
    ref["img_feats"].requires_grad_(True)
    que = f64(g.stage_que())
    dc, df = g.que_depth[:, sel].double().contiguous(), g.que_depth_fine[:, sel].double().contiguous()
    cfg = g.flat_cfg()
    oc = orc.render_by_depth(W, cfg, dc, que, ref, True, False)
    of = orc.render_by_depth(W, cfg, df, que, ref, True, True)
    assert oc["pixel_colors_nr"].dtype == torch.float64 and of["render_depth"].dtype == torch.float64
    lw = {k[3:]: v.double() for k, v in z.items() if k.startswith("lw_")}
    loss = (oc["pixel_colors_nr"] * lw["gw_c"]).sum() + (oc["hit_prob_nr"] * lw["gh_c"]).sum() \
        + (of["pixel_colors_nr"] * lw["gw_f"]).sum() + (of["render_depth"] * lw["gd_f"]).sum()
    loss.backward()
    within(oc["pixel_colors_nr"].detach(), z["out_c_pixel_colors_nr"], "coarse colours")
    within(of["pixel_colors_nr"].detach(), z["out_f_pixel_colors_nr"], "fine colours")
    gold = {k[5:]: v for k, v in z.items() if k.startswith("grad_")}
    worst = 0.0
    for k, ga in gold.items():
        got = ref[k[4:]].grad if k.startswith("ref_") else W[k].grad
        assert got is not None, k
        worst = max(worst, within(got, ga, k))
    # the reference had no gradient for exactly the parameters the golden lacks
    for k, p in W.items():
        if k not in gold and p.grad is not None:
            assert float(p.grad.abs().max()) < 1e-12, k
    assert len(gold) > 100
    print(f"{name}: worst relative error of the fp64 oracle against the reference's gradients {worst:.2e}")


@pytest.mark.parametrize("name", ["train8", "views10"])
def test_fp64_oracle_matches_the_reference_self_hit_prob(name):
    g, z = GoldenCase(name), load(name)
    sel = g.stage_sel
    W = {k: v.double().requires_grad_(True) for k, v in g.W.items()}
    que = f64(g.stage_que())
    qmap = z["self_map"].double().requires_grad_(True)
    que["ray_feats"] = qmap
    depth = g.que_depth[:, sel].double().contiguous()
    hit = orc.predict_self_hit_prob(W, g.flat_cfg(), que, depth, orc.depth2inv_dists(depth, que["depth_range"]), False)
    assert hit.dtype == torch.float64
    (hit * z["self_gs"].double()).sum().backward()
    assert float((hit.detach() - z["self_hit"].double()).abs().max()) <= 2e-6
    checked = 0
    for k, ga in z.items():
        if k.startswith("selfgrad_"):
            within(W[k[9:]].grad, ga, k)
            checked += 1
    assert checked >= 18
    within(qmap.grad, z["self_grad_map"], "self_grad_map")
