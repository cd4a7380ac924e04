"""GPU: every stand-alone render_ops drop-in against the oracle's restatement of the same reference function."""
import os

import numpy as np
import pytest
import torch

import neuray_oracle as orc
from neuray_b200 import render_ops, synthetic

pytestmark = pytest.mark.gpu


def close(a, b, atol=1e-5, rtol=1e-5, what=""):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    err = (a - b).abs()
    assert bool((err <= atol + rtol * b.abs()).all()), f"{what}: max abs err {err.max().item():.3e}"


@pytest.fixture(scope="module")
def scene():
    que, ref = synthetic.make_scene(40, 52, 5, que_h=20, que_w=24, seed=4, smooth=2)
    return que, ref, synthetic.to_device(que, "cuda"), synthetic.to_device(ref, "cuda")


def test_sampling_and_ray_geometry(scene):
    que, ref, dq, dr = scene
    d_o, dist_o = orc.sample_depth(que["depth_range"], que["coords"], 24, False)
    d_g, dist_g = render_ops.sample_depth(dq["depth_range"], dq["coords"], 24, False)
    assert torch.equal(d_g.cpu(), d_o)
    close(dist_g, dist_o, what="que_dists")
    c_o, v_o = orc.coords2rays(que["coords"], que["poses"], que["Ks"])
    c_g, v_g = render_ops.coords2rays(dq["coords"], dq["poses"], dq["Ks"])
    close(c_g, c_o, what="centers"); close(v_g, v_o, atol=2e-6, what="directions")
    p_o, dir_o = orc.depth2points(que, d_o)
    p_g, dir_g = render_ops.depth2points(dq, d_g)
    close(p_g, p_o, what="que_pts"); close(dir_g, dir_o, what="que_dir")
    close(render_ops.depth2dists(d_g), orc.depth2dists(d_o), what="depth2dists")
    close(render_ops.depth2inv_dists(d_g, dq["depth_range"]), orc.depth2inv_dists(d_o, que["depth_range"]), atol=2e-6, what="inv dists")


def test_projection_and_gather(scene):
    que, ref, dq, dr = scene
    d_o, _ = orc.sample_depth(que["depth_range"], que["coords"], 8, False)
    pts_o, _ = orc.depth2points(que, d_o)
    pts = pts_o.reshape(-1, 3)
    dir_o, pix_o, z_o, m_o = orc.project_points_ref_views(ref, pts)
    dir_g, pix_g, z_g, m_g = render_ops.project_points_ref_views(dr, pts.cuda())
    close(dir_g, dir_o, what="prj_dir"); close(pix_g, pix_o, atol=2e-4, what="prj_pts"); close(z_g, z_o, what="prj_depth")
    assert torch.equal(m_g.cpu(), m_o)
    pc_g, v_g, _ = render_ops.project_points_coords(pts.cuda(), dr["poses"], dr["Ks"])
    pc_o, v_o, _ = orc.project_points_coords(pts, ref["poses"], ref["Ks"])
    close(pc_g, pc_o, atol=2e-4, what="project_points_coords"); assert torch.equal(v_g.cpu(), v_o)
    close(render_ops.project_points_directions(dr["poses"], pts.cuda()), orc.project_points_directions(ref["poses"], pts), what="directions")
    h, w = ref["imgs"].shape[-2:]
    for key in ("ray_feats", "imgs"):
        g = render_ops.interpolate_feature_map(dr[key], pix_o.cuda(), m_o.cuda(), h, w)
        o = orc.interpolate_feature_map(ref[key], pix_o, m_o, h, w)
        close(g, o, atol=2e-5, what="interpolate_feature_map " + key)
    gt_g = render_ops.interpolate_feats(dq["imgs"], dq["coords"], align_corners=True)
    gt_o = orc.bilinear_sample(que["imgs"], que["coords"], align_corners=True)
    close(gt_g, gt_o, what="interpolate_feats zeros/align")
    d = render_ops.project_points_dict(dr, pts_o.cuda())
    o = orc.project_points_dict(ref, pts_o)
    for k in o:
        close(d[k], o[k], atol=2e-4 if k == "pts" else 2e-5, what="project_points_dict/" + k)


def test_compositing_and_resampling(scene):
    torch.manual_seed(0)
    alpha = torch.rand(3, 50, 24) * 0.3
    close(render_ops.alpha_values2hit_prob(alpha.cuda()), orc.alpha_values2hit_prob(alpha), atol=1e-6, what="alpha2hit")
    que = scene[0]
    depth, _ = orc.sample_depth(que["depth_range"], que["coords"][:, :200], 24, False)
    hit = orc.alpha_values2hit_prob(torch.rand(1, 200, 24) * 0.4)
    fd_o = orc.sample_fine_depth(depth, hit, que["depth_range"], 16, False)
    fd_g = render_ops.sample_fine_depth(depth.cuda(), hit.cuda(), que["depth_range"].cuda(), 16, False)
    close(fd_g, fd_o, atol=2e-5, what="sample_fine_depth")
    # inv_mode=False (render_ops.py:182,224): resampling directly in depth; both modes pinned to the unmodified reference's
    # results on these inputs (oracle/gen_golden_dropin.py)
    fd_o2 = orc.sample_fine_depth(depth, hit, que["depth_range"], 16, False, inv_mode=False)
    fd_g2 = render_ops.sample_fine_depth(depth.cuda(), hit.cuda(), que["depth_range"].cuda(), 16, False, inv_mode=False)
    close(fd_g2, fd_o2, atol=2e-5, what="sample_fine_depth inv_mode=False")
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dropin_eval.npz"))
    close(fd_o2, torch.from_numpy(z["fine_depth_lin"]), atol=1e-6, what="oracle vs reference, inv_mode=False")
    close(fd_o, torch.from_numpy(z["fine_depth_inv"]), atol=1e-5, what="oracle vs reference, inv_mode=True")


def test_interpolation_backward_matches_the_oracle_autograd(scene):
    """d out / d map of interpolate_feature_map (nr_interpolate_feats_bwd) against autograd over the oracle's bilinear taps, for
    the quarter-resolution maps (align_corners=False branch) and a full-resolution map, with a mask."""
    que, ref, dq, dr = scene
    torch.manual_seed(3)
    h, w = ref["imgs"].shape[-2:]
    for fmap in (ref["ray_feats"], torch.randn(5, 7, h, w)):
        pts = torch.rand(5, 300, 2) * torch.tensor([w + 4.0, h + 4.0]) - 2.0          # some outside: border clamp
        mask = (torch.rand(5, 300) > 0.25).float()
        g_out = torch.randn(5, 300, fmap.shape[1])
        fo = fmap.clone().requires_grad_(True)
        (orc.interpolate_feature_map(fo, pts, mask, h, w) * g_out).sum().backward()
        fg = fmap.cuda().requires_grad_(True)
        out = render_ops.interpolate_feature_map(fg, pts.cuda(), mask.cuda(), h, w)
        (out * g_out.cuda()).sum().backward()
        close(out, orc.interpolate_feature_map(fmap, pts, mask, h, w), atol=2e-5, what="forward")
        close(fg.grad, fo.grad, atol=2e-5, rtol=1e-4, what="d map")
