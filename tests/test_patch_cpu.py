"""CPU: patch.install() rebinds the reference's API onto the B200 path and patch.uninstall() puts it back.

The reference's `network` package is stood in for by empty modules that carry its module, class, function and loss names
(network.render_ops, network.renderer, network.init_net, network.loss): install() finds what it rebinds by those names."""
import sys
import types

import pytest
import torch.nn as nn

from neuray_b200 import _lib, losses, modules, patch, render_ops, renderer


def _placeholder(*a, **k):
    raise AssertionError("the reference's own function was called")


@pytest.fixture
def reference_names():
    """sys.modules['network.*'] with the reference's names bound to placeholders; removed again afterwards."""
    saved = {k: v for k, v in sys.modules.items() if k == "network" or k.startswith("network.")}
    ops = types.ModuleType("network.render_ops")
    ren = types.ModuleType("network.renderer")
    ini = types.ModuleType("network.init_net")
    loss = types.ModuleType("network.loss")
    for n in render_ops.__all__:
        setattr(ops, n, _placeholder)
        setattr(ren, n, _placeholder)          # renderer.py star-imports render_ops
    ini.get_diff_feats = _placeholder
    ini.interpolate_feature_map = _placeholder

    class NeuralRayBaseRenderer(nn.Module):
        """Builds the hot-path modules under the reference's names (renderer.py:36-73), nothing else."""

        def __init__(self, cfg):
            super().__init__()
            self.cfg = {**renderer.base_cfg, **cfg}
            self.dist_decoder = modules.name2dist_decoder[self.cfg["dist_decoder_type"]](self.cfg["dist_decoder_cfg"])
            self.agg_net = modules.name2agg_net[self.cfg["agg_net_type"]](self.cfg["agg_net_cfg"])
            if self.cfg["use_hierarchical_sampling"]:
                self.fine_dist_decoder = modules.name2dist_decoder[self.cfg["dist_decoder_type"]](self.cfg["fine_dist_decoder_cfg"])
                self.fine_agg_net = modules.name2agg_net[self.cfg["agg_net_type"]](self.cfg["fine_agg_net_cfg"])

        render_by_depth = fine_render_impl = render_impl = render = _placeholder

    class NeuralRayGenRenderer(NeuralRayBaseRenderer):
        predict_mean_for_depth_loss = _placeholder

    class DepthInitNet(nn.Module):
        forward = _placeholder

    class CostVolumeInitNet(nn.Module):
        forward = _placeholder

    ren.NeuralRayBaseRenderer, ren.NeuralRayGenRenderer = NeuralRayBaseRenderer, NeuralRayGenRenderer
    ini.DepthInitNet, ini.CostVolumeInitNet = DepthInitNet, CostVolumeInitNet
    loss.name2loss = {}
    for key, cls in losses.name2loss.items():
        placeholder = type(cls.__name__, (), {})
        setattr(loss, cls.__name__, placeholder)
        loss.name2loss[key] = placeholder
    pkg = types.ModuleType("network")
    pkg.__path__ = []
    mods = {"network": pkg, "network.render_ops": ops, "network.renderer": ren, "network.init_net": ini, "network.loss": loss}
    sys.modules.update(mods)
    try:
        yield mods
    finally:
        patch.uninstall()
        for k in mods:
            sys.modules.pop(k, None)
        sys.modules.update(saved)


def test_install_rebinds_reference_api(reference_names):
    ref_renderer, ref_ops, ref_loss, ref_init = (reference_names[f"network.{n}"] for n in ("renderer", "render_ops", "loss", "init_net"))
    orig = {k: getattr(ref_renderer.NeuralRayBaseRenderer, k) for k in ("render_by_depth", "render_impl", "fine_render_impl", "render")}
    orig_ops = {n: getattr(ref_ops, n) for n in render_ops.__all__ if hasattr(ref_ops, n)}
    orig_ren = {n: getattr(ref_renderer, n) for n in render_ops.__all__ if hasattr(ref_renderer, n)}
    orig_loss = dict(ref_loss.name2loss)
    orig_pm = ref_renderer.NeuralRayGenRenderer.predict_mean_for_depth_loss
    orig_init = (ref_init.get_diff_feats, ref_init.DepthInitNet.forward, ref_init.CostVolumeInitNet.forward)
    try:
        base = patch.install()
        assert base is ref_renderer.NeuralRayBaseRenderer
        assert base.render_impl is renderer.render_impl and base.render is renderer.render
        assert ref_loss.name2loss == losses.name2loss and ref_loss.DepthLoss is losses.DepthLoss
        assert ref_renderer.NeuralRayGenRenderer.predict_mean_for_depth_loss is losses.predict_mean_for_depth_loss
        assert ref_init.get_diff_feats is not orig_init[0] and ref_init.DepthInitNet.forward is not orig_init[1]
        assert ref_init.CostVolumeInitNet.forward is not orig_init[2]
        for n in orig_ops:
            assert getattr(ref_ops, n) is getattr(render_ops, n), n
        # the reference's own constructor still builds the network; the hot path now refuses CPU tensors (no fallback)
        net = base({"use_hierarchical_sampling": True})
        assert set(k.split(".")[0] for k in net.state_dict()) >= {"dist_decoder", "agg_net", "fine_dist_decoder", "fine_agg_net"}
        from neuray_b200 import synthetic
        que, ref = synthetic.make_scene(32, 32, 3, seed=0)
        with pytest.raises(_lib.NeurayB200Error):
            net.render_impl(que, dict(ref), False)
    finally:
        patch.uninstall()
    for k, v in orig.items():
        assert getattr(ref_renderer.NeuralRayBaseRenderer, k) is v, k
    assert ref_loss.name2loss == orig_loss and ref_renderer.NeuralRayGenRenderer.predict_mean_for_depth_loss is orig_pm
    assert (ref_init.get_diff_feats, ref_init.DepthInitNet.forward, ref_init.CostVolumeInitNet.forward) == orig_init
    for n, v in orig_ops.items():
        assert getattr(ref_ops, n) is v, n
    for n, v in orig_ren.items():
        assert getattr(ref_renderer, n) is v, n
