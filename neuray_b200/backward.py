"""Native backward of one render pass: `nr_render_pass_bwd` fills the tapes, the weight gradients are GEMMs over them.

Reference: the gradients `loss.backward()` sends through `NeuralRayBaseRenderer.render_by_depth` (renderer.py:168-203)
into `dist_decoder` / `agg_net` parameters and the encoder outputs `ray_feats` / `img_feats`.
"""
import ctypes as C

import torch

from . import _lib

HEADS = ("mean_decoder", "var_decoder", "aw_decoder", "vis_decoder")
TILE = 128


def tape_shapes(rfn, n_points):
    """Tape buffers as [tiles, slots, 128] (layout: include/neuray_b200.h, NrBwdParams)."""
    s = _lib.bwd_slot
    rows = rfn * n_points
    t = lambda m: (m + TILE - 1) // TILE
    return {"tape_row": (t(rows), s("R_SLOTS"), TILE), "grad_row": (t(rows), s("G_SLOTS"), TILE),
            "tape_point": (t(n_points), s("P_SLOTS"), TILE), "grad_point": (t(n_points), s("GP_SLOTS"), TILE)}


def _slots(tape, slot, n, rows):
    """[n, rows] view-copy of n consecutive slots of a tiled tape."""
    return tape[:, slot:slot + n, :].permute(1, 0, 2).reshape(n, -1)[:, :rows]


ROW, GROW, POINT, GPOINT = 0, 1, 2, 3      # tape numbers of nr_tape_gemms


def layer_table(names, dec, agg, n_heads):
    """Every Linear of the pass as (g_tape, g_slot, n_out, x_tape, x_slot, n_in, weight name, bias name, kind)."""
    s = _lib.bwd_slot
    T = []

    def add(gt, g_slot, n_out, xt, x_slot, n_in, w, b, kind="plain"):
        T.append((gt, g_slot, n_out, xt, x_slot, n_in, w, b, kind))

    for hd, head in enumerate(HEADS):
        # a head the pass does not evaluate (the fine decoder's vis head under a coarse use_vis=False) gets no gradient
        if f"{dec}.{head}.0.weight" not in names or hd >= n_heads:
            continue
        add(GROW, s("G_DD0") + 32 * hd, 32, ROW, s("R_RF"), 32, f"{dec}.{head}.0.weight", f"{dec}.{head}.0.bias")
        add(GROW, s("G_DD1") + 32 * hd, 32, ROW, s("R_H1") + 32 * hd, 32, f"{dec}.{head}.2.weight", f"{dec}.{head}.2.bias")
        add(GROW, s("G_DD2") + 2 * hd, 2 if hd < 2 else 1, ROW, s("R_H2") + 32 * hd, 32, f"{dec}.{head}.4.weight", f"{dec}.{head}.4.bias")
    ib = f"{agg}.agg_impl"
    at = f"{ib}.ray_attention"
    add(GROW, s("G_PE0"), 32, ROW, s("R_RF"), 34, f"{agg}.prob_embed.0.weight", f"{agg}.prob_embed.0.bias")
    add(GROW, s("G_PE1"), 32, ROW, s("R_P1"), 32, f"{agg}.prob_embed.2.weight", f"{agg}.prob_embed.2.bias")
    add(GROW, s("G_RD0"), 16, ROW, s("R_DD"), 4, f"{ib}.ray_dir_fc.0.weight", f"{ib}.ray_dir_fc.0.bias")
    add(GROW, s("G_RD1"), 35, ROW, s("R_R16"), 16, f"{ib}.ray_dir_fc.2.weight", f"{ib}.ray_dir_fc.2.bias")
    add(GROW, s("G_NF0"), 8, ROW, s("R_NF"), 32, f"{ib}.neuray_fc.0.weight", f"{ib}.neuray_fc.0.bias")
    add(GROW, s("G_NF1"), 1, ROW, s("R_Q8"), 8, f"{ib}.neuray_fc.2.weight", f"{ib}.neuray_fc.2.bias")
    add(GPOINT, s("GP_B0SUM"), 64, POINT, s("P_GLOB"), 140, f"{ib}.base_fc.0.weight", None, "base_glob")
    add(GROW, s("G_B0"), 64, ROW, s("R_RGBF"), 67, f"{ib}.base_fc.0.weight", f"{ib}.base_fc.0.bias", "base_row")
    add(GROW, s("G_B1"), 32, ROW, s("R_B1"), 64, f"{ib}.base_fc.2.weight", f"{ib}.base_fc.2.bias")
    add(GROW, s("G_V0"), 32, ROW, s("R_U"), 32, f"{ib}.vis_fc.0.weight", f"{ib}.vis_fc.0.bias")
    add(GROW, s("G_V1"), 33, ROW, s("R_VH"), 32, f"{ib}.vis_fc.2.weight", f"{ib}.vis_fc.2.bias")
    add(GROW, s("G_V20"), 32, ROW, s("R_U2"), 32, f"{ib}.vis_fc2.0.weight", f"{ib}.vis_fc2.0.bias")
    add(GROW, s("G_V21"), 1, ROW, s("R_WH"), 32, f"{ib}.vis_fc2.2.weight", f"{ib}.vis_fc2.2.bias")
    add(GROW, s("G_C0"), 16, ROW, s("R_X2"), 37, f"{ib}.rgb_fc.0.weight", f"{ib}.rgb_fc.0.bias")
    add(GROW, s("G_C1"), 8, ROW, s("R_CH1"), 16, f"{ib}.rgb_fc.2.weight", f"{ib}.rgb_fc.2.bias")
    add(GROW, s("G_C2"), 1, ROW, s("R_CH2"), 8, f"{ib}.rgb_fc.4.weight", f"{ib}.rgb_fc.4.bias")
    add(GPOINT, s("GP_GEO0"), 64, POINT, s("P_GIN"), 65, f"{ib}.geometry_fc.0.weight", f"{ib}.geometry_fc.0.bias")
    add(GPOINT, s("GP_GEO1"), 16, POINT, s("P_GH"), 64, f"{ib}.geometry_fc.2.weight", f"{ib}.geometry_fc.2.bias")
    add(GPOINT, s("GP_DQ"), 16, POINT, s("P_AX"), 16, f"{at}.w_qs.weight", None)
    add(GPOINT, s("GP_DK"), 16, POINT, s("P_AX"), 16, f"{at}.w_ks.weight", None)
    add(GPOINT, s("GP_DV"), 16, POINT, s("P_AX"), 16, f"{at}.w_vs.weight", None)
    add(GPOINT, s("GP_DFC"), 16, POINT, s("P_O"), 16, f"{at}.fc.weight", None)
    add(GPOINT, s("GP_DLNY"), 16, POINT, s("P_XH"), 16, f"{at}.layer_norm.weight", f"{at}.layer_norm.bias", "ln")
    add(GPOINT, s("GP_OG0"), 16, POINT, s("P_Y"), 16, f"{ib}.out_geometry_fc.0.weight", f"{ib}.out_geometry_fc.0.bias")
    add(GPOINT, s("GP_OG1"), 1, POINT, s("P_T16"), 16, f"{ib}.out_geometry_fc.2.weight", f"{ib}.out_geometry_fc.2.bias")
    return T


def _finish(names, table, blocks):
    """blocks[i] = [n_out, n_in + 1] (dW | db) of table[i] -> {name: grad or None}."""
    out, base = {}, {}
    for (gt, g_slot, n_out, xt, x_slot, n_in, w, b, kind), blk in zip(table, blocks):
        if kind == "ln":
            out[w] = torch.diagonal(blk[:, :n_in]).clone()
            out[b] = blk[:, n_in].clone()
            continue
        if kind in ("base_glob", "base_row"):
            base[kind] = blk[:, :n_in]
            if b is not None:
                out[b] = blk[:, n_in].clone()
            continue
        out[w] = blk[:, :n_in].clone()
        if b is not None:
            out[b] = blk[:, n_in].clone()
    wname = next(w for (*_, w, _b, kind) in table if kind == "base_glob")
    out[wname] = torch.cat([base["base_glob"], base["base_row"]], 1)
    return {n: out.get(n) for n in names}


def assemble_param_grads(names, dec, agg, n_heads, tape_row, grad_row, tape_point, grad_point, rows, points):
    """dW = dz @ x^T for every Linear of the pass (bias = row sums of dz) with torch GEMMs over the tapes (any device;
    the CUDA path uses one fused launch instead, `assemble_param_grads_fused`).  Returns {name: grad or None}."""
    tapes = (tape_row, grad_row, tape_point, grad_point)
    count = (rows, rows, points, points)
    table = layer_table(names, dec, agg, n_heads)
    blocks = []
    for gt, g_slot, n_out, xt, x_slot, n_in, *_ in table:
        dz = _slots(tapes[gt], g_slot, n_out, count[gt])
        blocks.append(torch.cat([dz @ _slots(tapes[xt], x_slot, n_in, count[xt]).t(), dz.sum(1, keepdim=True)], 1))
    return _finish(names, table, blocks)


_DESC_CACHE = {}


def assemble_param_grads_fused(names, dec, agg, n_heads, tape_row, grad_row, tape_point, grad_point, rows, points, stream):
    """Same result through nr_tape_gemms: all layers in one launch."""
    key = (tuple(names), dec, agg, n_heads)
    hit = _DESC_CACHE.get(key)
    if hit is None:
        table = layer_table(names, dec, agg, n_heads)
        descs = (_lib.NrGemmDesc * len(table))()
        off = 0
        offs = []
        for i, (gt, g_slot, n_out, xt, x_slot, n_in, *_rest) in enumerate(table):
            descs[i].g_tape, descs[i].g_slot, descs[i].n_out = gt, g_slot, n_out
            descs[i].x_tape, descs[i].x_slot, descs[i].n_in, descs[i].out_off = xt, x_slot, n_in, off
            offs.append(off)
            off += n_out * (n_in + 1)
        hit = (table, descs, offs, off)
        _DESC_CACHE[key] = hit
    table, descs, offs, total = hit
    out = torch.zeros(total, dtype=torch.float32, device=tape_row.device)
    _lib.call("nr_tape_gemms", descs, len(table), _lib.ptr(tape_row), _lib.ptr(grad_row), rows, _lib.ptr(tape_point), _lib.ptr(grad_point), points,
              _lib.ptr(out), on=out, stream=stream)
    blocks = [out[o:o + t[2] * (t[5] + 1)].view(t[2], t[5] + 1) for o, t in zip(offs, table)]
    return _finish(names, table, blocks)


def feat_grads_to_nchw(d_feat):
    """[rfn,fh,fw,64] channel-last gradient -> (d_ray_feats, d_img_feats), both [rfn,32,fh,fw]."""
    g = d_feat.permute(0, 3, 1, 2)
    return g[:, :32].contiguous(), g[:, 32:].contiguous()


def render_pass_backward(p, names, dec, agg, g_pix, g_hit, g_depth, want_feat_grads, feat_shape, stream):
    """p: the NrPassParams of the forward launch (CUDA).  Returns ({name: grad}, d_ray_feats, d_img_feats)."""
    dev = (g_pix if g_pix is not None else g_hit if g_hit is not None else g_depth).device
    n_points = p.rn * p.dn
    shapes = tape_shapes(p.rfn, n_points)
    bufs = {k: _lib.workspace(k, sh[0] * sh[1] * sh[2], dev, torch.float32).view(sh) for k, sh in shapes.items()}
    d_feat = torch.zeros(feat_shape, dtype=torch.float32, device=dev) if want_feat_grads else None
    b = _lib.NrBwdParams()
    keep = [_lib.f32(t) if t is not None else None for t in (g_pix, g_hit, g_depth)]
    b.d_pixel_colors, b.d_hit_prob, b.d_render_depth = (_lib.ptr(t) for t in keep)
    b.tape_row, b.grad_row = _lib.ptr(bufs["tape_row"]), _lib.ptr(bufs["grad_row"])
    b.tape_point, b.grad_point = _lib.ptr(bufs["tape_point"]), _lib.ptr(bufs["grad_point"])
    b.d_feat = _lib.ptr(d_feat)
    _lib.call("nr_render_pass_bwd", C.byref(p), C.byref(b), on=bufs["tape_row"], stream=stream, kernels=11)
    grads = assemble_param_grads_fused(names, dec, agg, 4 if p.use_vis else 3, bufs["tape_row"], bufs["grad_row"], bufs["tape_point"],
                                       bufs["grad_point"], p.rfn * n_points, n_points, stream)
    if d_feat is None:
        return grads, None, None
    drf, dimf = feat_grads_to_nchw(d_feat)
    return grads, drf, dimf


def unpack_point_grads(index_map, d_w_point):
    """Gradient in the packed w_point layout -> {name: grad}: every parameter element sits at exactly one packed
    position (weights.point_index_map: position -> 1 + flat parameter index, 0 = padding)."""
    i_point, names, sizes, shapes = index_map
    flat = torch.zeros(1 + sum(sizes), dtype=torch.float32, device=d_w_point.device).index_add_(0, i_point, d_w_point)
    out, off = {}, 1
    for name, n, shape in zip(names, sizes, shapes):
        out[name] = flat[off:off + n].view(shape)
        off += n
    return out


class RenderPassFn(torch.autograd.Function):
    """forward = the fused CUDA pass (values), backward = nr_render_pass_bwd + nr_tape_gemms."""

    @staticmethod
    def forward(ctx, runner, meta, ray_feats, img_feats, *params):
        with torch.no_grad():
            res = runner()
        ctx.meta = meta
        ctx.bwd = res.pop("_bwd", None)
        ctx.save_for_backward(ray_feats, img_feats, *params)
        ctx.mark_non_differentiable(res["ray_mask_u8"])
        fine = res.get("fine_depth")
        outs = (res["pixel_colors"], res["hit_prob"], res["render_depth"], res["ray_mask_u8"])
        if fine is not None:
            ctx.mark_non_differentiable(fine)
            return outs + (fine,)
        return outs

    @staticmethod
    def backward(ctx, g_pix, g_hit, g_depth, *unused):
        meta = ctx.meta
        ray_feats, img_feats, *params = ctx.saved_tensors
        if ctx.bwd is None:          # an empty chunk: nothing was launched, nothing flows back
            return (None, None, None, None, *[None] * len(params))
        p, _keep, feat_shape, stream = ctx.bwd
        want_feat = ray_feats.requires_grad or img_feats.requires_grad
        grads, drf, dimf = render_pass_backward(p, meta["names"], meta["dec"], meta["agg"], g_pix, g_hit, g_depth, want_feat, feat_shape, stream)
        gp = [grads[n] if t.requires_grad else None for n, t in zip(meta["names"], params)]
        return (None, None, drf if ray_feats.requires_grad else None, dimf if img_feats.requires_grad else None, *gp)


class SelfHitProbFn(torch.autograd.Function):
    """predict_self_hit_prob (reference renderer.py:137-155) through nr_self_hit_prob, forward and backward."""

    @staticmethod
    def forward(ctx, meta, que_ray_feats, *dec_params):
        p = meta["params"]()
        hit = torch.empty(p.rn, p.dn, dtype=torch.float32, device=que_ray_feats.device)
        p.hit = _lib.ptr(hit)
        _lib.call("nr_self_hit_prob", C.byref(p), on=que_ray_feats, stream=meta["stream"])
        ctx.meta = meta
        ctx.feats_need = que_ray_feats.requires_grad
        ctx.need = [t.requires_grad for t in dec_params]
        return hit[None]

    @staticmethod
    def backward(ctx, g_hit):
        meta = ctx.meta
        index_map = meta["index_map"]
        p = meta["params"]()
        dev = g_hit.device
        g = _lib.f32(g_hit[0])
        hit = torch.empty(p.rn, p.dn, dtype=torch.float32, device=dev)
        d_w = torch.zeros(index_map[0].numel(), dtype=torch.float32, device=dev)
        d_map = torch.zeros(meta["map_shape"], dtype=torch.float32, device=dev) if ctx.feats_need else None
        p.hit, p.d_hit, p.d_w_point, p.d_map = _lib.ptr(hit), _lib.ptr(g), _lib.ptr(d_w), _lib.ptr(d_map)
        _lib.call("nr_self_hit_prob", C.byref(p), on=g_hit, stream=meta["stream"], what="nr_self_hit_prob (backward)")
        grads = unpack_point_grads(index_map, d_w)
        gp = [grads[n] if need else None for n, need in zip(meta["dec_names"], ctx.need)]
        return (None, d_map[None] if d_map is not None else None, *gp)
