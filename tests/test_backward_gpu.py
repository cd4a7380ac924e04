"""GPU: the CUDA training backward (nr_render_pass_bwd + nr_tape_gemms, nr_self_hit_prob) where it can be wrong.

A. nr_tape_gemms on its own, at row counts around every 64-row chunk and 128-row tile edge and at the training shape:
   bit-exact on integer operands, accuracy against fp64 relative to a plain fp32 cuBLAS GEMM, and the mapping of its
   output blocks onto parameter gradients.
B. Whole passes (coarse + fine) against the float64 oracle at ragged shapes, every view-count plan, 3 to 256 samples,
   masked and looking-away rays, maps-only and parameters-only gradients; the tape workspaces are poisoned with NaN
   before every backward, so a tape entry the GEMMs read but the backward did not write shows up.
C. The unmodified reference's own gradient goldens (tests/golden/grads_*.npz) through the CUDA backward.
D. A training render() split into chunks that share the tape workspaces, with use_self_hit_prob on both passes.

The float64 oracle is itself pinned to the reference's gradients by tests/test_backward_reference_cpu.py."""
import os

import numpy as np
import pytest
import torch

import neuray_oracle as orc
from gen_golden import flat_cfg
from golden_io import GOLDEN_DIR, GoldenCase
from neuray_b200 import _lib, backward, renderer, synthetic

pytestmark = pytest.mark.gpu
NAN = float("nan")
TILE = backward.TILE


# ----------------------------------------------------------------------------------------------------------------------
# A. nr_tape_gemms

def pass_names(use_vis):
    W = synthetic.make_weights({"dist_decoder_cfg": {"use_vis": use_vis}}, seed=0)
    return [k for k in W if k.startswith("dist_decoder.") or k.startswith("agg_net.")]


def layer_table(use_vis):
    return backward.layer_table(pass_names(use_vis), "dist_decoder", "agg_net", 4 if use_vis else 3)


def make_tapes(rfn, points, fill, seed):
    """The four tapes of a pass with rfn * points rows, valid rows drawn by fill(shape, generator), every row >= M of the
    last tile NaN (allocated, so reading it cannot fault; the kernel must not use it).  rows == 0 still allocates a tile."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    count = {"tape_row": rfn * points, "grad_row": rfn * points, "tape_point": points, "grad_point": points}
    tapes = {}
    for k, sh in backward.tape_shapes(rfn, points).items():
        sh = (max(sh[0], 1),) + sh[1:]
        t = fill(sh, gen)
        pad = torch.arange(sh[0] * TILE, device="cuda").view(sh[0], 1, TILE) >= count[k]
        tapes[k] = t.masked_fill_(pad, NAN)
    return tapes


def ints(sh, gen):
    # exact in tf32 (zero lo part); every partial sum is an integer below 2^24 even at 262 144 rows
    return torch.randint(-2, 3, sh, generator=gen, device="cuda").float()


def same_sign(sh, gen):
    return torch.rand(sh, generator=gen, device="cuda") * 0.5 + 0.5


def normal(sh, gen):
    return torch.randn(sh, generator=gen, device="cuda")


def spread(sh, gen):
    # magnitudes spread over three decades along the contraction index (per row)
    mag = 10.0 ** (torch.rand((sh[0], 1, sh[2]), generator=gen, device="cuda") * 3 - 1.5)
    return torch.randn(sh, generator=gen, device="cuda") * mag


def native_blocks(table, tapes, rows, points, prefill):
    """nr_tape_gemms called directly: [n_out, n_in + 1] (dW | db) per layer, added onto `prefill`."""
    descs = (_lib.NrGemmDesc * len(table))()
    offs, off = [], 0
    for i, (gt, g_slot, n_out, xt, x_slot, n_in, *_rest) in enumerate(table):
        descs[i].g_tape, descs[i].g_slot, descs[i].n_out = gt, g_slot, n_out
        descs[i].x_tape, descs[i].x_slot, descs[i].n_in, descs[i].out_off = xt, x_slot, n_in, off
        offs.append(off)
        off += n_out * (n_in + 1)
    out = torch.full((off,), prefill, dtype=torch.float32, device="cuda")
    p = _lib.ptr
    _lib.call("nr_tape_gemms", descs, len(table), p(tapes["tape_row"]), p(tapes["grad_row"]), rows, p(tapes["tape_point"]),
              p(tapes["grad_point"]), points, p(out), on=out)
    torch.cuda.synchronize()
    return [out[o:o + t[2] * (t[5] + 1)].view(t[2], t[5] + 1) for o, t in zip(offs, table)]


def operands(layer, tapes, rows, points, dtype):
    """(dz [n_out, M], x [n_in + 1, M] with the constant-1 bias input last) of one layer."""
    gt, g_slot, n_out, xt, x_slot, n_in = layer[:6]
    T = (tapes["tape_row"], tapes["grad_row"], tapes["tape_point"], tapes["grad_point"])
    count = (rows, rows, points, points)
    dz = backward._slots(T[gt], g_slot, n_out, count[gt]).to(dtype)
    x = backward._slots(T[xt], x_slot, n_in, count[xt]).to(dtype)
    return dz, torch.cat([x, torch.ones(1, count[xt], dtype=dtype, device=x.device)], 0)


SIZES = [(rfn, pts) for rfn in (1, 3, 10) for pts in (1, 63, 64, 65, 127, 128, 129, 191, 4097)] + \
        [(8, 32768), (8, 32768 + 37), (1, 0)]


@pytest.mark.parametrize("use_vis", [True, False])
@pytest.mark.parametrize("rfn,points", SIZES)
def test_tape_gemms_exact_on_integer_operands(rfn, points, use_vis):
    """Integer operands in {-2..2}: every product and partial sum is exact in tf32 / fp32, so the output must equal the
    exact sum bit for bit whatever the summation order.  Any error in the chunk / tile indexing, the fragment layout, the
    zero fill of the partial chunk, the CTA partition, ksplit or the bias column is a mismatch.  `out` starts at 0.5: the
    ABI adds to it.  (fp64 sums of these integers are exact, so the fp64 GEMM below is the exact reference.)"""
    table = layer_table(use_vis)
    rows = rfn * points
    tapes = make_tapes(rfn, points, ints, seed=rfn * 7919 + points)
    got = native_blocks(table, tapes, rows, points, 0.5)
    for layer, blk in zip(table, got):
        dz, x = operands(layer, tapes, rows, points, torch.float64)
        want = dz @ x.t() + 0.5
        bad = (blk.double() != want)
        assert not bool(bad.any()), (layer[6], rows, int(bad.sum()), float((blk.double() - want).abs().max()))


@pytest.mark.parametrize("fill", [same_sign, normal, spread], ids=["same_sign", "normal", "spread"])
@pytest.mark.parametrize("rfn,points", [(8, 32768), (3, 4097)])
def test_tape_gemms_accuracy_against_fp64(rfn, points, fill, monkeypatch):
    """Real operands against an fp64 GEMM, error normalised element-wise by (|dz| |x|^T)[o, i].  The bar is what a plain
    fp32 cuBLAS GEMM gets on the same data (the GEMM the reference's autograd runs), times 4, plus 2e-6.  The same-sign set
    is the one that exposes a biased (truncating) accumulation: its error grows with the number of chained MMAs."""
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    table = layer_table(True)
    rows = rfn * points
    tapes = make_tapes(rfn, points, fill, seed=11 + points)
    got = native_blocks(table, tapes, rows, points, 0.0)
    worst = (0.0, 0.0, "")
    for layer, blk in zip(table, got):
        dz, x = operands(layer, tapes, rows, points, torch.float64)
        want = dz @ x.t()
        norm = (dz.abs() @ x.abs().t()).clamp_min(1e-300)
        dz32, x32 = dz.float(), x.float()
        blas = (dz32 @ x32.t()).double()
        e_nat = float(((blk.double() - want).abs() / norm).max())
        e_blas = float(((blas - want).abs() / norm).max())
        assert e_nat <= 4 * e_blas + 2e-6, (layer[6], e_nat, e_blas)
        if e_nat > worst[0]:
            worst = (e_nat, e_blas, layer[6])
    print(f"\ntape GEMM {fill.__name__} rows={rows}: worst normalised error {worst[0]:.2e} ({worst[2]}; cuBLAS fp32 {worst[1]:.2e})")


@pytest.mark.parametrize("use_vis", [True, False])
@pytest.mark.parametrize("rfn,points", [(3, 129), (10, 65)])
def test_fused_assembly_maps_blocks_onto_parameters(rfn, points, use_vis):
    """assemble_param_grads_fused (one nr_tape_gemms launch, then the block -> parameter mapping: the LayerNorm diagonal,
    the two-part base_fc.0 weight, weights without bias) against assemble_param_grads on fp64 copies of the same tapes.
    Integer operands: equal bit for bit."""
    names = pass_names(use_vis)
    n_heads = 4 if use_vis else 3
    rows = rfn * points
    tapes = make_tapes(rfn, points, ints, seed=rows)
    t = tapes
    fused = backward.assemble_param_grads_fused(names, "dist_decoder", "agg_net", n_heads, t["tape_row"], t["grad_row"],
                                                t["tape_point"], t["grad_point"], rows, points, _lib.stream_of(t["tape_row"]))
    ref = backward.assemble_param_grads(names, "dist_decoder", "agg_net", n_heads, *(t[k].double() for k in
                                        ("tape_row", "grad_row", "tape_point", "grad_point")), rows, points)
    torch.cuda.synchronize()
    assert set(fused) == set(ref) == set(names)
    n = 0
    for k in names:
        if ref[k] is None:
            assert fused[k] is None, k
            continue
        assert fused[k].shape == ref[k].shape, k
        assert torch.equal(fused[k].double(), ref[k]), (k, float((fused[k].double() - ref[k]).abs().max()))
        n += 1
    assert n == len(names)
    assert fused["agg_net.agg_impl.base_fc.0.weight"].shape == (64, 207)


# ----------------------------------------------------------------------------------------------------------------------
# B. whole passes against the float64 oracle

def f64(d):
    return {k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in d.items()}


def poison_tapes(rfn, points):
    """NaN into the grow-only tape workspaces the next backward will reuse (at least the size it asks for)."""
    for k, sh in backward.tape_shapes(rfn, points).items():
        _lib.workspace(k, sh[0] * sh[1] * sh[2], torch.device("cuda", torch.cuda.current_device()), torch.float32).fill_(NAN)


def check_grads(pairs, what):
    """pairs: [(name, native grad or None, fp64 grad or None)].  Per tensor max|native - fp64| <= 5e-4 max|fp64| + 1e-6 G,
    G = the largest max|fp64| of the test (some gradients are analytically zero, e.g. rgb_fc.4.bias by the shift invariance
    of the view softmax, and come out at rounding level).  Returns [(error / bound, relative error, name)], worst first."""
    G = max((float(b.abs().max()) for _, _, b in pairs if b is not None and b.numel()), default=0.0)
    errs = []
    for name, a, b in pairs:
        if b is None or float(b.abs().max()) == 0.0:
            assert a is None or float(a.abs().max()) <= 1e-6 * G, (what, name)
            continue
        assert a is not None, (what, name)
        assert a.shape == b.shape, (what, name)
        assert bool(torch.isfinite(a).all()), (what, name)
        err, scale = float((a.double().cpu() - b).abs().max()), float(b.abs().max())
        bound = 5e-4 * scale + 1e-6 * G
        assert err <= bound, (what, name, err, scale, G)
        errs.append((err / bound, err / scale, name))
    return sorted(errs, reverse=True)


def report(errs):
    """The tensors closest to the bound, with their error relative to max|fp64|."""
    return "closest to the bound " + ", ".join(f"{n} {f:.2f} of it ({r:.1e} rel)" for f, r, n in errs[:3])


def check_values(a, b, what):
    """The north-star bound of the forward: 1e-4 abs + 1e-3 rel."""
    a, b = a.detach().double().cpu(), b.detach().double()
    assert a.shape == b.shape, what
    assert bool(((a - b).abs() <= 1e-4 + 1e-3 * b.abs()).all()), (what, float((a - b).abs().max()))


# (rfn, rays, coarse dn, fine dn, fine_depth_use_all, coarse use_vis, kind, weight seed); the seeds are picked so that
# neither pass is entirely masked or transparent (every gradient zero)
PASS_CASES = [
    (1, 1, 3, 3, False, False, "plain", 3),
    (2, 7, 5, 6, False, True, "plain", 0),
    (3, 43, 3, 3, False, False, "plain", 0),          # 129 points per pass
    (5, 37, 24, 24, True, True, "plain", 0),          # fine pass 48 samples
    (6, 3, 128, 128, True, False, "plain", 0),        # fine pass 256 samples = NR_MAX_SAMPLES
    (7, 21, 9, 11, False, True, "plain", 0),
    (10, 13, 16, 8, True, False, "plain", 0),
    (13, 11, 7, 7, False, True, "plain", 0),
    (17, 9, 12, 12, False, False, "plain", 0),
    (32, 5, 6, 10, False, True, "plain", 0),
    (4, 64, 8, 8, False, True, "border", 0),          # the image's top row: rays leaving the reference views at the edges
    (4, 24, 8, 8, False, False, "look_away", 0),      # every ray masked (test_parity_gpu::test_rays_looking_away_from_the_scene)
    (5, 17, 10, 10, True, True, "maps_only", 0),
    (3, 17, 10, 10, False, False, "params_only", 0),  # d_feat is NULL
    (8, 65, 4, 4, False, True, "plain", 0),
]


def pass_cfg(dc, df, use_all, use_vis):
    return {"use_hierarchical_sampling": True, "depth_sample_num": dc, "fine_depth_sample_num": df, "fine_depth_use_all": use_all,
            "agg_net_cfg": {"sample_num": dc}, "fine_agg_net_cfg": {"sample_num": df + (dc if use_all else 0)},
            "dist_decoder_cfg": {"use_vis": use_vis}, "render_depth": True}


def loss_weights(shapes, seed):
    gen = torch.Generator().manual_seed(seed)
    return {k: torch.randn(sh, generator=gen, dtype=torch.float64) for k, sh in shapes.items()}


def linear_loss(outs, lw):
    return sum((outs[k] * (lw[k] if outs[k].dtype == torch.float64 else lw[k].to(outs[k]))).sum() for k in lw)


@pytest.mark.parametrize("rfn,rays,dc,df,use_all,use_vis,kind,wseed", PASS_CASES,
                         ids=[f"v{c[0]}_r{c[1]}_d{c[2]}-{c[3]}{'all' if c[4] else ''}_{'vis' if c[5] else 'novis'}_{c[6]}" for c in PASS_CASES])
def test_render_passes_backward_matches_fp64_oracle(rfn, rays, dc, df, use_all, use_vis, kind, wseed):
    seed = rfn * 100 + rays
    cfg = pass_cfg(dc, df, use_all, use_vis)
    que, ref = synthetic.make_scene(48, 64, rfn, seed=seed, smooth=2)
    start = 0 if kind == "border" else 1184
    que = synthetic.slice_rays(que, start, start + rays)
    if kind == "look_away":
        que["poses"] = que["poses"].clone()
        que["poses"][:, :, :3] = que["poses"][:, :, :3] * torch.tensor([1.0, 1.0, -1.0])[None, :, None]
    W = synthetic.make_weights(cfg, seed=wseed)
    want_params, want_maps = kind != "maps_only", kind != "params_only"
    depth = orc.sample_depth(que["depth_range"], que["coords"], dc, False)[0]

    # float64 oracle; the fine pass runs on depths resampled from the oracle's coarse hit probabilities, given to both sides
    Wo = {k: v.double().requires_grad_(want_params) for k, v in W.items()}
    ro, qo = f64(ref), f64(que)
    ro["ray_feats"].requires_grad_(want_maps)
    ro["img_feats"].requires_grad_(want_maps)
    ocfg = flat_cfg({**renderer.base_cfg, **cfg})
    oc = orc.render_by_depth(Wo, ocfg, depth.double(), qo, ro, True, False)
    fd = orc.sample_fine_depth(depth, oc["hit_prob_nr"].detach().float(), que["depth_range"], df, False)
    fd = torch.sort(torch.cat([depth, fd], -1) if use_all else fd, -1)[0].contiguous()
    of = orc.render_by_depth(Wo, ocfg, fd.double(), qo, ro, True, True)
    keys = ("pixel_colors_nr", "hit_prob_nr", "render_depth")
    lw_c = loss_weights({k: oc[k].shape for k in keys}, seed)
    lw_f = loss_weights({k: of[k].shape for k in keys}, seed + 1)
    (linear_loss(oc, lw_c) + linear_loss(of, lw_f)).backward()
    if kind == "look_away":
        assert not bool(oc["ray_mask"].any())

    # CUDA: RenderPassFn -> nr_render_pass_bwd + nr_tape_gemms, one backward per pass, each on poisoned tapes
    net = renderer.NeuralRayRenderPath(cfg)
    net.load_state_dict(W, strict=True)
    net.cuda()
    if not want_params:
        net.requires_grad_(False)
    dq, dr = synthetic.to_device(que, "cuda"), synthetic.to_device(ref, "cuda")
    dr["ray_feats"].requires_grad_(want_maps)
    dr["img_feats"].requires_grad_(want_maps)
    pc = net.render_by_depth(depth.cuda(), dq, dr, True, False)
    pf = net.render_by_depth(fd.cuda(), dq, dr, True, True)
    for k in keys:
        check_values(pc[k], oc[k], f"{k} coarse")
        check_values(pf[k], of[k], f"{k} fine")
    for outs, lw, n_pts in ((pf, lw_f, rays * fd.shape[-1]), (pc, lw_c, rays * dc)):
        torch.cuda.synchronize()
        poison_tapes(rfn, n_pts)
        linear_loss(outs, lw).backward()
    torch.cuda.synchronize()

    pairs = [(k, p.grad, Wo[k].grad) for k, p in net.named_parameters()]
    pairs += [(k, dr[k].grad, ro[k].grad) for k in ("ray_feats", "img_feats")]
    if not want_params:
        assert all(p.grad is None for p in net.parameters())
    if not want_maps:
        assert dr["ray_feats"].grad is None and dr["img_feats"].grad is None
    errs = check_grads(pairs, kind)
    assert len(errs) == 2 if not want_params else len(errs) > 100
    print(f"\n{kind} rfn={rfn} rays={rays} dn={dc}/{fd.shape[-1]}: " + report(errs))


# ----------------------------------------------------------------------------------------------------------------------
# C. the reference's own gradient goldens through the CUDA backward

def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, f"grads_{name}.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def golden_bound(got, gold, what):
    """The bound of the host-build tests (tests/test_backward_cpu.py)."""
    err, scale = float((got.detach().cpu() - gold).abs().max()), float(gold.abs().max())
    assert err <= 3e-4 * max(scale, 1e-3) + 3e-6, (what, err, scale)
    return err / max(scale, 1e-3)


def golden_path(g):
    net = renderer.NeuralRayRenderPath(g.cfg)
    net.load_state_dict(g.W, strict=True)
    return net.cuda()


@pytest.mark.parametrize("name", ["train8", "views10"])
def test_cuda_backward_matches_the_reference_gradients(name):
    """tests/test_backward_cpu.py::test_hand_written_backward_matches_the_reference_gradients on the GPU: coarse + fine
    render_by_depth on the golden case's stage rays, the generator's linear loss, every parameter and both maps."""
    g, z = GoldenCase(name), load_golden(name)
    sel = g.stage_sel
    net = golden_path(g)
    dq, dr = synthetic.to_device(g.stage_que(), "cuda"), synthetic.to_device(g.ref, "cuda")
    dr["ray_feats"].requires_grad_(True)
    dr["img_feats"].requires_grad_(True)
    pc = net.render_by_depth(g.que_depth[:, sel].contiguous().cuda(), dq, dr, True, False)
    pf = net.render_by_depth(g.que_depth_fine[:, sel].contiguous().cuda(), dq, dr, True, True)
    lw = {k[3:]: v.cuda() for k, v in z.items() if k.startswith("lw_")}
    loss = (pc["pixel_colors_nr"] * lw["gw_c"]).sum() + (pc["hit_prob_nr"] * lw["gh_c"]).sum() \
        + (pf["pixel_colors_nr"] * lw["gw_f"]).sum() + (pf["render_depth"] * lw["gd_f"]).sum()
    loss.backward()
    torch.cuda.synchronize()
    gold = {k[5:]: v for k, v in z.items() if k.startswith("grad_")}
    worst = (0.0, "")
    for k, p in net.named_parameters():
        if k not in gold:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        assert p.grad is not None, k
        worst = max(worst, (golden_bound(p.grad, gold[k], k), k))
    for k in ("ray_feats", "img_feats"):
        worst = max(worst, (golden_bound(dr[k].grad, gold["ref_" + k], k), k))
    assert len(gold) > 100
    print(f"\n{name}: worst error against the reference's gradients {worst[0]:.1e} ({worst[1]})")


@pytest.mark.parametrize("name", ["train8", "views10"])
def test_cuda_self_hit_prob_matches_the_reference(name):
    """nr_self_hit_prob on the GPU against predict_self_hit_prob of the unmodified reference: values, every decoder
    parameter gradient and the query feature map gradient."""
    g, z = GoldenCase(name), load_golden(name)
    sel = g.stage_sel
    net = golden_path(g)
    dq = synthetic.to_device(g.stage_que(), "cuda")
    dq["ray_feats"] = z["self_map"].cuda().requires_grad_(True)
    hit = renderer._self_hit_prob(net, g.que_depth[:, sel].contiguous().cuda(), dq, False)
    (hit * z["self_gs"].cuda()).sum().backward()
    torch.cuda.synchronize()
    assert float((hit.detach().cpu() - z["self_hit"]).abs().max()) <= 2e-6
    named = dict(net.named_parameters())
    checked = 0
    for k, ga in z.items():
        if k.startswith("selfgrad_"):
            assert named[k[9:]].grad is not None, k
            golden_bound(named[k[9:]].grad, ga, k)
            checked += 1
    assert checked >= 18
    golden_bound(dq["ray_feats"].grad, z["self_grad_map"], "self_grad_map")


# ----------------------------------------------------------------------------------------------------------------------
# D. a training render() in several chunks

def test_chunked_training_render_matches_fp64_oracle(monkeypatch):
    """render(que, ref, True) over 257 rays in chunks of 100, 100 and 57: the chunks' backwards share the grow-only tape
    workspaces (poisoned first) and their gradients add up in the same leaves.  fine_depth_use_all, use_self_hit_prob on
    both passes with a query ray_feats that wants a gradient, a seeded linear loss over every output.  The oracle runs
    chunk by chunk on the depths each chunk's passes were given; separately, the fused resampling that made the fine depths
    is checked against the oracle's sample_fine_depth on the same uniforms."""
    cfg = {"use_hierarchical_sampling": True, "depth_sample_num": 16, "fine_depth_sample_num": 16, "fine_depth_use_all": True,
           "agg_net_cfg": {"sample_num": 16}, "fine_agg_net_cfg": {"sample_num": 32}, "dist_decoder_cfg": {"use_vis": True},
           "render_depth": True, "use_self_hit_prob": True, "ray_batch_num": 100}
    rfn, rays = 5, 257
    que, ref = synthetic.make_scene(48, 64, rfn, seed=57, smooth=2)
    que = synthetic.slice_rays(que, 1200, 1200 + rays)
    qmap = torch.from_numpy(np.random.RandomState(3).standard_normal((1, 32, 12, 16)).astype(np.float32))
    W = synthetic.make_weights(cfg, seed=12)
    net = renderer.NeuralRayRenderPath(cfg)
    net.load_state_dict(W, strict=True)
    net.cuda()
    dq, dr = synthetic.to_device(que, "cuda"), synthetic.to_device(ref, "cuda")
    dq["ray_feats"] = qmap.cuda().requires_grad_(True)
    dr["ray_feats"].requires_grad_(True)
    dr["img_feats"].requires_grad_(True)

    passes = []
    run_pass = renderer.run_pass

    def recording_run_pass(owner, que_depth, que_imgs_info, ref_imgs_info, is_fine, **kw):
        passes.append((is_fine, que_imgs_info["coords"].shape[1], que_depth.detach().cpu().clone()))
        return run_pass(owner, que_depth, que_imgs_info, ref_imgs_info, is_fine, **kw)

    monkeypatch.setattr(renderer, "run_pass", recording_run_pass)
    torch.manual_seed(4321)
    out = net.render(dq, dr, True)
    monkeypatch.undo()
    torch.cuda.synchronize()
    assert [(f, n) for f, n, _ in passes] == [(False, 100), (True, 100), (False, 100), (True, 100), (False, 57), (True, 57)]
    diff = [k for k, v in out.items() if v.dtype.is_floating_point and v.requires_grad]
    assert {"pixel_colors_nr", "hit_prob_nr", "render_depth", "hit_prob_self", "pixel_colors_nr_fine", "hit_prob_nr_fine",
            "render_depth_fine", "hit_prob_self_fine"} <= set(diff)
    lw = loss_weights({k: out[k].shape for k in diff}, 99)
    fd_n = passes[1][2].shape[-1]
    poison_tapes(rfn, 100 * fd_n)
    linear_loss(out, lw).backward()
    torch.cuda.synchronize()

    # float64 oracle, chunk by chunk on the recorded depths
    Wo = {k: v.double().requires_grad_(True) for k, v in W.items()}
    ro, qo = f64(ref), f64(que)
    for k in ("ray_feats", "img_feats"):
        ro[k].requires_grad_(True)
    qmo = qmap.double().requires_grad_(True)
    ocfg = flat_cfg({**renderer.base_cfg, **cfg})
    loss, chunk_outs, s = 0.0, [], 0
    for i in range(3):
        dc, df = passes[2 * i][2], passes[2 * i + 1][2]
        n = dc.shape[1]
        q = dict(qo, coords=qo["coords"][:, s:s + n], ray_feats=qmo)
        o = {}
        for suffix, depth, is_fine in (("", dc.double(), False), ("_fine", df.double(), True)):
            r = orc.render_by_depth(Wo, ocfg, depth, q, ro, True, is_fine)
            r["hit_prob_self"] = orc.predict_self_hit_prob(Wo, ocfg, q, depth, orc.depth2inv_dists(depth, q["depth_range"]), is_fine)
            o.update({k + suffix: v for k, v in r.items()})
        loss = loss + sum((o[k] * lw[k][:, s:s + n]).sum() for k in diff)
        chunk_outs.append(o)
        s += n
    loss.backward()
    for k in diff:
        check_values(out[k], torch.cat([o[k] for o in chunk_outs], 1), k)
    pairs = [(k, p.grad, Wo[k].grad) for k, p in net.named_parameters()]
    pairs += [(k, dr[k].grad, ro[k].grad) for k in ("ray_feats", "img_feats")]
    pairs.append(("que ray_feats", dq["ray_feats"].grad, qmo.grad))
    errs = check_grads(pairs, "chunked render")
    assert len(errs) > 120
    print("\nchunked render: " + report(errs))

    # the fused resampling of each chunk against the oracle's, same uniforms in the same order
    torch.manual_seed(4321)
    close_bad, total = 0, 0
    for i in range(3):
        dc, df = passes[2 * i][2], passes[2 * i + 1][2]
        n = dc.shape[1]
        u = torch.rand([1, n, cfg["fine_depth_sample_num"]])
        hit = chunk_outs[i]["hit_prob_nr"].detach().float()
        fd = orc.sample_fine_depth(dc, hit, que["depth_range"], cfg["fine_depth_sample_num"], True, u)
        fd = torch.sort(torch.cat([dc, fd], -1), -1)[0]
        ok = (df - fd).abs() <= 1e-4 + 1e-3 * fd.abs()
        close_bad += int((~ok).sum())
        total += ok.numel()
    assert close_bad <= 5e-3 * total, (close_bad, total)
