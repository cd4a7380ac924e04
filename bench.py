#!/usr/bin/env python
"""bench.py -- ray-samples/s of the per-ray rendering hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload black_800|black_400|cfg1|fern_high|train_dtu] [--shard images|rays] [--dump-outputs DIR]

Headline (default flags): a "step" renders ONE full synthetic query image through the hot path (sample_depth -> coarse
pass -> fused resampling -> fine pass), encoder outputs given.  Workload `black_800` = the geometry BASELINE.json's metric
is quoted on: 800x800 query, 8 reference views 800x800 (feature maps 32ch @ 200x200), 64 coarse + 64 fine samples,
neuray_gen_depth cfg (coarse decoder use_vis:false), random-init weights, synthetic maps; one image per rank (weak scaling).

  value     ray-samples/s, whole job, inputs resident in HBM, device-timed (CUDA events, max over ranks)
  e2e       same metric through NeuralRayRenderPath.render() from pinned HOST buffers: every step copies all inputs
            host->device and the rendered tiles device->host inside the timed region
  roofline  the dominant kernel (point kernel): algorithmic FLOPs per launch / CUDA-event time, vs MEASURED_PEAKS.json
  cpu_baseline  the reference's own CPU implementation of the path on this box's host cores, bounded ray sample

Other BASELINE.json configurations (selectable as the main line with --workload, and measured as auxiliary objects
`aux.fern_high_sharded` / `aux.train_dtu` at every N of the default run so that the driver's 1/2/4/8 scaling runs carry them):
  fern_high  cfg4: ONE 1008x756 image, 10 reference views, 64+64, rays sharded over the ranks (dist.render_sharded, every
             output key gathered in one NCCL all-gather) = strong scaling; the collective is timed separately
  train_dtu  cfg5: one optimisation step per rank on 512 rays of a DTU-shape scene (8 views 304x400), native backward,
             flat-bucket gradient all-reduce (timed separately), Adam = weak scaling

--dump-outputs DIR writes what the headline's device-resident arm rendered in its last timed step (rank 0), one
DIR/<key>.npy per output key in float32 (float64 for integer keys), at most 64 MB in all: a larger output keeps the same
seeded sample of rays in every key (DIR/ray_index.npy).  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.

--impl reference times the UNMODIFIED reference's own implementation of the path (baseline/_ref, the verbatim copy made by
baseline/install_ref.py: NeuralRayBaseRenderer.render_impl over the chunk loop of renderer.py:237-254, encoder outputs
given) on the box's host cores; when the copy is absent it falls back to the oracle port and says so (`kind`).
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: dict(scene kwargs for synthetic.make_scene, rfn, dn coarse, dn fine, description)
    "black_800": dict(scene=dict(h=800, w=800), rfn=8, dn=(64, 64),
                      desc="nerf_synthetic/lego/black_800 geometry: 800x800 query, 8 ref views, 64+64 samples, neuray_gen_depth cfg"),
    "black_400": dict(scene=dict(h=400, w=400), rfn=8, dn=(64, 64),
                      desc="nerf_synthetic/lego/black_400 geometry: 400x400 query, 8 ref views, 64+64 samples, neuray_gen_depth cfg"),
    "cfg1": dict(scene=dict(h=64, w=64), rfn=3, dn=(32, 32), desc="64x64 query, 3 ref views, 32+32 samples"),
    "fern_high": dict(scene=dict(h=756, w=1008, depth_range=(1.2, 12.0), arc_deg=100.0, focal=0.83 * 1008), rfn=10, dn=(64, 64),
                      desc="llff_colmap/fern/high geometry: 1008x756 query, 10 ref views padded to 1008x768, 64+64 samples, depth (1.2,12)"),
    "train_dtu": dict(scene=dict(h=300, w=400, depth_range=(0.8, 4.0), radius=2.4), rfn=8, dn=(64, 64),
                      desc="DTU-train shape: 8 ref views 300x400 padded to 304x400, 512 rays per rank, 64+64 samples, training step"),
}
METRIC = "ray-samples/sec (800x800x64 coarse+64 fine, 8 ref views)"
TRAIN_RAYS = 512


def model_cfg(dn_c, dn_f):
    return {"use_hierarchical_sampling": True, "dist_decoder_cfg": {"use_vis": False}, "depth_sample_num": dn_c,
            "fine_depth_sample_num": dn_f, "agg_net_cfg": {"sample_num": dn_c}, "fine_agg_net_cfg": {"sample_num": dn_f},
            "render_depth": True, "ray_batch_num": 65536}


def make_workload(name, seed=0, with_que_imgs=False, **over):
    from neuray_b200 import synthetic
    wl = WORKLOADS[name]
    kw = dict(wl["scene"], rfn=wl["rfn"], seed=seed, smooth=2, with_que_imgs=with_que_imgs)
    kw.update(over)
    return synthetic.make_scene(**kw)


def point_kernel_flops_per_sample(rfn, use_vis_head):
    """Algorithmic FLOPs (2*MAC of the reference's Linear layers, no hoist credit) executed by the point kernel per
    ray-sample: SURVEY.md 8a -- per (point,view): dist decoder 12,608 (+4,160 with a vis head) + agg per-view 44,320;
    per point: geometry_fc 2*(65*64+64*16)."""
    return rfn * (12608 + (4160 if use_vis_head else 0) + 44320) + 2 * (65 * 64 + 64 * 16)


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons = index, False, [], set()
        self.max_mhz = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.1)
        except Exception as e:  # NVML missing: report that rather than fail the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


class Ctx:
    """Process-wide bench state: rank, device, timing helpers."""

    def __init__(self):
        import torch.distributed as dist
        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps, warmup):
        """W untimed calls, then exactly K calls bracketed by barrier + synchronize; seconds, max over ranks."""
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return ms.item() / 1e3

    def max_over_ranks(self, x):
        t = torch.tensor([float(x)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def build_net(cfg, dev, seed=0):
    from neuray_b200 import renderer, synthetic
    net = renderer.NeuralRayRenderPath(cfg)
    net.load_state_dict(synthetic.make_weights(cfg, seed=seed), strict=True)
    return net.to(dev)


class Uploader:
    """End-to-end arm: double-buffered uploads.  The inputs of step i+1 go up on a copy stream while step i runs (what a
    frame / batch loop does); every step still uploads all of its inputs inside the timed region."""

    def __init__(self, dev, host_dicts):
        self.dev, self.host = dev, host_dicts
        self.stream = torch.cuda.Stream(device=dev)
        self.pending = None
        self.bytes = sum(v.numel() * v.element_size() for d in host_dicts for v in d.values())

    def _upload(self):
        with torch.cuda.stream(self.stream):
            out = [{k: v.to(self.dev, non_blocking=True) for k, v in d.items()} for d in self.host]
            ev = torch.cuda.Event()
            ev.record(self.stream)
        return out, ev

    def next(self):
        out, ev = self.pending if self.pending is not None else self._upload()
        cur = torch.cuda.current_stream()
        cur.wait_event(ev)
        for d in out:
            for t in d.values():
                t.record_stream(cur)
        self.pending = self._upload()
        return out


def pin(d):
    return {k: v.pin_memory() for k, v in d.items()}


# ---- cfg4: one image, rays sharded over the ranks ---------------------------------------------------------------------------

def sharded_image(ctx, steps, warmup, e2e=True):
    """fern_high: ONE 1008x756 image, 10 views, 64+64; rank r renders its contiguous ray range, every output key is
    all-gathered (dist.render_sharded).  Strong scaling: total work fixed as N grows."""
    from neuray_b200 import dist as nrd
    wl = WORKLOADS["fern_high"]
    cfg = model_cfg(*wl["dn"])
    que, ref = make_workload("fern_high", seed=7)
    net = build_net(cfg, ctx.dev, seed=5)
    rays = que["coords"].shape[1]
    samples = rays * sum(wl["dn"])
    dq, dr = ({k: v.to(ctx.dev) for k, v in d.items()} for d in (que, ref))
    coll = []

    @torch.no_grad()
    def step(q=dq, r=dr):
        return nrd.render_sharded(lambda a, b, t: net.render(a, b, t), q, r, False, timing=coll)

    t = ctx.timed(step, steps, warmup)
    coll_ms = [a.elapsed_time(b) for a, b in coll[-steps:]] if coll else []
    # correctness of the sharded path, checked where it is measured (the driver's GPU test box has one GPU): every rank renders
    # the same 4096-ray stretch that straddles a shard boundary on its own and compares it with the gathered image, bit for bit
    identical = None
    if ctx.world > 1:
        full = step()
        lo = max(0, nrd.ray_range(rays, 1, ctx.world)[0] - 2048)
        q = dict(dq, coords=dq["coords"][:, lo:lo + 4096].contiguous())
        with torch.no_grad():
            local = net.render(q, dr, False)
        same = torch.tensor([float(all(torch.equal(local[k], full[k][:, lo:lo + 4096]) for k in local))], device=ctx.dev)
        ctx.dist.all_reduce(same, op=ctx.dist.ReduceOp.MIN)
        identical = bool(same.item())
    res = {"workload": wl["desc"], "value": samples * steps / t, "unit": "ray-samples/s", "ms_per_step": t / steps * 1e3,
           "scaling": "strong", "rays": rays, "n_gpus": ctx.world, "sharded_equals_single_gpu_bitwise": identical,
           "allgather_ms": ctx.max_over_ranks(sum(coll_ms) / len(coll_ms)) if coll_ms else 0.0,
           "allgather_bytes": int(-(-rays // ctx.world) * ctx.world * 4 * 8) if ctx.world > 1 else 0,
           "parallelism": f"rays of one image sharded over {ctx.world} rank(s); one NCCL all-gather of all output keys per frame"}
    if e2e:
        up = Uploader(ctx.dev, [pin(que), pin(ref)])
        host_out = {}

        def step_e2e():
            q, r = up.next()
            out = step(q, r)
            for k in ("pixel_colors_nr", "pixel_colors_nr_fine", "render_depth_fine", "ray_mask_fine"):
                if k not in host_out:
                    host_out[k] = torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory()
                host_out[k].copy_(out[k], non_blocking=True)
        t2 = ctx.timed(step_e2e, steps, warmup)
        res["e2e"] = {"value": samples * steps / t2, "unit": "ray-samples/s", "h2d_bytes_per_step": up.bytes,
                      "d2h_bytes_per_step": sum(v.numel() * v.element_size() for v in host_out.values()), "ms_per_step": t2 / steps * 1e3}
    return res


# ---- cfg5: data-parallel training step --------------------------------------------------------------------------------------

def train_step_bench(ctx, steps, warmup, e2e=True):
    """train_dtu: per rank one sampled batch of 512 rays x (64+64) samples on a DTU-shape scene (8 views 304x400): kernel
    forward (training mode: random fine quantiles, hit_prob kept) + render loss on both passes + native backward
    (nr_render_pass_bwd + nr_tape_gemms) + flat-bucket gradient all-reduce + Adam.  Weak scaling: 512 rays per rank."""
    from neuray_b200 import _lib, dist as nrd, synthetic
    wl = WORKLOADS["train_dtu"]
    cfg = dict(model_cfg(*wl["dn"]), fine_dist_decoder_cfg={"use_vis": True}, ray_batch_num=TRAIN_RAYS)
    que, ref = make_workload("train_dtu", seed=5, with_que_imgs=True)
    net = build_net(cfg, ctx.dev, seed=1)
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    dr = {k: v.to(ctx.dev) for k, v in ref.items()}
    gen = torch.Generator().manual_seed(100 + ctx.rank)          # distinct batches per rank
    n = que["coords"].shape[1]
    host_batches = []
    for _ in range(4):
        idx = torch.randperm(n, generator=gen)[:TRAIN_RAYS]
        host_batches.append(dict(que, coords=que["coords"][:, idx].contiguous()))
    batches = [synthetic.to_device(b, ctx.dev) for b in host_batches]
    coll = []
    state = {"i": 0, "loss": None}

    def step(batch=None):
        b = batch if batch is not None else batches[state["i"] % 4]
        state["i"] += 1
        out = net.render(b, dr, True)
        loss = ((out["pixel_colors_nr"] - out["pixel_colors_gt"]) ** 2).mean() + ((out["pixel_colors_nr_fine"] - out["pixel_colors_gt_fine"]) ** 2).mean()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        nrd.allreduce_gradients(net.parameters(), timing=coll)
        opt.step()
        state["loss"] = loss.detach()
        return loss

    l0 = _lib.LAUNCHES
    t = ctx.timed(step, steps, warmup)
    launches = (_lib.LAUNCHES - l0) // (steps + warmup)
    # after the all-reduce every rank must hold the same gradients (checked here because the driver's GPU test box has one GPU)
    grads_agree = None
    if ctx.world > 1:
        flat = torch.cat([p.grad.reshape(-1) for p in net.parameters() if p.grad is not None])
        ref_flat = flat.clone()
        ctx.dist.broadcast(ref_flat, 0)
        diff = (flat - ref_flat).abs().max().reshape(1)
        ctx.dist.all_reduce(diff, op=ctx.dist.ReduceOp.MAX)
        grads_agree = bool(diff.item() == 0.0)
    coll_ms = [a.elapsed_time(b) for a, b in coll[-steps:]] if coll else []
    samples = TRAIN_RAYS * sum(wl["dn"]) * ctx.world
    res = {"workload": wl["desc"], "value": samples * steps / t, "unit": "ray-samples/s", "ms_per_step": t / steps * 1e3, "scaling": "weak",
           "rays_per_rank": TRAIN_RAYS, "n_gpus": ctx.world, "kernels_per_step": launches, "gradients_identical_on_all_ranks": grads_agree,
           "allreduce_ms": ctx.max_over_ranks(sum(coll_ms) / len(coll_ms)) if coll_ms else 0.0,
           "allreduce_bytes": sum(p.numel() for p in net.parameters()) * 4 if ctx.world > 1 else 0,
           "loss": float(state["loss"]),
           "parallelism": f"data parallel x{ctx.world}: one 512-ray batch per rank, flat-bucket NCCL all-reduce of the gradients, Adam",
           "note": "device-timed over whole steps (host work included); forward + nr_render_pass_bwd + nr_tape_gemms + all-reduce + Adam"}
    if e2e:
        ups = Uploader(ctx.dev, [pin({"coords": b["coords"]}) for b in host_batches[:1]])
        host_loss = torch.empty(1).pin_memory()

        def step_e2e():
            (c,) = ups.next()                    # the sampled ray coordinates of this step come from the host (the data loader's part)
            loss = step(dict(batches[0], coords=c["coords"]))
            host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
        t2 = ctx.timed(step_e2e, steps, warmup)
        res["e2e"] = {"value": samples * steps / t2, "unit": "ray-samples/s", "h2d_bytes_per_step": ups.bytes, "d2h_bytes_per_step": 4,
                      "ms_per_step": t2 / steps * 1e3}
    return res


# ---- reference arm / CPU baselines ------------------------------------------------------------------------------------------

def _load_reference():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_import
    if not ref_import.available():
        return None
    return ref_import.load_reference()


def reference_net(ref_mod, cfg, seed=0, device="cpu"):
    from neuray_b200 import synthetic
    net = ref_mod.NeuralRayBaseRenderer(cfg)
    missing, unexpected = net.load_state_dict(synthetic.make_weights(cfg, seed=seed), strict=False)
    assert not unexpected
    net = net.eval().to(device)
    for m in net.modules():        # the reference pins this plain attribute to "cuda:0" (ibrnet.py:312); put it where the net runs
        if hasattr(m, "pos_encoding") and torch.is_tensor(m.pos_encoding):
            m.pos_encoding = m.pos_encoding.to(device)
    return net


def reference_render_chunks(net, que, ref, ray_batch_num):
    """The chunk loop of the reference's render() (renderer.py:237-254) with the encoders' outputs given: its own
    render_impl per chunk, hit_prob keys dropped, chunks concatenated."""
    coords = que["coords"]
    acc = {}
    for s in range(0, coords.shape[1], ray_batch_num):
        q = dict(que, coords=coords[:, s:s + ray_batch_num])
        for k, v in net.render_impl(q, dict(ref), False).items():
            if not k.startswith("hit_prob"):
                acc.setdefault(k, []).append(v)
    return {k: torch.cat(v, 1) for k, v in acc.items()}


def cpu_arm(wl_name, n_rays, steps, warmup, threads=None):
    """ray-samples/s of the reference's CPU implementation on `n_rays` rays of the workload (same maps, same weights).
    Returns (value, seconds per pass, kind, threads).  kind = "reference" (baseline/_ref) or "port" (oracle)."""
    from neuray_b200 import synthetic, renderer
    wl = WORKLOADS[wl_name]
    dn_c, dn_f = wl["dn"]
    cfg = model_cfg(dn_c, dn_f)
    que, ref = make_workload(wl_name, seed=0)
    w = que["coords"][0, :, 0].max().int().item() + 1
    total = que["coords"].shape[1]
    start = (total // 2 // w) * w + w // 4         # a stretch of rays through the middle of the image
    q = synthetic.slice_rays(que, start, start + n_rays)
    ref_mod = _load_reference()
    if ref_mod is not None:
        net = reference_net(ref_mod, cfg)
        run = lambda: reference_render_chunks(net, q, ref, 4096)
        kind = "reference"
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import neuray_oracle as orc
        from gen_golden import flat_cfg
        W = synthetic.make_weights(cfg, seed=0)
        ocfg = flat_cfg({**renderer.base_cfg, **cfg})
        run = lambda: orc.render(W, ocfg, q, ref, False, ray_batch_num=4096)
        kind = "port"
    cores = os.cpu_count() or 1
    with torch.no_grad():
        if threads is None:
            # "all the host threads it can use": torch's intra-op pool stops scaling long before 128 threads on this op mix
            # of many small tensors (round 1: 8 -> 61 k, 16 -> 67 k, 32 -> 63 k, 64 -> 22 k, 128 -> 1.6 k ray-samples/s), so the
            # arm picks the best of a short scan on a 128-ray probe and reports the count it used
            probe = synthetic.slice_rays(que, start, start + min(128, n_rays))
            best = (None, 0.0)
            for th in [t for t in (8, 16, 32, 64) if t <= cores] or [cores]:
                torch.set_num_threads(th)
                fn = (lambda: reference_render_chunks(net, probe, ref, 4096)) if kind == "reference" else (lambda: orc.render(W, ocfg, probe, ref, False, ray_batch_num=4096))
                fn()
                t0 = time.perf_counter()
                fn()
                rate = 1.0 / (time.perf_counter() - t0)
                if rate > best[1]:
                    best = (th, rate)
            threads = best[0]
        torch.set_num_threads(threads)
        times = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            run()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    return n_rays * (dn_c + dn_f) / t, t, kind, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    dn_c, dn_f = wl["dn"]
    n_rays = args.ref_rays
    v, t, kind, threads = cpu_arm(args.workload, n_rays, args.steps, max(1, min(args.warmup, 1)))
    sample = f"{n_rays} rays x ({dn_c}+{dn_f}) samples of the workload per step (a contiguous stretch of image rows)"
    what = ("the UNMODIFIED reference (baseline/_ref): NeuralRayBaseRenderer.render_impl over render()'s chunk loop, encoder outputs given"
            if kind == "reference" else "oracle port of the reference's PyTorch path (baseline/_ref missing)")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "ray-samples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "rays_per_step": n_rays, "note": what + ", host cores"},
        "cpu_baseline": {"value": v, "unit": "ray-samples/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "ray-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def eager_gpu_baseline(dq, dr, cfg, dn, dev, rays=4096, reps=3):
    """GPU-vs-GPU baseline (SURVEY.md 8d): the UNMODIFIED reference's own render_impl (coarse + fine pass) as PyTorch-eager
    CUDA ops on the same B200, on one 4096-ray chunk (render.py's default chunk) of the same workload and weights."""
    ref_mod = _load_reference()
    if ref_mod is None:
        return {"unavailable": "baseline/_ref missing (run baseline/install_ref.py before gpurun)"}
    net = reference_net(ref_mod, cfg, device=dev)
    n = dq["coords"].shape[1]
    start = max(0, n // 2 - rays // 2)                 # a stretch of rays through the middle of the image
    q = dict(dq, coords=dq["coords"][:, start:start + rays].contiguous())
    r = {k: v for k, v in dr.items() if torch.is_tensor(v)}

    def run():
        with torch.no_grad():
            return net.render_impl(q, dict(r), False)

    run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return {"value": rays * 2 * dn / ms * 1e3, "unit": "ray-samples/s", "ms_per_chunk": ms, "rays": rays, "samples_per_ray": 2 * dn,
            "kind": "reference", "what": "the unmodified reference's render_impl (coarse + fine) as PyTorch-eager CUDA ops on the same GPU, one 4096-ray chunk"}


def encoder_flops(h, w):
    """Algorithmic FLOP (2 x MAC, convolutions only) of image_encoder + vis_encoder for one h x w view
    (ResUNetLight(3,[1,2,6,4],32,inplanes=16), ops.py:150-230; DefaultVisEncoder, vis_encoder.py:6-21)."""
    c = lambda n: (n - 1) // 2 + 1
    h0, w0 = c(h), c(w); h1, w1 = c(h0), c(w0); h2, w2 = c(h1), c(w1); h3, w3 = c(h2), c(w2)
    u3, u2 = (2 * h3) * (2 * w3), (4 * h3) * (4 * w3)
    mac = h0 * w0 * 16 * 147
    mac += h1 * w1 * (32 * 16 * 9 + 32 * 32 * 9 + 32 * 16)
    mac += h2 * w2 * (64 * 32 * 9 + 64 * 64 * 9 + 64 * 32 + 2 * 64 * 64 * 9)
    mac += h3 * w3 * (128 * 64 * 9 + 128 * 128 * 9 + 128 * 64 + 10 * 128 * 128 * 9)
    mac += u3 * 2 * 64 * 128 * 9 + u2 * (2 * 32 * 64 * 9 + 32 * 32)
    mac += u2 * (32 * 64 * 9 + 4 * 32 * 32 * 9 + 32 * 32)
    return 2 * mac


def encoders_bench(dr, dev, reps=5):
    """Auxiliary (SURVEY.md 8f row 1): the per-frame encoders of the headline workload's reference views -- native
    (nr_image_encoder_fwd + nr_vis_encoder_fwd writing the frame pack in place) against the UNMODIFIED reference modules as
    PyTorch / cuDNN ops on the same GPU, same random-init parameters, same inputs."""
    import types
    from neuray_b200 import encoders
    imgs, ray_in = dr["imgs"], dr["ray_feats"]
    rfn, _, h, w = imgs.shape
    fh, fw = encoders.image_dims(h, w)
    torch.manual_seed(0)
    owner = types.SimpleNamespace(image_encoder=encoders.ImageEncoder().to(dev), vis_encoder=encoders.VisEncoder().to(dev))
    feat = torch.empty(rfn, fh, fw, 64, device=dev)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    info = {"imgs": imgs, "ray_feats": ray_in}
    with torch.no_grad():
        ms = timed(lambda: encoders.encode_frame(owner, dict(info), feat))
        feat32 = feat.clone()
        encoders.set_precision("tf32")
        try:
            ms_tf32x1 = timed(lambda: encoders.encode_frame(owner, dict(info), feat))
            tf32_diff = float((feat - feat32).abs().max())
        finally:
            encoders.set_precision("fp32")
        encoders.encode_frame(owner, dict(info), feat)
    fl = encoder_flops(h, w) * rfn
    res = {"ms_per_frame": ms, "views": rfn, "image": [h, w], "algorithmic_tflops": fl / ms / 1e9, "flop_per_frame": fl,
           "kernels_per_frame": encoders.IMAGE_LAUNCHES + encoders.VIS_LAUNCHES + 3,
           "single_pass_tf32": {"ms_per_frame": ms_tf32x1, "algorithmic_tflops": fl / ms_tf32x1 / 1e9, "max_abs_diff_to_fp32_mode": tf32_diff,
                                "what": "encoders.set_precision('tf32'): one TF32 pass per product, the arithmetic of cuDNN under torch's default allow_tf32"},
           "what": "image_encoder + vis_encoder of all reference views into the channel-last frame pack (3xTF32 tensor-core convolutions: fp32 accuracy)"}
    ref_mod = _load_reference()
    if ref_mod is None:
        res["reference"] = {"unavailable": "baseline/_ref missing"}
        return res
    from network.ops import ResUNetLight
    from network.vis_encoder import DefaultVisEncoder
    ie, ve = ResUNetLight(3, [1, 2, 6, 4], 32, inplanes=16).to(dev).eval(), DefaultVisEncoder({}).to(dev).eval()
    ie.load_state_dict(owner.image_encoder.state_dict(), strict=True)
    ve.load_state_dict(owner.vis_encoder.state_dict(), strict=True)

    def ref_run():
        f = ie(imgs)
        return f, ve(ray_in, f)

    old = torch.backends.cudnn.allow_tf32
    with torch.no_grad():
        ms_tf32 = timed(ref_run)                       # torch default: cuDNN may use TF32 for fp32 convolutions
        torch.backends.cudnn.allow_tf32 = False
        ms_fp32 = timed(ref_run)
        f_img, f_ray = ref_run()
        torch.backends.cudnn.allow_tf32 = old
    res["reference"] = {"ms_per_frame_cudnn_default_tf32": ms_tf32, "ms_per_frame_cudnn_fp32": ms_fp32, "kind": "reference",
                        "max_abs_diff_img_feats": float((feat[..., 32:].permute(0, 3, 1, 2) - f_img).abs().max()),
                        "max_abs_diff_ray_feats": float((feat[..., :32].permute(0, 3, 1, 2) - f_ray).abs().max()),
                        "what": "the unmodified reference's ResUNetLight + DefaultVisEncoder (PyTorch eager / cuDNN) on the same GPU"}
    try:
        res["depth_init_net"] = init_net_bench(dr, dev, reps, timed)
    except Exception as e:
        res["depth_init_net"] = {"error": f"{type(e).__name__}: {e}"}
    try:
        res["cost_volume_init_net"] = cost_volume_bench(dr, dev, max(2, reps // 2), timed)
    except Exception as e:
        res["cost_volume_init_net"] = {"error": f"{type(e).__name__}: {e}"}
    return res


def cost_volume_bench(dr, dev, reps, timed):
    """CostVolumeInitNet of the same frame (init_net.py:205-254: MVSNet cost volumes of the 8 reference views from 3 neighbouring
    source views each, 64 depth planes, evaluation resize 800 -> 640; ResUNetLight + the three conv heads), native against the
    unmodified reference module (its frozen mvsnet_pl.ckpt weights in both) on the same GPU."""
    from neuray_b200 import init_nets
    imgs = dr["imgs"]
    rfn, _, h, w = imgs.shape
    nn_ids = torch.stack([torch.tensor([(i + 1) % rfn, (i + 2) % rfn, (i + 3) % rfn]) for i in range(rfn)]).to(dev)
    ref = {"imgs": imgs, "depth_range": dr["depth_range"], "poses": dr["poses"], "Ks": dr["Ks"], "nn_ids": nn_ids}
    src = {"imgs": imgs, "poses": dr["poses"], "Ks": dr["Ks"]}          # the reference views double as each other's source views
    torch.manual_seed(0)
    net = init_nets.CostVolumeInitNet().to(dev).eval()
    ref_mod = _load_reference()
    rnet = None
    if ref_mod is not None:
        import network.init_net as ref_init
        import ref_import
        cwd = os.getcwd()
        os.chdir(ref_import.REFERENCE_ROOT)
        try:
            rnet = ref_init.CostVolumeInitNet({}).to(dev).eval()          # loads network/mvsnet/mvsnet_pl.ckpt
        finally:
            os.chdir(cwd)
        sd = {k: v for k, v in rnet.state_dict().items()}
        net.load_state_dict(sd, strict=False)                            # same weights in both (the head is random-init)
    fh, fw = h // 4, w // 4
    buf = torch.empty(rfn, fh, fw, 64, device=dev)
    with torch.no_grad():
        ms = timed(lambda: init_nets.cost_volume_forward_into(net, ref, src, False, buf, 0))
        ms_mvs = timed(lambda: init_nets.mvsnet_cost_volume(net, ref, src, False))
    out = {"ms_per_frame": ms, "ms_mvsnet_part": ms_mvs, "views": rfn, "neighbours": 3, "depth_planes": 64,
           "what": "nr_mvsnet_fwd (FeatureNet on 16 images at 640x640, 8 variance volumes 64x160x160x32, CostRegNet, softmax + regression) + "
                   "nr_extract_depth + nr_cost_volume_head_fwd into the frame pack"}
    if rnet is None:
        return out
    with torch.no_grad():
        ms_ref = timed(lambda: rnet(dict(ref), dict(src), False))
        want = rnet(dict(ref), dict(src), False)
    err = (buf[..., :32].permute(0, 3, 1, 2) - want).abs()
    out["reference"] = {"ms_per_frame": ms_ref, "kind": "reference", "max_abs_diff": float(err.max()), "mean_abs_diff": float(err.mean()),
                        "output_abs_max": float(want.abs().max()),
                        "what": "the unmodified reference's CostVolumeInitNet (PyTorch eager / cuDNN, torch's default TF32 convolutions) on the same GPU"}
    return out


def init_net_bench(dr, dev, reps, timed):
    """DepthInitNet of the same frame (init_net.py:63-101: extract_depth + get_diff_feats + ResEncoder + depth_skip + conv_out),
    native against the unmodified reference module on the same GPU; the depth maps are synthetic smooth fields inside the range."""
    from neuray_b200 import init_nets
    imgs = dr["imgs"]
    rfn, _, h, w = imgs.shape
    g = torch.Generator(device="cpu").manual_seed(4)
    rng = dr["depth_range"]
    base = torch.rand(rfn, 1, h // 16, w // 16, generator=g).to(dev)
    depth = rng[:, 0].view(-1, 1, 1, 1) + (rng[:, 1] - rng[:, 0]).view(-1, 1, 1, 1) * (0.15 + 0.7 * torch.nn.functional.interpolate(base, size=(h, w), mode="bilinear", align_corners=True))
    ref = {"imgs": imgs, "depth": depth, "depth_range": rng, "poses": dr["poses"], "Ks": dr["Ks"]}
    torch.manual_seed(0)
    net = init_nets.DepthInitNet().to(dev)
    fh, fw = init_nets.dims(h, w)
    buf = torch.empty(rfn, fh, fw, 64, device=dev)
    with torch.no_grad():
        ms = timed(lambda: init_nets.forward_into(net, ref, buf, 0))
    out = {"ms_per_frame": ms, "what": "nr_extract_depth + nr_diff_feats + nr_depth_init_fwd (ResEncoder on the tensor cores, fp32 accuracy) into the frame pack"}
    ref_mod = _load_reference()
    if ref_mod is None:
        return out
    import network.init_net as ref_init
    rnet = ref_init.DepthInitNet({}).to(dev).eval()
    rnet.load_state_dict(net.state_dict(), strict=True)
    old = torch.backends.cudnn.allow_tf32
    with torch.no_grad():
        ms_tf32 = timed(lambda: rnet(dict(ref), None, False))
        torch.backends.cudnn.allow_tf32 = False
        ms_fp32 = timed(lambda: rnet(dict(ref), None, False))
        want = rnet(dict(ref), None, False)
        torch.backends.cudnn.allow_tf32 = old
    err = (buf[..., :32].permute(0, 3, 1, 2) - want).abs()
    out["reference"] = {"ms_per_frame_cudnn_default_tf32": ms_tf32, "ms_per_frame_cudnn_fp32": ms_fp32, "kind": "reference",
                        "max_abs_diff": float(err.max()), "frac_above_1e-3": float((err > 1e-3).float().mean()),
                        "what": "the unmodified reference's DepthInitNet (PyTorch eager: get_diff_feats as torch ops + cuDNN) on the same GPU"}
    return out


# ---- headline -----------------------------------------------------------------------------------------------------------------

DUMP_BYTES = 64 << 20


def dump_outputs(out, rays, path):
    """Writes a render's output dict as path/<key>.npy (float32; float64 for integer keys).  Keys are [1, rays, ...]; when
    they come to more than DUMP_BYTES, every key keeps the same rays, a sorted sample drawn with a fixed seed."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    per_ray = sum(v[0, 0].numel() * (8 if v.dtype in (torch.int32, torch.int64) else 4) for v in out.values())
    idx = None
    if per_ray * rays > DUMP_BYTES:
        keep = DUMP_BYTES // per_ray
        idx = torch.randperm(rays, generator=torch.Generator().manual_seed(0))[:keep].sort()[0]
        np.save(os.path.join(path, "ray_index.npy"), idx.numpy().astype(np.float64))
    for k, v in out.items():
        assert v.shape[:2] == (1, rays), (k, tuple(v.shape))
        v = v.detach()[:, idx.to(v.device)] if idx is not None else v.detach()
        v = v.cpu().numpy()
        np.save(os.path.join(path, k + ".npy"), v.astype(np.float64 if v.dtype.kind in "iu" else np.float32))


def run_headline(ctx, args):
    from neuray_b200 import _lib
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    wl = WORKLOADS[args.workload]
    rfn, (dn_c, dn_f) = wl["rfn"], wl["dn"]
    cfg = model_cfg(dn_c, dn_f)
    cfg["ray_batch_num"] = args.ray_batch
    # one image per rank: same reference views, a different query pose per rank (seeded)
    que, ref = make_workload(args.workload, seed=0)
    if rank > 0:
        q2, _ = make_workload(args.workload, seed=0, arc_deg=wl["scene"].get("arc_deg", 60.0) + 3.0 * rank)
        que["poses"] = q2["poses"]
    net = build_net(cfg, dev, seed=0)
    rays = que["coords"].shape[1]
    samples_per_step = rays * (dn_c + dn_f)
    out_keys = ("pixel_colors_nr", "pixel_colors_nr_fine", "render_depth_fine", "ray_mask_fine")
    host_out = {}
    gathered = [torch.empty(1, rays, 3, device=dev) for _ in range(world)] if world > 1 else None

    @torch.no_grad()                      # inference, like the reference's render.py (renderer(data) under torch.no_grad())
    def step_device(dq, dr):
        out = net.render(dq, dr, False)
        if world > 1:   # the rendered tiles of all ranks are gathered (north_star: all-gather of the final tiles)
            ctx.dist.all_gather(gathered, out["pixel_colors_nr_fine"])
        return out

    up = Uploader(dev, [pin(que), pin(ref)])

    def step_e2e():
        dq, dr = up.next()
        out = step_device(dq, dr)
        for k in out_keys:
            if k not in host_out:
                host_out[k] = torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory()
            host_out[k].copy_(out[k], non_blocking=True)
        return out

    # ---- device-resident arm (value) with per-kernel event timing of the two kernels of a pass ----
    dq = {k: v.to(dev) for k, v in que.items()}
    dr = {k: v.to(dev) for k, v in ref.items()}
    last = {}

    def step_resident():                  # the per-frame map repack runs inside every render() call
        last["out"] = step_device(dict(dq), dr)

    sampler = ClockSampler(ctx.local)
    for _ in range(args.warmup):
        step_resident()
    ctx.barrier()
    _lib.PROFILE = []
    l0 = _lib.LAUNCHES
    sampler.start()
    t_res = ctx.timed(step_resident, args.steps, 0)
    sampler.stop_flag = True
    launches = _lib.LAUNCHES - l0
    prof, _lib.PROFILE = _lib.PROFILE, None
    pk_ms = [a.elapsed_time(b) for a, b, *_ in prof]
    rk_ms = [b.elapsed_time(c) for _, b, _, c in prof]
    pk_samples = [n for _, _, n, _ in prof]
    value = world * samples_per_step * args.steps / t_res

    # ---- end-to-end arm ----
    t_e2e = ctx.timed(step_e2e, args.steps, args.warmup)
    d2h = sum(v.numel() * v.element_size() for v in host_out.values())
    e2e_value = world * samples_per_step * args.steps / t_e2e

    # ---- the other BASELINE configurations, measured at this N too (auxiliary; a failure cannot cost the headline) ----
    aux = {}
    if not args.no_aux:
        del up
        torch.cuda.empty_cache()
        for name, fn in (("fern_high_sharded", lambda: sharded_image(ctx, 3, 2, e2e=False)), ("train_dtu", lambda: train_step_bench(ctx, 20, 5, e2e=False))):
            ok = torch.ones(1, device=dev)
            try:
                res = fn()
            except Exception as e:      # keep the ranks in lock step: if any rank failed, all drop this leg
                res = {"error": f"{type(e).__name__}: {e}"}
                ok.zero_()
            if world > 1:
                ctx.dist.all_reduce(ok, op=ctx.dist.ReduceOp.MIN)
            aux[name] = res if ok.item() > 0 or "error" in res else {"error": "failed on another rank"}
            torch.cuda.empty_cache()

    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(last["out"], rays, args.dump_outputs)

    peaks, peaks_src = {}, "fallback"
    pth = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pth):
        peaks = json.load(open(pth))
        peaks_src = "measured"
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)      # kernel timed inside a long step -> sustained figure
    peak_hbm = peaks.get("hbm_gbs", 6650.0)
    fl = point_kernel_flops_per_sample(rfn, False)
    pk_time = sum(pk_ms) / 1e3
    achieved_tf = sum(pk_samples) * fl / pk_time / 1e12
    gather_gbs = sum(pk_samples) * rfn * 1072 / pk_time / 1e9
    n_launch = len(pk_ms)

    cpu = None
    if not args.no_cpu_baseline and world == 1:      # rank 0 at N=1 only (torchrun pins OMP_NUM_THREADS=1)
        v, t, kind, threads = cpu_arm(args.workload, args.cpu_rays, 1, 1)
        cpu = {"value": v, "unit": "ray-samples/s", "cores": threads, "kind": kind,
               "sample": f"{args.cpu_rays} rays x ({dn_c}+{dn_f}) samples of the same workload, 1 warm-up + 1 timed pass, {t:.1f} s"}

    # DRAM bytes of one point-kernel launch: from the ncu --set full capture of this kernel at this launch size, kept next
    # to the other profile summaries (profiles/point_kernel_traffic.json: {"<workload>/<ray_batch>": {...}}); null when no
    # capture of this exact launch shape has been committed
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "point_kernel_traffic.json")
    if os.path.exists(tp):
        ent = json.load(open(tp)).get(f"{args.workload}/{args.ray_batch}")
        if ent:
            traffic, traffic_src = ent["dram_bytes_read"] + ent["dram_bytes_write"], ent.get("source")
    line = {
        "metric": METRIC, "value": value, "unit": "ray-samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_res / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "rays_per_image": rays, "images_per_step_per_gpu": 1, "ray_batch_num": args.ray_batch,
                   "parallelism": f"one image per rank x{world}" + (", NCCL all-gather of rendered tiles" if world > 1 else ""),
                   "e2e_pipeline": "inputs of step i+1 are uploaded on a copy stream while step i renders",
                   "l2": "inputs (143 MB of maps at black_800) exceed the 126 MB L2; no explicit flush"},
        "per_gpu": value / world,
        "e2e": {"value": e2e_value, "unit": "ray-samples/s", "h2d_bytes_per_step": up_bytes(que, ref), "d2h_bytes_per_step": d2h,
                "ms_per_step": t_e2e / args.steps * 1e3},
        "gpu_launches": launches,
        "clocks": sampler.summary(),
        "roofline": {"bound": "tensor", "kernel": "nr::pkt::pm3::point_kernel_pm3", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": achieved_tf / peak_tf, "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu --set full)",
                     "traffic_source": traffic_src, "peak_source": f"{peaks_src} bf16_tflops_sustained",
                     "flops_per_ray_sample": fl, "launches": n_launch, "avg_launch_ms": sum(pk_ms) / max(n_launch, 1),
                     "share_of_step": pk_time / t_res, "ray_kernel_share_of_step": sum(rk_ms) / 1e3 / t_res,
                     "note": "dense layers on tcgen05 with 3xTF32 (3 MMAs per algorithmic one)"},
        "roofline_gather": {"bound": "hbm", "achieved": gather_gbs, "peak": peak_hbm, "unit": "GB/s", "frac": gather_gbs / peak_hbm,
                            "bytes_per_ray_sample": rfn * 1072,
                            "note": "gather runs inside the point kernel; algorithmic bytes / point-kernel time"},
        "cpu_baseline": cpu,
        "aux": aux,
    }
    if world == 1 and not args.no_aux:
        try:          # auxiliary: never let it cost the headline line
            line["eager_gpu_baseline"] = eager_gpu_baseline(dq, dr, cfg, dn_c, dev)
        except Exception as e:
            line["eager_gpu_baseline"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            torch.cuda.empty_cache()
            enc = encoders_bench(dr, dev)
            # SURVEY.md 8d: the metric is quoted on render() with the encoder outputs given; the same frame INCLUDING both
            # encoders (they run once per frame, before the chunk loop) for the "with encoders" figure
            frame_ms = t_res / args.steps * 1e3
            enc["frame_with_encoders"] = {"ms_per_frame": frame_ms + enc["ms_per_frame"], "unit": "ray-samples/s",
                                          "value": samples_per_step / (frame_ms + enc["ms_per_frame"]) * 1e3,
                                          "what": "headline step (render, encoder outputs given) + native encoders of the 8 reference views"}
            cvn = enc.get("cost_volume_init_net", {}).get("ms_per_frame")
            if cvn is not None:
                tot = frame_ms + enc["ms_per_frame"] + cvn
                enc["frame_gen_cost_volume"] = {"ms_per_frame": tot, "unit": "ray-samples/s", "value": samples_per_step / tot * 1e3,
                                                "what": "headline step + native encoders + native CostVolumeInitNet (MVSNet included)"}
            di = enc.get("depth_init_net", {}).get("ms_per_frame")
            if di is not None:      # the whole per-frame path of the gen_depth model in inference: init net -> encoders -> render
                tot = frame_ms + enc["ms_per_frame"] + di
                enc["frame_gen_depth"] = {"ms_per_frame": tot, "unit": "ray-samples/s", "value": samples_per_step / tot * 1e3,
                                          "what": "headline step + native encoders + native DepthInitNet (sum of the three device-timed stages)"}
            line["aux"]["encoders"] = enc
        except Exception as e:
            line["aux"]["encoders"] = {"error": f"{type(e).__name__}: {e}"}
    print(json.dumps(line))


def up_bytes(que, ref):
    return sum(v.numel() * v.element_size() for d in (que, ref) for v in d.values())


def run_aux_as_main(ctx, args):
    """--workload fern_high / train_dtu as the main line (same schema)."""
    sampler = ClockSampler(ctx.local)
    sampler.start()
    res = sharded_image(ctx, args.steps, args.warmup) if args.workload == "fern_high" else train_step_bench(ctx, args.steps, args.warmup)
    sampler.stop_flag = True
    if ctx.rank != 0:
        return
    coll = {k: res[k] for k in ("allgather_ms", "allgather_bytes", "allreduce_ms", "allreduce_bytes", "kernels_per_step", "loss") if k in res}
    line = {"metric": "ray-samples/sec", "value": res["value"], "unit": "ray-samples/s", "n_gpus": ctx.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": res["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": res["workload"], "parallelism": res["parallelism"]},
            "e2e": res.get("e2e"), "collective": coll, "clocks": sampler.summary(), "gpu_launches": None}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="black_800", choices=sorted(WORKLOADS))
    ap.add_argument("--shard", default=None, choices=["images", "rays"], help="fern_high is always ray-sharded; accepted for explicitness")
    ap.add_argument("--ray-batch", type=int, default=65536)
    ap.add_argument("--cpu-rays", type=int, default=512, help="rays of the workload timed on the CPU arm (cpu_baseline)")
    ap.add_argument("--ref-rays", type=int, default=512, help="rays per step for --impl reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true", help="skip the auxiliary legs (fern_high sharded, train_dtu, eager GPU baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's outputs of its last timed step as DIR/<key>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload in ("fern_high", "train_dtu")):
        ap.error("--dump-outputs writes the headline's outputs: --impl b200 with black_800, black_400 or cfg1")
    if args.impl == "reference":
        if args.workload in ("fern_high", "train_dtu"):
            args.workload = "fern_high" if args.workload == "fern_high" else "black_800"
        run_reference(args)
        return
    ctx = Ctx()
    try:
        if args.workload in ("fern_high", "train_dtu"):
            run_aux_as_main(ctx, args)
        else:
            run_headline(ctx, args)
    finally:
        ctx.close()


if __name__ == "__main__":
    main()
