#!/usr/bin/env python
"""bench.py -- rays/sec of the layered ray-march hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--precision exact|exact_cf|mixed|fp32|fast]
                    [--workload taekwondo2|walking4|walking6_4k] [--no-extra] [--no-cpu-baseline] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): taekwondo 2-layer scene, 1080p, 16 views, 64 coarse + 128 fine samples.
A *step* renders one 1080p view (2 073 600 rays; view = step mod 16) through the whole hot path: ray generation ->
bbox-clipped sampling -> MotionNet/SpaceNet MLPs -> compositing + resampling -> fine MLPs -> per-layer + merged compositing
of every image (coarse AND fine, i.e. everything `LayeredRFRender.forward` returns).  Scene geometry and cameras are
synthetic (SURVEY 8d: the dataset is not shipped); weights are the shipped taekwondo checkpoint when its copy is present
under oracle/_ref/ckpt, else seeded random weights of the same architecture (the cost of the path does not depend on weight
values).

value  = device-resident throughput: cameras/rays already on the device, CUDA events around the K steps, max over ranks.
         N ranks: each view's rows are interleaved over the ranks, every rank's compositing kernel writes its pixels straight
         into its slot of a persistent all-gather buffer and ONE in-place all-gather per view assembles the fine images on
         every rank (strong scaling: total work per step is fixed).
e2e    = same metric through the host-buffer C-ABI call (stnerf_render_host): pinned host rays -> H2D (chunk-pipelined) ->
         render -> D2H of every image plane (chunk-pipelined), inside the timed region, same K steps.
--impl reference : the UNMODIFIED reference (`LayeredRFRender.forward`, run out of process from the archive packed by
         oracle/stash_reference.py) on the host cores, on a bounded sample of the same workload per step; rank 0 only.
         Falls back to the oracle port (kind "port") only if no reference archive / checkout is available.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "st-nerf_b200"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

FLOP_SPACE_NOTIME, FLOP_SPACE_TIME, FLOP_MOTION = 924672.0, 930048.0, 153344.0   # SURVEY 8(d), 2*MAC per point

# BASELINE.json configs.  The headline line is always configs[1]; the others are timed briefly as `extra_workloads`.
WORKLOADS = {
    "taekwondo2": dict(H=1080, W=1920, views=16, n1=64, n2=128, layers=2, ckpt="taekwondo", space_time=True, thr=(0.0, 0.0), near=0.0,
                       frame_ids=[0.0, 10.0, 11.0], fixture="scale_tkd2_16k",                       # demo/taekwondo_demo.py:44
                       name="taekwondo 2-layer 1080p, 16 views, 64+128 samples (BASELINE configs[1])"),
    # configs[2]: walking nets replicated round-robin to 4 performers (SURVEY 8d), demo/walking_demo.py:43-50 thresholds
    "walking4": dict(H=1080, W=1920, views=16, n1=64, n2=128, layers=4, ckpt="walking", space_time=False, thr=(20.0, 0.8), near=4.0,
                     frame_ids=[0.0, 30.0, 31.0, 32.0, 33.0], fixture="scale_walk4_16k",
                     name="walking 4-layer 1080p, 16 views, 64+128 samples (BASELINE configs[2])"),
    # configs[4]: 6 performers, 4K, 32 views, 64+192
    "walking6_4k": dict(H=2160, W=3840, views=32, n1=64, n2=192, layers=6, ckpt="walking", space_time=False, thr=(20.0, 0.8), near=4.0,
                        frame_ids=[0.0, 30.0, 31.0, 32.0, 33.0, 34.0, 35.0], fixture="scale_walk6_4k",
                        name="walking 6-layer 4K, 32 views, 64+192 samples (BASELINE configs[4])"),
}
PRECISION_TERMS = {"exact": 3.0, "exact_cf": 3.0, "mixed": 3.0 - 2.0 * (256 * 128) / 462336.0, "fast": 1.0, "fp32": 1.0}
DTYPES = {"exact": "f32 via fp16x3 split products (tcgen05), f32 accumulate", "fp32": "f32",
          "exact_cf": "f32 via fp16x3 split products (tcgen05), correction products first in the coarse pass and the MotionNets, f32 accumulate", "fast": "f16 products, f32 accumulate",
          "mixed": "f32 via fp16x3 split products on everything the density depends on, single f16 pass on the colour-only layer "
                   "rgb_net.1 (tcgen05), f32 accumulate"}


def load_weights(wl):
    import torch
    from stnerf_b200 import checkpoint_io
    p = checkpoint_io.find_checkpoint(wl["ckpt"])
    if p is not None:
        sd = checkpoint_io.replicate_layers(torch.load(p, map_location="cpu")["model"], wl["layers"])
        return sd, "%s checkpoint (oracle/_ref/ckpt)%s" % (
            wl["ckpt"], ", nets replicated round-robin to %d performers" % wl["layers"] if wl["layers"] > 2 else "")
    from stnerf_b200 import synthetic
    return synthetic.synthetic_state_dict(wl["layers"], wl["space_time"], seed=7), "seeded random weights (checkpoint copy absent)"


def scene_setup(wl):
    from stnerf_b200 import synthetic              # synthetic scene description (inputs only)
    bkgd, frames = synthetic.synthetic_boxes(wl["layers"])
    cams = [synthetic.synthetic_camera(v, wl["views"], wl["H"], wl["W"]) for v in range(wl["views"])]
    return bkgd, frames, cams


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 9 for i in range(4) if r[5 + i].lower() == "active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_median": statistics.median(pw) if pw else None, "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference itself (kind "reference"), out of process; the oracle port only as a fallback
# ---------------------------------------------------------------------------------------------------------------------
def cpu_sample(wl, cams, step, per_band):
    """Rays of one step's bounded sample: 4 row bands of the step's view (representative layer hit fractions, BASELINE.md 3)."""
    import torch
    from oracle import stnerf_oracle as O          # ray generation for the CPU arm only (test infrastructure)
    H, W = wl["H"], wl["W"]
    K, T = cams[step % wl["views"]]
    full = O.generate_rays(K, T, H, W)
    idx = torch.cat([torch.arange(per_band) + (H * (2 * q + 1) // 8) * W + (W - per_band) // 2 for q in range(4)])
    fid = torch.tensor(wl["frame_ids"])[None]
    return torch.cat([full[idx], fid.expand(idx.numel(), -1)], 1).contiguous()


def cpu_reference_rate(wl, steps, warmup, rays_per_worker):
    """rays/s of the reference algorithm on the host cores.  Returns (rate, ms_per_step, sample_rays, data, cores, kind, sample)."""
    import torch
    from oracle import stash_reference
    import cases as C                                  # job plumbing of oracle/run_reference.py (tests/golden/cases.py)
    sd, data = load_weights(wl)
    bkgd, frames, cams = scene_setup(wl)
    ncpu = os.cpu_count() or 1
    l = wl["layers"] + 1
    gen = torch.Generator().manual_seed(1234)
    have_ref = stash_reference.reference_root() is not None
    # the reference's eager fp32 ops stop scaling near 16 threads (measured on this pool's 128-thread hosts): use every core as
    # independent workers of <= 16 threads, each on its own slice of the sample (rays are independent, SURVEY C.6)
    workers = max(1, ncpu // 16)
    threads = ncpu
    per_band = max(64, (rays_per_worker * workers) // 4)
    times = []
    if have_ref:
        multi = []
        for s in range(warmup + steps):
            rays = cpu_sample(wl, cams, s, per_band)
            multi.append(dict(rays=rays, jitter=torch.rand((l, rays.shape[0], wl["n1"]), generator=gen),
                              u=torch.rand((l, rays.shape[0], wl["n2"]), generator=gen)))
        job = dict(sd=sd, L=wl["layers"], space_time=wl["space_time"], n1=wl["n1"], n2=wl["n2"], bkgd=bkgd, frames=frames,
                   thr=tuple(wl["thr"]), near=wl["near"], alpha=1.0, hidden=[], shift=None, scale=None, multi=multi)
        res = C.run_reference_job(job, workers=workers, threads=threads)      # one interpreter start-up per worker for the whole run
        # per step: the slowest worker's time inside LayeredRFRender.forward on its slice of the step's sample
        times = [(res["rays_each"][s], res["seconds_each"][s]) for s in range(warmup, warmup + steps)]
        kind = "reference"
        how = "unmodified reference LayeredRFRender.forward (out of process), torch fp32, %d workers x %d threads = %d of %d host threads" % (
            workers, max(1, threads // workers), workers * max(1, threads // workers), ncpu)
    else:
        from oracle import stnerf_oracle as O
        nets = O.split_state_dict(sd, wl["layers"])
        sc = O.resolve_scene(frames, bkgd, wl["frame_ids"], None, None)
        sc.update(scale=None, shift=None, shown=[True] * l, near=wl["near"], alpha=1.0, boarder=1e10)
        threads = min(ncpu, 16)
        workers = 1
        torch.set_num_threads(threads)
        per_band = max(64, rays_per_worker // 4)
        for s in range(warmup + steps):
            rays = cpu_sample(wl, cams, s, per_band)
            jit = torch.rand((l, rays.shape[0], wl["n1"]), generator=gen)
            u = torch.rand((l, rays.shape[0], wl["n2"]), generator=gen)
            t0 = time.perf_counter()
            with torch.no_grad():
                O.render(nets, sc, rays, wl["n1"], wl["n2"], jit, u, density_threshold=wl["thr"][0], bkgd_density_threshold=wl["thr"][1])
            if s >= warmup:
                times.append((rays.shape[0], time.perf_counter() - t0))
        kind = "port"
        how = "oracle port (no reference archive found), torch fp32, %d of %d host threads" % (threads, ncpu)
    n = sum(a for a, _ in times)
    t = sum(b for _, b in times)
    cores = workers * max(1, threads // workers) if have_ref else threads
    sample = "%d steps x %d rays (4 row bands of the step's view), full %d+%d path; %s" % (len(times), times[0][0], wl["n1"], wl["n2"], how)
    return n / t, t / len(times) * 1e3, times[0][0], data, cores, kind, sample


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def cpu_leg_parity(wl, model, dev, precision="exact"):
    """Checker of the CPU leg (rank 0, N = 1): the committed fixture of the UNMODIFIED reference for this workload
    (tests/golden/scale_*.npz: 16 384 / 4 096 rays of a full-size view, injected uniforms; inputs regenerated by the test
    infrastructure's seeded generator) against the GPU path in the bench's precision mode."""
    import numpy as np
    import torch
    import cases as C                                  # test infrastructure (imports the oracle's input generators)
    case = C.SCALE_CASES[wl["fixture"]]
    gold = C.load_golden(wl["fixture"])
    if gold is None:
        return None
    rays, jit, u = C.scale_inputs(case)
    ref = gold["fine_mixed.rgb"]

    def one():
        model.inject_uniforms(jit.to(dev).contiguous(), u.to(dev).contiguous())
        with torch.no_grad():
            out = model(rays.to(dev), None, None, density_threshold=case["thr"][0], bkgd_density_threshold=case["thr"][1])
        got = out[0][0].float().cpu().numpy()
        err = np.abs(got - ref).max(1)
        mse = float(((got.astype(np.float64) - ref) ** 2).mean())
        return {"max_abs_rgb_err": float(err.max()), "frac_pixels_over_1e-3": float((err > 1e-3).mean()),
                "pixels_over_1e-3": int((err > 1e-3).sum()), "median_abs_rgb_err": float(np.median(err)),
                "psnr_db": 99.0 if mse == 0 else float(10.0 * math.log10(1.0 / mse))}

    rep = one()
    other = None
    if precision == "exact":       # the opt-in accuracy variant on the same fixture (STNERF_PREC_TC_3XF16_CF; not the timed mode)
        model.set_precision("exact_cf")
        other = one()
        model.set_precision("exact")
    return {"rays": int(rays.shape[0]), **rep, "same_fixture_in_exact_cf_mode": other,
            "against": "unmodified reference LayeredRFRender.forward on CPU (fixture tests/golden/%s.npz), identical rays / weights / "
                       "uniforms; every ray over 1e-3 is attributed (fine-sample placement within the reference's own conditioning, or an "
                       "instability of the reference) in tests/test_gpu_parity_scale.py" % wl["fixture"]}


DUMP_BYTES_PER_ARRAY = 30 * 10**6    # two arrays stay under 64 MB together


def dump_outputs(out_dir, svr, rows, rank, world):
    """Writes the fine and coarse images of the last timed step (every plane: merged + per layer; rgb, depth, acc) as
    float32 `fine_images.npy` / `coarse_images.npy` of shape (planes, pixels, 5).  Where a full view is larger than the
    budget, the same seeded sample of pixels (ascending flat indices) is taken from both."""
    import numpy as np
    import torch
    from stnerf_b200.dist import all_gather_inplace, rows_view
    coarse_local = svr._coarse[1]                               # (1, planes, rows_pad*W, 5): this rank's rows only
    coarse = coarse_local.new_zeros((world,) + tuple(coarse_local.shape))
    coarse[rank].copy_(coarse_local)
    all_gather_inplace(coarse, rank, world)
    if rank != 0:
        return
    images = {"fine_images": svr.assembled(rows)[0], "coarse_images": svr.assembled(rows_view(coarse, svr.W))[0]}
    planes, hw = images["fine_images"].shape[0], svr.H * svr.W
    n = min(hw, DUMP_BYTES_PER_ARRAY // (planes * 5 * 4))
    idx = torch.arange(hw) if n == hw else torch.randperm(hw, generator=torch.Generator().manual_seed(0))[:n].sort()[0]
    os.makedirs(out_dir, exist_ok=True)
    for name, img in images.items():
        a = img.reshape(planes, hw, 5)[:, idx.to(img.device)].float().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(wl, precision, steps, warmup, rank, world, local_rank, want_e2e=True, parity_fn=None, dump_dir=None):
    """One workload on this process' GPU (all ranks call it).  Returns a dict of measurements (complete on rank 0).
    `dump_dir`: write the images of the last timed step there (dump_outputs)."""
    import torch
    import torch.distributed as dist
    import stnerf_b200 as S
    from stnerf_b200.dist import ShardedViewRenderer
    from stnerf_b200.config import make_cfg
    from stnerf_b200 import ops
    import modeling

    dev = torch.device("cuda", local_rank)
    H, W, N1, N2, LAYERS, VIEWS = wl["H"], wl["W"], wl["n1"], wl["n2"], wl["layers"], wl["views"]
    sd, data = load_weights(wl)
    bkgd, frames, cams = scene_setup(wl)
    model = modeling.build_layered_model(make_cfg(LAYERS, N1, N2, wl["space_time"], precision))
    model.load_state_dict(sd)
    model.set_bkgd_bbox(bkgd); model.set_bboxes(frames)
    nat = model._ensure_native(dev)
    model.near = wl["near"]
    model.retiming = True
    scene = model._resolve_scene(torch.tensor(wl["frame_ids"]), wl["thr"][0], wl["thr"][1])   # the demo's thresholds
    svr = ShardedViewRenderer(nat, H, W, N1, N2, rank, world)
    n_local = svr.rp * W
    nat.reserve_host(n_local, 6 + LAYERS + 1)
    rays_per_step = H * W

    def step(i):
        v = nat.make_view(cams[i % VIEWS][0], cams[i % VIEWS][1], wl["frame_ids"], scene, i + 1)
        return svr.render([v], time_collective=(world > 1), with_coarse=True)

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = ClockSampler(local_rank); clocks.start()
    try:                                              # the sampler's nvidia-smi child must not outlive a failed run
        launches0 = S.launch_count()
        nat.profile_begin()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        coll_ms = []
        e0.record()
        for i in range(steps):
            rows = step(warmup + i)
            if world > 1:
                coll_ms.append(svr._timing)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms_total = e0.elapsed_time(e1)
        prof = nat.profile_end()
        launches = S.launch_count() - launches0
    finally:
        clk = clocks.stop()
    if dump_dir is not None:
        dump_outputs(dump_dir, svr, rows, rank, world)
    t = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        lt = torch.tensor([float(launches)], device=dev); dist.all_reduce(lt); launches = int(lt.item())
    ms_total = float(t.item())
    res = {"value": rays_per_step * steps / (ms_total * 1e-3), "ms_per_step": ms_total / steps, "clocks": clk,
           "gpu_launches": int(launches), "data": data, "prof": prof, "n_local": n_local}
    if world > 1:
        ms = [a.elapsed_time(b) for a, b in coll_ms]
        res["collective"] = {"op": "ncclAllGather, in place (send buffer = the rank's slot of the receive buffer), 1 per view",
                             "bytes_per_rank": int((LAYERS + 2) * n_local * 5 * 4), "ms_mean": sum(ms) / len(ms), "ms_max": max(ms),
                             "timed": "CUDA events around the collective on the compute stream (includes waiting for slower ranks)"}

    # ---- e2e: host buffers through the C-ABI (H2D rays + D2H every plane inside the timed region), same step count ------
    if want_e2e:
        n_views_host = min(VIEWS, max(1, steps))           # the SAME views as the timed steps of `value` (work depends on the view)
        rays_host = []
        for v in range(n_views_host):
            K, T = cams[(warmup + v) % VIEWS]
            r = ops.generate_rays(K, T, H, W, frame_ids=wl["frame_ids"], row0=rank, row_step=world, n_rows=svr.rp)
            rays_host.append(r.cpu().pin_memory())
            del r
        out_host = torch.empty((2, LAYERS + 2, 5 * n_local), dtype=torch.float32).pin_memory()
        mask_host = torch.empty((LAYERS + 1, n_local), dtype=torch.uint8).pin_memory()
        nat.set_scene(scene)
        nat.render_host(rays_host[0], N1, N2, seed=99, out_host=out_host, mask_host=mask_host)   # warm
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            nat.render_host(rays_host[i % n_views_host], N1, N2, seed=100 + i, out_host=out_host, mask_host=mask_host)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        te = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        res["e2e"] = {"value": rays_per_step * steps / float(te.item()), "unit": "rays/s",
                      "h2d_bytes_per_step": int(rays_host[0].numel() * 4 * world),
                      "d2h_bytes_per_step": int((out_host.numel() * 4 + mask_host.numel()) * world),
                      "api": "stnerf_render_host (C-ABI, pinned host buffers; rays up and image planes down chunk by chunk on copy "
                             "streams while other chunks render), %d steps, max over ranks of the host wall clock" % steps}
    if parity_fn is not None and rank == 0:
        res["parity"] = parity_fn(wl, model, dev, precision)
    del svr, model
    torch.cuda.empty_cache()
    return res


def roofline_of(wl, res, precision, steps, peaks):
    prof, n_local = res["prof"], res["n_local"]
    N1, N2, LAYERS = wl["n1"], wl["n2"], wl["layers"]
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    sp = prof["spacenet"]
    # algorithmic FLOPs: 2*MAC per evaluated point (nets with a PE(time) input have the wider rgb head); the split between
    # background and performer points comes from the per-launch point counts
    pts = sp["points"]
    bk_pts = float(n_local) * (N1 + N1 + N2) * steps
    flop_perf = FLOP_SPACE_TIME if wl["space_time"] else FLOP_SPACE_NOTIME
    flops = bk_pts * FLOP_SPACE_NOTIME + max(0.0, pts - bk_pts) * flop_perf
    ach = flops / (sp["ms"] * 1e-3) / 1e12 if sp["ms"] > 0 else 0.0
    terms = PRECISION_TERMS[precision]
    traffic, traffic_note = None, None
    try:      # DRAM bytes per point of the same kernel from the committed `ncu --set full` capture, scaled to the mean launch
        cap = json.load(open(os.path.join(ROOT, "profiles", "r02_spacenet_traffic.json")))
        traffic = cap["dram_bytes_per_point"] * pts / max(1, sp["launches"])
        traffic_note = ("NOT measured in this run: dram__bytes_read+write per point (%.1f B) from the committed ncu --set full capture "
                        "profiles/r02_spacenet_traffic.json (%s) x this run's mean points per launch" % (cap["dram_bytes_per_point"], cap["kernel"]))
    except Exception:
        pass
    ms_total = res["ms_per_step"] * steps
    roof = {"kernel": "spacenet MLP (%s)" % precision, "bound": "tensor", "achieved": ach, "peak": peak_tf,
            "unit": "TFLOP/s", "frac": ach / peak_tf, "executed": ach * terms, "frac_executed": ach * terms / peak_tf,
            "peak_source": ("measured bf16_tflops_sustained (MEASURED_PEAKS.json)" if peaks else "fallback 1400 (B200_PROFILING.md)"),
            "traffic": traffic, "traffic_note": traffic_note, "launches": sp["launches"], "avg_launch_ms": sp["ms"] / max(1, sp["launches"]),
            "share_of_step": sp["ms"] / ms_total,
            "note": "achieved/frac = algorithmic FLOPs (2*MAC/point x points evaluated) / CUDA-event launch durations of this run; the split modes "
                    "execute %.2f fp16 MMAs per product (frac = frac_executed / %.2f); executed/frac_executed = what the tensor pipe runs -- the "
                    "denominator is a cuBLAS rate SUSTAINED UNDER THE POWER CAP, not the silicon peak, so frac_executed may pass 1" % (terms, terms),
            "other_kernels_ms": {k: v["ms"] for k, v in prof.items() if k != "spacenet"}}
    # compositing + resampling kernels: algorithmic bytes (depths + raw rgb-sigma in, depths + images out) against the HBM peak,
    # reported for completeness -- they are instruction-issue-bound (sort / search / scan per sample), see DESIGN.md
    cp = prof["composite"]
    hit_frac = max(0.0, pts - bk_pts) / max(1.0, bk_pts)
    bytes_comp = float(n_local) * steps * ((1 + hit_frac) * (N1 * 24 + (N1 + N2) * 20 + (N1 + N2) * 4) + (LAYERS + 2) * 40)
    roof["composite_hbm"] = {"achieved_GBps": bytes_comp / (cp["ms"] * 1e-3) / 1e9 if cp["ms"] > 0 else 0.0,
                             "peak_GBps": peaks.get("hbm_gbs", 6650.0), "share_of_step": cp["ms"] / ms_total}
    return roof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--precision", default="exact", choices=["exact", "exact_cf", "mixed", "fp32", "fast"])
    ap.add_argument("--cpu-sample-rays", type=int, default=1024, help="rays per CPU worker per step of the reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--workload", default="taekwondo2", choices=list(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the fine and coarse images of the last timed step as DIR/<name>.npy (float32, a seeded pixel "
                         "sample where a view exceeds 30 MB per array), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    H, W = wl["H"], wl["W"]
    config = {"workload": wl["name"],
              "step": "one %dx%d view = %d rays (view = step mod %d), coarse + fine images of every layer" % (W, H, H * W, wl["views"]),
              "layers": wl["layers"] + 1, "n1": wl["n1"], "n2": wl["n2"],
              "parallelism": "rows interleaved over %d GPU(s); compositing kernel writes into the rank's slot of a persistent buffer; "
                             "1 in-place all-gather of the fine images per view" % world,
              "l2": "no explicit flush: per-chunk working set (~1.2 GB of samples/raw rgb-sigma buffers) >> 126 MB L2"}

    if args.impl == "reference":
        if rank != 0:
            return
        rate, ms, nr, data, cores, kind, sample = cpu_reference_rate(wl, args.steps, args.warmup, args.cpu_sample_rays)
        print(json.dumps({"impl": "reference", "metric": "rays/sec", "value": rate, "unit": "rays/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic scene; " + data,
                          "config": config,
                          "cpu_baseline": {"value": rate, "unit": "rays/s", "cores": cores, "kind": kind, "sample": sample},
                          "e2e": {"value": rate, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # the reference-fixture parity check belongs to the CPU leg: rank 0 of a single-GPU run, unless --no-cpu-baseline
    parity_fn = cpu_leg_parity if (world == 1 and not args.no_cpu_baseline) else None
    res = measure(wl, args.precision, args.steps, args.warmup, rank, world, local_rank, parity_fn=parity_fn,
                  dump_dir=args.dump_outputs)

    extra = {}
    if not args.no_extra and args.workload == "taekwondo2":
        # the other BASELINE configs, briefly (1 warm-up + 2 / 1 timed steps): driver-visible lines, not the headline
        for name, (k, w_) in (("walking4", (2, 1)), ("walking6_4k", (1, 1))):
            try:
                r = measure(WORKLOADS[name], args.precision, k, w_, rank, world, local_rank, want_e2e=False, parity_fn=parity_fn)
                extra[name] = {"workload": WORKLOADS[name]["name"], "value": r["value"], "unit": "rays/s", "ms_per_step": r["ms_per_step"],
                               "steps": k, "warmup": w_, "n_gpus": world, "parity": r.get("parity"), "collective": r.get("collective"),
                               "spacenet_share_of_step": r["prof"]["spacenet"]["ms"] / (r["ms_per_step"] * k)}
            except Exception as e:                       # an extra line must never take the headline down with it
                extra[name] = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    roof = roofline_of(wl, res, args.precision, args.steps, peaks)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        rate, _, nr, _, cores, kind, sample = cpu_reference_rate(wl, 2, 1, args.cpu_sample_rays)
        cpu = {"value": rate, "unit": "rays/s", "cores": cores, "kind": kind, "sample": sample}

    print(json.dumps({"metric": "rays/sec", "value": res["value"], "unit": "rays/s", "n_gpus": world, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
                      "scaling": "strong", "vs_baseline": None, "dtype": DTYPES[args.precision],
                      "data": "synthetic scene + cameras (SURVEY 8d); " + res["data"], "config": config, "clocks": res["clocks"],
                      "e2e": res.get("e2e"), "gpu_launches": res["gpu_launches"], "roofline": roof, "cpu_baseline": cpu,
                      "parity": res.get("parity"), "collective": res.get("collective"), "precision": args.precision,
                      "extra_workloads": extra or None}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
