"""Deterministic definitions of the golden / parity cases.

Shared by ``make_golden.py`` (which runs the unmodified reference in the build
container), the ``not gpu`` oracle-pinning tests and the ``gpu`` parity tests.
Everything here is regenerated from seeds; only the reference's *outputs* are
stored in ``tests/golden/*.npz``.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for _p in (ROOT, os.path.join(ROOT, "st-nerf_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from oracle import stnerf_oracle as O  # noqa: E402

GOLDEN_DIR = os.path.dirname(os.path.abspath(__file__))

# name -> spec.  weights: "taekwondo" | "walking" (shipped checkpoints) | "synthetic"
CASES = {
    # BASELINE config #1 flavour: 1 performer, coarse only, 64 samples
    "syn_L1_coarse": dict(weights="synthetic", seed=11, L=1, space_time=True, n1=64, n2=0, only_coarse=True,
                          frame_ids=[0, 10], thr=(1e-4, 0.0), n_rays=160, ray_seed=1),
    "syn_L2_64_128": dict(weights="synthetic", seed=12, L=2, space_time=True, n1=64, n2=128,
                          frame_ids=[0, 10, 11], thr=(0.0, 0.0), n_rays=160, ray_seed=2),
    # the demo configuration of taekwondo (thresholds 0/0), integer frame ids
    "tkd_64_128": dict(weights="taekwondo", L=2, space_time=True, n1=64, n2=128,
                       frame_ids=[0, 10, 11], thr=(0.0, 0.0), n_rays=192, ray_seed=3),
    # fractional frame ids (MotionNet lerp + bbox lerp) and the shift/scale edits of demo/taekwondo_demo.py:55,65
    "tkd_edit_frac": dict(weights="taekwondo", L=2, space_time=True, n1=64, n2=128,
                          frame_ids=[0, 10.5, 11.25], thr=(1e-4, 0.0), n_rays=192, ray_seed=4,
                          shift=[[0, 0, 0], [0, 2, 0], [0, -2, 0]], scale=[1, 0.75, 1.5], alpha=0.5),
    # demo/walking_demo.py:43-50: thresholds 20/0.8, near=4; reference sample counts 90+30; layer 1 hidden
    "walk_90_30_hide": dict(weights="walking", L=2, space_time=False, n1=90, n2=30,
                            frame_ids=[0, 30, 31], thr=(20.0, 0.8), near=4.0, hidden=[1], n_rays=160, ray_seed=5),
    # evaluator layout: 7-column rays [o,d,frame_id], boxes by index_select, no thresholds (engine/layered_trainer.py:36,383)
    "tkd_eval_7col": dict(weights="taekwondo", L=2, space_time=True, n1=64, n2=128, seven=True,
                          frame_ids=[10, 10, 10], thr=(20.0, 0.8), n_rays=128, ray_seed=8),
    # a mixed-frame batch as the trainer draws it: 7-column rays, every ray with its OWN integer frame id -> boxes per ray by
    # index_select(frame_id - 1) (modeling/layered_rfrender.py:193), shift/scale edits on top
    "tkd_train_7col_mixed": dict(weights="taekwondo", L=2, space_time=True, n1=64, n2=128, seven=True, mixed_frames=(3, 60),
                                 frame_ids=[10, 10, 10], thr=(20.0, 0.8), n_rays=160, ray_seed=9,
                                 shift=[[0, 0, 0], [0, 0.5, 0], [0, -0.5, 0]], scale=[1, 0.9, 1.2]),
    # BASELINE config #3 flavour: walking nets replicated round-robin to 4 performer layers
    "walk_L4_64_128": dict(weights="walking", L=4, space_time=False, n1=64, n2=128,
                           frame_ids=[0, 30, 31, 32, 33], thr=(20.0, 0.8), near=4.0, n_rays=128, ray_seed=6),
}


from stnerf_b200.checkpoint_io import find_checkpoint, replicate_layers  # noqa: E402,F401  (shared with bench / examples)


def state_dict_for(case: dict):
    """Returns the fp32 state_dict of the case, or None when it needs a checkpoint that is not present."""
    if case["weights"] == "synthetic":
        return O.synthetic_state_dict(case["L"], case["space_time"], seed=case["seed"])
    path = find_checkpoint(case["weights"])
    if path is None:
        return None
    sd = torch.load(path, map_location="cpu")
    sd = sd["model"] if "model" in sd else sd
    return replicate_layers(sd, case["L"])


def boxes_for(case: dict):
    return O.synthetic_boxes(case["L"])


def rays_for(case: dict) -> torch.Tensor:
    """n_rays rays from the 1080p synthetic camera (view 1 of 16) + frame-id columns.

    A quarter are pixel-grid rays (incl. the four image corners, which miss every performer);
    the rest are aimed at random points in and just around each (edited) performer box so that
    every layer gets hits, grazing rays and near misses.
    """
    K, T = O.synthetic_camera(1, 16, 1080, 1920)
    rs = np.random.RandomState(case["ray_seed"])
    n = case["n_rays"]
    n_grid = n // 4
    rows = rs.randint(250, 900, size=n_grid)
    cols = rs.randint(350, 1570, size=n_grid)
    rows[:4], cols[:4] = [0, 0, 1079, 1079], [0, 1919, 0, 1919]
    full = O.generate_rays(K, T, 1080, 1920)
    grid = full[torch.from_numpy(rows * 1920 + cols)]
    sc = scene_for(case)
    eye = T[:3, 3]
    aimed = []
    L = case["L"]
    for j in range(n - n_grid):
        i = 1 + (j % L)
        lo, hi = sc["bmin"][i], sc["bmax"][i]
        c, half = (lo + hi) / 2, (hi - lo) / 2
        p = c + half * 1.25 * torch.from_numpy(rs.uniform(-1, 1, 3).astype(np.float32))
        dvec = p - eye
        aimed.append(torch.cat([eye, dvec / dvec.norm()]))
    rays = torch.cat([grid, torch.stack(aimed, 0)], 0)
    ids = case["frame_ids"][:1] if case.get("seven") else case["frame_ids"]
    fid = torch.tensor(ids, dtype=torch.float32)[None].expand(n, -1)
    if case.get("mixed_frames"):                      # one integer frame id per ray
        lo_f, hi_f = case["mixed_frames"]
        fid = torch.from_numpy(rs.randint(lo_f, hi_f + 1, size=(n, 1)).astype(np.float32))
    return torch.cat([rays, fid], 1).contiguous()


def uniforms_for(case: dict):
    l = case["L"] + 1
    rs = np.random.RandomState(1000 + case["ray_seed"])
    jit = torch.from_numpy(rs.random_sample((l, case["n_rays"], case["n1"])).astype(np.float32))
    u = torch.from_numpy(rs.random_sample((l, case["n_rays"], max(case["n2"], 1))).astype(np.float32))
    # float32 rounding of a double in [0,1) can give exactly 1.0; torch.rand never does
    jit.clamp_(max=float(np.nextafter(np.float32(1), np.float32(0))))
    u.clamp_(max=float(np.nextafter(np.float32(1), np.float32(0))))
    return jit, (u if case["n2"] > 0 else None)


def scene_for(case: dict):
    """Oracle-side scene dict (edited boxes etc.) for the case."""
    bkgd, frames = boxes_for(case)
    sc = O.resolve_scene(frames, bkgd, case["frame_ids"], case.get("scale"), case.get("shift"))
    l = case["L"] + 1
    sc.update(scale=case.get("scale"), shift=case.get("shift"),
              shown=[i not in case.get("hidden", []) for i in range(l)],
              near=case.get("near", 0.0), alpha=case.get("alpha", 1.0), boarder=1e10)
    if case.get("mixed_frames"):
        sc["box_table"] = O.box_table(frames, bkgd, case.get("scale"), case.get("shift"))
    return sc


OUTPUT_KEYS = ("fine_mixed", "coarse_mixed", "fine_layer", "coarse_layer")


def flatten_outputs(fine_mixed, coarse_mixed, fine_layer, coarse_layer, ray_mask) -> dict:
    """5-tuple of the reference / facade -> flat dict of numpy arrays (the .npz schema)."""
    d = {}
    for name, trip in (("fine_mixed", fine_mixed), ("coarse_mixed", coarse_mixed)):
        for part, v in zip(("rgb", "depth", "acc"), trip):
            d["%s.%s" % (name, part)] = np.asarray(v.detach().cpu().reshape(v.shape[0], -1), dtype=np.float32)
    for name, lst in (("fine_layer", fine_layer), ("coarse_layer", coarse_layer)):
        for i, trip in enumerate(lst):
            for part, v in zip(("rgb", "depth", "acc"), trip):
                d["%s.%d.%s" % (name, i, part)] = np.asarray(v.detach().cpu().reshape(v.shape[0], -1), dtype=np.float32)
    for i, m in enumerate(ray_mask):
        d["ray_mask.%d" % i] = np.asarray(m.detach().cpu()).astype(np.uint8)
    return d


def load_golden(name: str):
    p = os.path.join(GOLDEN_DIR, name + ".npz")
    return dict(np.load(p)) if os.path.isfile(p) else None


# --------------------------------------------------------------------------- per-function vectors
def function_inputs() -> dict:
    """Seeded inputs for the per-stage goldens (functions.npz).  Pure function of the seeds below."""
    rs = np.random.RandomState(77)
    f = lambda *s: torch.from_numpy(rs.standard_normal(s).astype(np.float32))  # noqa: E731
    uni = lambda *s: torch.from_numpy(rs.random_sample(s).astype(np.float32)).clamp_(max=0.99999994)  # noqa: E731
    d = {}
    # rays around two boxes (some start inside, some miss, some axis-parallel)
    n = 256
    o = f(n, 3) * 2.0
    dirs = f(n, 3)
    dirs = dirs / dirs.norm(dim=1, keepdim=True)
    dirs[:8, 0] = 0.0            # exactly axis-parallel components (the +eps branch)
    o[8:16] = o[8:16] * 0.2      # origins inside the box
    d["isect.rays"] = torch.cat([o, dirs], 1)
    d["isect.bmin"] = torch.tensor([-1.0, -0.5, -0.25])
    d["isect.bmax"] = torch.tensor([1.0, 0.75, 1.5])
    d["sample.jitter"] = uni(2, n, 48)
    # compositing
    t = torch.sort(uni(64, 96) * 6.0, 1)[0]
    d["comp.t"] = t
    d["comp.rgb"] = f(64, 96, 3) * 3.0
    d["comp.sigma"] = f(64, 96) * 40.0
    # sample_pdf
    d["pdf.t"] = torch.sort(uni(64, 64) * 5.0 + 1.0, 1)[0]
    w = uni(64, 64) ** 8
    w[:4] = 0.0                  # all-zero weights -> uniform pdf
    w[4:8, 10] = 50.0            # one dominant bin
    d["pdf.w"] = w
    d["pdf.u"] = uni(64, 128)
    # encodings / nets
    d["pe.x3"] = f(200, 3) * 3.0
    d["pe.x1"] = uni(50, 1) * 100.0
    d["net.pos"] = f(300, 3) * 1.5
    dd = f(300, 3)
    d["net.dirs"] = dd / dd.norm(dim=1, keepdim=True)
    d["net.time_int"] = torch.full((300, 1), 37.0)
    d["net.time_frac"] = torch.full((300, 1), 37.25)
    # ray generation: a small image with an off-centre principal point
    d["rays.K"] = torch.tensor([[31.2, 0.0, 19.5], [0.0, 30.7, 12.25], [0.0, 0.0, 1.0]])
    K, T = O.synthetic_camera(3, 16, 24, 40)
    d["rays.T"] = T
    return d


# --------------------------------------------------------------------------- camera-path scenarios (SURVEY 8f row 2)
CAMERA_PATH_SCENARIOS = {
    # demo/taekwondo_demo.py:41-52
    "taekwondo": dict(offset=0, steps=101, around=False, smooth_time=False,
                      retime=[(1, [21, 49, 74, 87], [20, 50, 74, 85]), (2, [13, 42, 80, 90], [20, 50, 74, 85])]),
    # demo/walking_demo.py:46-50 (FRAME_OFFSET 25, pose duration [1,14), inverted path), one layer hidden
    "walking": dict(offset=25, steps=100, around=False, smooth_time=False, pose_duration=(1, 14), invert=True, hidden=[1]),
    # all cameras as rotation keys, fractional frame ids, edit schedules
    "around_smooth": dict(offset=0, steps=37, around=True, smooth_time=True,
                          s_shift=[[[0, 0, 0], [0, 0, 0], [0, 0, 0]], [[0, 0, 0], [0, 2, 0], [0, -2, 0]]],
                          s_alpha=[1.0, 0.25]),
}


def camera_path_inputs():
    """16 ground-truth cameras of the synthetic rig as the torch tensors the reference's dataset object holds."""
    cams = [O.synthetic_camera(v, 16, 1080, 1920) for v in range(16)]
    gt_poses = torch.stack([T for (_, T) in cams], 0)
    gt_Ks = [K * (1.0 + 0.01 * i) for i, (K, _) in enumerate(cams)]
    return gt_poses, gt_Ks


def drive_camera_path(r, sc):
    """The same call sequence for the reference class (golden generation) and for stnerf_b200.CameraPath (test)."""
    if "pose_duration" in sc:
        r.set_pose_duration(*sc["pose_duration"])
    r.set_smooth_path_poses(sc["steps"], around=sc["around"], smooth_time=sc["smooth_time"])
    for layer_id, kfl, kf in sc.get("retime", []):
        r.retime_by_key_frames(layer_id, kfl, kf)
    if sc.get("invert"):
        r.invert_poses()


CHECKPOINT_FILE_NAMES = ("layered_rfnr_checkpoint_3.pt", "layered_rfnr_checkpoint_12.pt", "layered_rfnr_checkpoint_5_200.pt",
                         "other.pt")


def camera_file_inputs():
    """Rows of K.txt (5, 9) and camera poses (5, 12) for the camera-file parsers (checkpoint_io.npz)."""
    rs = np.random.RandomState(3)
    return rs.rand(5, 9) * 1000, rs.rand(5, 12)


# ---------------------------------------------------------------------------------------------------------------------
# Synthetic captured-scene directory (SURVEY 8f row 4): the files FrameLayerDataset / Ray_Dataset_Render read.
# ---------------------------------------------------------------------------------------------------------------------
DATASET_SPEC = dict(layer_num=2, frame_num=3, frame_offset=2, scale=0.5, size_test=(96, 54), original=(192, 108), cams=4)


def dataset_points(layer_id: int, frame_id: int) -> np.ndarray:
    """float32-representable points of one layer at one frame (float64 array, as open3d hands them out)."""
    rng = np.random.RandomState(100 * layer_id + frame_id)
    if layer_id == 0:
        p = rng.uniform([-6, -6, -1], [6, 6, 4], size=(257, 3))
    else:
        c = np.array([-2.0 + 2.0 * layer_id + 0.1 * frame_id, 0.3 * frame_id, 0.9])
        p = c + rng.normal(size=(150 + frame_id, 3)) * np.array([0.3, 0.3, 0.5])
    return p.astype(np.float32).astype(np.float64)


def write_ply(path: str, pts: np.ndarray, fmt: str):
    """fmt: 'ascii' | 'le_f4' | 'le_f8_extra' (binary little endian doubles with colour bytes interleaved) | 'be_f4'."""
    n = pts.shape[0]
    with open(path, "wb") as f:
        if fmt == "ascii":
            hdr = "ply\nformat ascii 1.0\ncomment synthetic\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\nend_header\n" % n
            f.write(hdr.encode())
            for p in pts:
                f.write(("%.9g %.9g %.9g\n" % tuple(np.float32(p))).encode())
        elif fmt in ("le_f4", "be_f4"):
            end = "little" if fmt == "le_f4" else "big"
            hdr = "ply\nformat binary_%s_endian 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\nelement face 0\nproperty list uchar int vertex_indices\nend_header\n" % (end, n)
            f.write(hdr.encode())
            f.write(pts.astype("<f4" if fmt == "le_f4" else ">f4").tobytes())
        elif fmt == "le_f8_extra":
            hdr = ("ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty uchar red\nproperty double x\nproperty double y\n"
                   "property uchar green\nproperty double z\nend_header\n" % n)
            f.write(hdr.encode())
            dt = np.dtype([("red", "u1"), ("x", "<f8"), ("y", "<f8"), ("green", "u1"), ("z", "<f8")])
            rec = np.zeros(n, dtype=dt)
            rec["x"], rec["y"], rec["z"], rec["red"], rec["green"] = pts[:, 0], pts[:, 1], pts[:, 2], 7, 9
            f.write(rec.tobytes())
        else:
            raise ValueError(fmt)


def write_synthetic_dataset(root: str, with_image: bool = True, spec: dict = None):
    sp = spec or DATASET_SPEC
    os.makedirs(os.path.join(root, "pose"), exist_ok=True)
    os.makedirs(os.path.join(root, "background"), exist_ok=True)
    Ks, Ts = [], []
    for v in range(sp["cams"]):
        K, T = O.synthetic_camera(v, sp["cams"], sp["original"][1], sp["original"][0])
        Ks.append(np.asarray(K, dtype=np.float64).reshape(-1)); Ts.append(np.asarray(T, dtype=np.float64)[:3].reshape(-1))
    np.savetxt(os.path.join(root, "pose", "K.txt"), np.stack(Ks), fmt="%.10g")
    np.savetxt(os.path.join(root, "pose", "RT_c2w.txt"), np.stack(Ts), fmt="%.10g")
    write_ply(os.path.join(root, "background", "0.ply"), dataset_points(0, 0), "le_f8_extra")
    fmts = {1: "ascii", 2: "le_f4"}
    for frame_id in range(1 + sp["frame_offset"], sp["frame_offset"] + sp["frame_num"] + 1):
        d = os.path.join(root, "frame%d" % frame_id, "pointclouds")
        os.makedirs(d, exist_ok=True)
        for layer_id in (1, 2):
            write_ply(os.path.join(d, "%d.ply" % layer_id), dataset_points(layer_id, frame_id),
                      "be_f4" if (layer_id == 2 and frame_id % 2 == 0) else fmts[layer_id])
        if with_image:
            from PIL import Image
            os.makedirs(os.path.join(root, "frame%d" % frame_id, "images"), exist_ok=True)
            Image.new("RGB", sp["original"], (10, 20, 30)).save(os.path.join(root, "frame%d" % frame_id, "images", "000.png"))


# ---------------------------------------------------------------------------------------------------------------------
# Parity at scale (BASELINE configs[1], configs[2] and the 64+192 sampling of configs[4]): thousands of rays of a full-size
# view, spread evenly over the image.  `make_golden_scale.py` stores the UNMODIFIED reference's fine images for these inputs;
# the gpu test compares the B200 path with them and attributes every pixel over the 1e-3 gate (tests/test_gpu_parity_scale.py).
# ---------------------------------------------------------------------------------------------------------------------
SCALE_CASES = {
    "scale_tkd2_16k": dict(weights="taekwondo", L=2, space_time=True, n1=64, n2=128, frame_ids=[0, 10, 11], thr=(0.0, 0.0),
                           near=0.0, n_rays=16384, H=1080, W=1920, view=3, views=16, seed=11),
    "scale_walk4_16k": dict(weights="walking", L=4, space_time=False, n1=64, n2=128, frame_ids=[0, 30, 31, 32, 33],
                            thr=(20.0, 0.8), near=4.0, n_rays=16384, H=1080, W=1920, view=5, views=16, seed=12),
    "scale_walk6_4k": dict(weights="walking", L=6, space_time=False, n1=64, n2=192, frame_ids=[0, 30, 31, 32, 33, 34, 35],
                           thr=(20.0, 0.8), near=4.0, n_rays=4096, H=2160, W=3840, view=9, views=32, seed=13),
}


def scale_inputs(case: dict):
    """rays (N, 6+l), jitter (l,N,n1), u (l,N,n2): pixel rays at evenly spaced flat indices of the view, seeded uniforms."""
    K, T = O.synthetic_camera(case["view"], case["views"], case["H"], case["W"])
    full = O.generate_rays(K, T, case["H"], case["W"])
    n, l = case["n_rays"], case["L"] + 1
    idx = torch.linspace(0, case["H"] * case["W"] - 1, n).long()
    rays = torch.cat([full[idx], torch.tensor(case["frame_ids"], dtype=torch.float32)[None].expand(n, -1)], 1).contiguous()
    g = torch.Generator().manual_seed(case["seed"])
    jit = torch.rand((l, n, case["n1"]), generator=g)
    u = torch.rand((l, n, case["n2"]), generator=g)
    return rays, jit, u


def reference_job(case: dict, rays, jit, u, sd=None, **extra) -> dict:
    """Job dict of oracle/run_reference.py for a case of CASES / SCALE_CASES."""
    sd = sd if sd is not None else state_dict_for(case)
    bkgd, frames = boxes_for(case)
    job = dict(sd=sd, L=case["L"], space_time=case["space_time"], n1=case["n1"], n2=case["n2"], bkgd=bkgd, frames=frames,
               rays=rays, jitter=jit, u=u, thr=tuple(case["thr"]), near=case.get("near", 0.0), alpha=case.get("alpha", 1.0),
               hidden=list(case.get("hidden", [])), shift=case.get("shift"), scale=case.get("scale"),
               only_coarse=bool(case.get("only_coarse", False)))
    job.update(extra)
    return job


def run_reference_job(job: dict, workers: int = 1, threads: int = 0) -> dict:
    """Run the unmodified reference on `job` in a separate process (oracle/run_reference.py); returns its result dict.
    threads = 0: min(16, cores) per worker (the reference's eager fp32 ops stop scaling there; 128 threads on a few hundred
    rays are slower than 8)."""
    if threads <= 0:
        threads = min(16, os.cpu_count() or 1) * max(1, workers)
    import subprocess
    import tempfile
    d = tempfile.mkdtemp(prefix="stnerf_refcall_")
    jin, jout = os.path.join(d, "job.pt"), os.path.join(d, "res.pt")
    torch.save(job, jin)
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "run_reference.py"), "--in", jin, "--out", jout,
           "--workers", str(workers), "--threads", str(threads)]
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)                      # the child must not see the facade packages
    subprocess.check_call(cmd, env=env, cwd=ROOT)
    res = torch.load(jout, weights_only=False)
    import shutil
    shutil.rmtree(d, ignore_errors=True)
    return res


SCALE_KEYS_STORED = ("fine_mixed", "fine_layer", "ray_mask")


def scale_golden_path(name: str) -> str:
    return os.path.join(GOLDEN_DIR, name + ".npz")
