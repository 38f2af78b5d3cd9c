#!/usr/bin/env python
"""Generate the committed golden vectors by running the UNMODIFIED reference on CPU.

Run in the build container (where /root/reference exists):

    python tests/golden/make_golden.py            # all cases + functions.npz
    python tests/golden/make_golden.py tkd_64_128 # one case

Also refreshes ``oracle/_ref/ckpt/*.pt`` (git-ignored copies of the shipped
checkpoints -- weights are input data, not source -- so the GPU box, which has no
/root/reference, can run the checkpoint parity cases).
"""
from __future__ import annotations

import os
import shutil
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import cases as C  # noqa: E402
from oracle import reference_shim as R  # noqa: E402


def stash_checkpoints():
    dst = os.path.join(C.ROOT, "oracle", "_ref", "ckpt")
    os.makedirs(dst, exist_ok=True)
    for scene in ("taekwondo", "walking"):
        src = os.path.join(R.REFERENCE_ROOT, "outputs", scene, "layered_rfnr_checkpoint_1.pt")
        out = os.path.join(dst, scene + ".pt")
        if os.path.isfile(src) and not os.path.isfile(out):
            shutil.copyfile(src, out)


def run_case(name: str):
    case = C.CASES[name]
    sd = C.state_dict_for(case)
    bkgd, frames = C.boxes_for(case)
    model = R.build_model(sd, case["L"], case["n1"], case["n2"], case["space_time"], bkgd, frames,
                          scale=case.get("scale"), shift=case.get("shift"))
    model.near = case.get("near", 0.0)
    model.alpha = case.get("alpha", 1.0)
    for i in case.get("hidden", []):
        model.hide_layer(i)
    rays = C.rays_for(case)
    jit, u = C.uniforms_for(case)
    t0 = time.time()
    out = R.forward(model, rays, jit, u, only_coarse=case.get("only_coarse", False),
                    density_threshold=case["thr"][0], bkgd_density_threshold=case["thr"][1])
    dt = time.time() - t0
    flat = C.flatten_outputs(*out)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **flat)
    hits = [int(m.sum()) for m in out[4]]
    print("%-18s %4d rays  %.2fs  hits=%s" % (name, rays.shape[0], dt, hits))


def run_functions():
    m = R.modules()
    from layers.RaySamplePoint import intersection, RaySamplePoint
    from layers.render_layer import VolumeRenderer
    from utils.sample_pdf import sample_pdf
    from utils.dimension_kernel import Trigonometric_kernel
    from utils.render_helpers import generate_rays
    from modeling.spacenet import SpaceNet
    from modeling.motion_net import MotionNet
    import contextlib, io

    d = C.function_inputs()
    out = {}
    n = d["isect.rays"].shape[0]
    bbox = C.O.corners_from_minmax(d["isect.bmin"], d["isect.bmax"])[None].expand(n, 8, 3)
    out["isect.t"] = intersection(d["isect.rays"], bbox)
    # RaySamplePoint over two layers (layer 0 = bkgd clamp branch) with injected jitter
    rsp = RaySamplePoint(48)
    with R.injected_uniforms([d["sample.jitter"][0], d["sample.jitter"][1]]):
        ts, xyz, mask = rsp.forward(d["isect.rays"], torch.stack([bbox, bbox], 1))
    for i in range(2):
        out["sample.t.%d" % i], out["sample.xyz.%d" % i], out["sample.mask.%d" % i] = ts[i][..., 0], xyz[i], mask[i].to(torch.uint8)
    vr = VolumeRenderer(boarder_weight=1e10)
    c, dp, a, w = vr(d["comp.t"][..., None], d["comp.rgb"], d["comp.sigma"][..., None])
    out["comp.color"], out["comp.depth"], out["comp.acc"], out["comp.w"] = c, dp, a, w[..., 0]
    with R.injected_uniforms([d["pdf.u"]]):
        out["pdf.z"] = sample_pdf(d["pdf.t"], d["pdf.w"][:, 1:-1], N_samples=d["pdf.u"].shape[1])
    out["pe.x3_L10"] = Trigonometric_kernel(L=10)(d["pe.x3"])
    out["pe.x3_L4"] = Trigonometric_kernel(L=4)(d["pe.x3"])
    out["pe.x1_L10"] = Trigonometric_kernel(L=10, input_dim=1)(d["pe.x1"])
    with R.cpu_cuda_shim():
        rays, _ = generate_rays(d["rays.K"], d["rays.T"], None, 24, 40)
    out["rays.rays"] = rays
    # networks: seeded synthetic weights always; checkpoint nets when present
    def space(sd_prefix, sd, use_time):
        net = SpaceNet(include_input=True, use_dir=True, use_time=use_time)
        net.load_state_dict({k[len(sd_prefix):]: v for k, v in sd.items() if k.startswith(sd_prefix)})
        with torch.no_grad():
            return net(d["net.pos"], torch.cat([d["net.pos"], d["net.dirs"]], 1), d["net.time_int"])

    def motion(sd_prefix, sd, tcol):
        net = MotionNet(include_input=True, c_input=4, input_time=True)
        net.load_state_dict({k[len(sd_prefix):]: v for k, v in sd.items() if k.startswith(sd_prefix)})
        with torch.no_grad():
            return net(torch.cat([d["net.pos"], tcol], 1))

    srcs = {"syn": C.O.synthetic_state_dict(1, True, seed=5)}
    if R.available():
        srcs["tkd"] = R.load_checkpoint("taekwondo")
        srcs["walk"] = R.load_checkpoint("walking")
    for tag, sd in srcs.items():
        ut = sd["spacenets.0.rgb_net.1.weight"].shape[1] == 304
        r, s = space("spacenets.0.", sd, ut)
        out["net.%s.perf.rgb" % tag], out["net.%s.perf.sigma" % tag] = r, s
        r, s = space("bkgd_spacenet_fine.", sd, False)
        out["net.%s.bkgd.rgb" % tag], out["net.%s.bkgd.sigma" % tag] = r, s
        out["net.%s.motion_int" % tag] = motion("time_deform_nets.0.", sd, d["net.time_int"])
        out["net.%s.motion_frac" % tag] = motion("time_deform_nets.0.", sd, d["net.time_frac"])
    np.savez_compressed(os.path.join(HERE, "functions.npz"),
                        **{k: np.asarray(v.detach()) for k, v in out.items()})
    print("functions.npz: %d arrays" % len(out))


def reference_path_class():
    """The reference's camera-path / retiming methods, executed from its own source: the class cannot be imported
    (module-level `from config import cfg`, imageio, robopy), so the FunctionDef nodes of the methods are lifted out of
    render/layered_neural_renderer.py unchanged and compiled into a bare class."""
    import ast
    from scipy.spatial.transform import Rotation, Slerp
    from scipy.interpolate import splprep, splev
    src = open(os.path.join(R.REFERENCE_ROOT, "render", "layered_neural_renderer.py")).read()
    tree = ast.parse(src)
    cls = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "LayeredNeuralRenderer"][0]
    want = {"set_smooth_path_poses", "retime_by_key_frames", "set_frame_duration", "set_pose_duration", "invert_poses",
            "is_shown_layer", "load_path_poses"}
    cls.body = [n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name in want]
    mod = ast.Module(body=[cls], type_ignores=[])
    ns = {"np": np, "torch": torch, "R": Rotation, "Slerp": Slerp, "splprep": splprep, "splev": splev}
    exec(compile(mod, "layered_neural_renderer.py", "exec"), ns)
    return ns["LayeredNeuralRenderer"]


def run_camera_path():
    Ref = reference_path_class()
    out = {}
    for name, sc in C.CAMERA_PATH_SCENARIOS.items():
        gt_poses, gt_Ks = C.camera_path_inputs()
        r = Ref.__new__(Ref)
        r.gt_poses, r.gt_Ks = gt_poses, gt_Ks
        r.layer_num = 2
        r.min_frame = [1 + sc["offset"]] * 3
        r.max_frame = [101 + sc["offset"]] * 3
        r.display_layers = {i: (0 if i in sc.get("hidden", []) else 1) for i in range(3)}
        r.min_camera_id, r.max_camera_id = 0, gt_poses.shape[0] - 1
        r.s_shift, r.s_scale, r.s_alpha = sc.get("s_shift"), sc.get("s_scale"), sc.get("s_alpha")
        r.poses, r.Ks, r.layer_frame_pairs = [], [], []
        C.drive_camera_path(r, sc)
        out[name + ".poses"] = np.stack([np.asarray(p, dtype=np.float64) for p in r.poses])
        out[name + ".Ks"] = np.stack([np.asarray(k, dtype=np.float64) for k in r.Ks])
        out[name + ".pairs"] = np.array([[f for (_, f) in pair] for pair in r.layer_frame_pairs], dtype=np.float64)
        if sc.get("s_shift") is not None:
            out[name + ".s_shift_frame"] = np.array(r.s_shift_frame, dtype=np.float64)
        if sc.get("s_alpha") is not None:
            out[name + ".s_alpha_frame"] = np.array(r.s_alpha_frame, dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, "camera_path.npz"), **out)
    print("camera_path.npz: %d arrays" % len(out))


def run_dataset():
    """FrameLayerDataset (data/datasets/frame_dataset.py:94-247) executed unmodified on the synthetic scene directory of
    cases.write_synthetic_dataset.  `open3d` is not installed: a stub module hands the reference the same point arrays the
    PLY files were written from (the PLY reader itself is tested against those arrays in tests/test_scene_data.py).
    `data/__init__` is bypassed (it pulls the training loaders); only data.datasets.{utils,frame_dataset} are imported."""
    import tempfile, types, importlib
    sp = C.DATASET_SPEC
    root = tempfile.mkdtemp(prefix="stnerf_ds_")
    C.write_synthetic_dataset(root)

    class _Cloud:
        def __init__(self, pts): self.points = pts
    o3d = types.ModuleType("open3d"); o3d.io = types.SimpleNamespace()
    def read_point_cloud(path):
        layer_id = int(os.path.basename(path).split(".")[0])
        parent = os.path.basename(os.path.dirname(os.path.dirname(path)))
        frame_id = int(parent[len("frame"):]) if parent.startswith("frame") else 0
        return _Cloud(C.dataset_points(layer_id, frame_id))
    o3d.io.read_point_cloud = read_point_cloud
    sys.modules["open3d"] = o3d
    R.modules()                                  # puts the reference on sys.path (its `utils` package must resolve first)
    for name, sub in (("data", "data"), ("data.datasets", os.path.join("data", "datasets"))):
        m = types.ModuleType(name); m.__path__ = [os.path.join(R.REFERENCE_ROOT, sub)]; sys.modules[name] = m
    fd = importlib.import_module("data.datasets.frame_dataset")
    out = {}
    for fixed in ((-1.0, -1.0), (0.5, 20.0)):
        cfg = types.SimpleNamespace(
            DATASETS=types.SimpleNamespace(TRAIN=root, FIXED_NEAR=fixed[0], FIXED_FAR=fixed[1], SCALE=sp["scale"], CAMERA_STEPSIZE=1,
                                           FILE_OFFSET=0, CAMERA_NUM=0, VIEW_MASK=None))
        tag = "auto" if fixed[0] == -1.0 else "fixed"
        for layer_id in range(sp["layer_num"] + 1):
            for frame_id in range(1 + sp["frame_offset"], sp["frame_offset"] + sp["frame_num"] + 1):
                import contextlib, io
                with contextlib.redirect_stdout(io.StringIO()):
                    d = fd.FrameLayerDataset(cfg, None, frame_id, layer_id)
                k = "%s.l%d.f%d." % (tag, layer_id, frame_id)
                out[k + "bbox"] = np.asarray(d.bbox); out[k + "center"] = np.asarray(d.center, dtype=np.float64)
                out[k + "near"] = np.asarray(d.near); out[k + "far"] = np.asarray(d.far)
                if layer_id == 0 and frame_id == 1 + sp["frame_offset"] and tag == "auto":
                    out["Ts"], out["Ks"] = np.asarray(d.Ts), np.asarray(d.Ks)
                    out["original_size"] = np.asarray(d.get_original_size())
        import shutil
        shutil.rmtree(os.path.join(root, "bbox_tmp"), ignore_errors=True)
        shutil.rmtree(os.path.join(root, "near_far_tmp"), ignore_errors=True)
    np.savez_compressed(os.path.join(HERE, "dataset.npz"), **out)
    print("dataset.npz: %d arrays" % len(out))


def run_checkpoint_io():
    """data/datasets/utils.py (numpy only): checkpoint discovery and camera-file parsing on cases.CHECKPOINT_FILE_NAMES /
    cases.camera_file_inputs().  Paths are stored relative to the checkpoint directory."""
    import importlib.util, tempfile
    spec = importlib.util.spec_from_file_location("_ref_dataset_utils", os.path.join(R.REFERENCE_ROOT, "data", "datasets", "utils.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    d = tempfile.mkdtemp(prefix="stnerf_ckpt_")
    for name in C.CHECKPOINT_FILE_NAMES:
        open(os.path.join(d, name), "w").close()
    Ks, poses = C.camera_file_inputs()
    fn = os.path.join(d, "K.txt")
    np.savetxt(fn, Ks)
    assert ref.get_iteration_path(os.path.join(d, "nope")) is None
    out = dict(iteration_path=np.array(os.path.relpath(ref.get_iteration_path(d), d)),
               iteration_path_fix7=np.array(os.path.relpath(ref.get_iteration_path(d, 7), d)),
               intrinsics=ref.read_intrinsics(fn), extrinsics=ref.campose_to_extrinsic(poses))
    shutil.rmtree(d, ignore_errors=True)
    np.savez_compressed(os.path.join(HERE, "checkpoint_io.npz"), **out)
    print("checkpoint_io.npz: %d arrays" % len(out))


if __name__ == "__main__":
    assert R.available(), "needs /root/reference (build container only)"
    torch.set_num_threads(os.cpu_count())
    stash_checkpoints()
    names = sys.argv[1:] or (list(C.CASES) + ["functions", "camera_path", "dataset", "checkpoint_io"])
    for nm in names:
        if nm == "checkpoint_io":
            run_checkpoint_io()
        elif nm == "functions":
            run_functions()
        elif nm == "camera_path":
            run_camera_path()
        elif nm == "dataset":
            run_dataset()
        else:
            run_case(nm)
