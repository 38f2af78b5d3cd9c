"""Checkpoint discovery / loading and camera-file parsing (SURVEY 8f rows 3-4).  CPU only.  checkpoint_io.npz holds what
the reference's own functions (data/datasets/utils.py) return for the same inputs (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

import cases as C
from tests_support import make_cfg


def test_get_iteration_path(tmp_path):
    from stnerf_b200 import checkpoint_io as io
    ref = C.load_golden("checkpoint_io")
    d = str(tmp_path)
    assert io.get_iteration_path(os.path.join(d, "nope")) is None
    assert io.get_iteration_path(d) is None                                   # empty directory
    for name in C.CHECKPOINT_FILE_NAMES:
        open(os.path.join(d, name), "w").close()
    assert io.get_iteration_path(d) == os.path.join(d, "layered_rfnr_checkpoint_12.pt")
    assert io.get_iteration_path(d, fix_iter=7) == os.path.join(d, "frame", "layered_rfnr_checkpoint_7.pt")
    assert io.get_iteration_path(d) == os.path.join(d, str(ref["iteration_path"]))
    assert io.get_iteration_path(d, 7) == os.path.join(d, str(ref["iteration_path_fix7"]))


def test_camera_file_parsing(tmp_path):
    from stnerf_b200 import checkpoint_io as io
    ref = C.load_golden("checkpoint_io")
    Ks, poses = C.camera_file_inputs()
    fn = os.path.join(str(tmp_path), "K.txt")
    np.savetxt(fn, Ks)
    got = io.read_intrinsics(fn)
    assert got.shape == (5, 3, 3) and np.array_equal(got, np.loadtxt(fn).reshape(5, 3, 3))
    ext = io.campose_to_extrinsic(poses)
    assert ext.shape == (5, 4, 4) and np.array_equal(ext[:, :3, :].reshape(5, 12), poses) and np.all(ext[:, 3] == [0, 0, 0, 1])
    with pytest.raises(Exception):
        io.campose_to_extrinsic(np.random.RandomState(3).rand(5, 11))
    assert np.array_equal(got, ref["intrinsics"])
    assert np.array_equal(ext, ref["extrinsics"])


def test_load_checkpoint_backfills_missing_keys(tmp_path):
    import modeling
    from stnerf_b200 import checkpoint_io as io
    case = C.CASES["syn_L2_64_128"]
    sd = C.state_dict_for(case)
    partial = {k: v for k, v in sd.items() if not k.startswith("time_deform_nets.1.")}
    path = os.path.join(str(tmp_path), "layered_rfnr_checkpoint_1.pt")
    torch.save({"model": partial}, path)
    m = modeling.build_layered_model(make_cfg(2, 64, 128, True))
    fresh = m.state_dict()
    missing = io.load_checkpoint(m, io.get_iteration_path(str(tmp_path)))
    assert sorted(missing) == sorted(k for k in sd if k.startswith("time_deform_nets.1."))
    now = m.state_dict()
    assert torch.equal(now["spacenets.0.stage1.0.weight"], sd["spacenets.0.stage1.0.weight"])
    assert torch.equal(now["time_deform_nets.1.motion_net.0.weight"], fresh["time_deform_nets.1.motion_net.0.weight"])


# ---- packed-weight cache (SURVEY 8f row 3) ---------------------------------------------------------------------------------
def test_weight_cache_file_format(tmp_path):
    from stnerf_b200 import checkpoint_io as CK
    pt = tmp_path / "layered_rfnr_checkpoint_1.pt"
    pt.write_bytes(b"checkpoint bytes v1")
    assert CK.read_weight_cache(str(pt)) is None                                  # nothing cached yet
    image = bytes(range(256)) * 3
    cache = CK.write_weight_cache(str(pt), image)
    assert cache == str(pt) + CK.CACHE_SUFFIX and CK.read_weight_cache(str(pt)) == image
    pt.write_bytes(b"checkpoint bytes v2")                                        # retrained: the hash no longer matches
    assert CK.read_weight_cache(str(pt)) is None
    CK.write_weight_cache(str(pt), image)
    raw = open(cache, "rb").read()
    open(cache, "wb").write(raw[:-5])                                             # truncated
    assert CK.read_weight_cache(str(pt)) is None
    open(cache, "wb").write(raw + b"x")                                           # trailing garbage
    assert CK.read_weight_cache(str(pt)) is None
    open(cache, "wb").write(b"BADMAGIC" + raw[8:])
    assert CK.read_weight_cache(str(pt)) is None


@pytest.mark.gpu
def test_packed_weights_round_trip_bit_identical(tmp_path):
    import time
    import modeling
    from stnerf_b200 import checkpoint_io as CK
    from stnerf_b200._lib import StnerfError
    from stnerf_b200.config import make_cfg
    from stnerf_b200.synthetic import synthetic_state_dict, synthetic_boxes
    import cases as C
    case = C.CASES["syn_L2_64_128"]
    sd = synthetic_state_dict(2, True, seed=21)
    pt = str(tmp_path / "layered_rfnr_checkpoint_7.pt")
    torch.save({"model": sd}, pt)
    bkgd, frames = C.boxes_for(case)
    rays = C.rays_for(case).cuda()
    jit, u = C.uniforms_for(case)

    def render(m):
        m.set_bkgd_bbox(bkgd); m.set_bboxes(frames)
        m.inject_uniforms(jit.cuda(), u.cuda())
        with torch.no_grad():
            out = m(rays, None, None, density_threshold=0.0, bkgd_density_threshold=0.0)
        return [t.clone() for t in out[0]] + [t.clone() for t in out[1]]

    for prec in ("exact", "fp32"):
        a = modeling.build_layered_model(make_cfg(2, 64, 128, True, prec))
        t0 = time.time(); how = CK.load_checkpoint_cached(a, pt); t_first = time.time() - t0
        assert how == ("checkpoint" if prec == "exact" else "cache")
        ref = render(a)
        b = modeling.build_layered_model(make_cfg(2, 64, 128, True, prec))
        t0 = time.time(); how = CK.load_checkpoint_cached(b, pt); t_cached = time.time() - t0
        assert how == "cache"
        got = render(b)
        for x, y in zip(ref, got):
            assert torch.equal(x, y)                                               # same device bytes -> same pixels
        print("load %s: checkpoint+pack %.1f ms, cached image %.1f ms" % (prec, 1e3 * t_first, 1e3 * t_cached))
        # the tensors behind a packed model are still reachable (lazily) for state_dict() users
        sd_b = b.state_dict()
        assert torch.equal(sd_b["spacenets.1.stage2.4.weight"], sd["spacenets.1.stage2.4.weight"])

    image = a.export_packed()
    assert image[:8] == b"STNB200W"
    # an image for another layer configuration, a damaged image, a truncated image: rejected before any network is touched
    c3 = modeling.build_layered_model(make_cfg(3, 64, 128, True, "exact"))
    c3.load_packed(image)
    with pytest.raises(StnerfError):
        c3._ensure_native(torch.device("cuda", 0))
    for bad in (image[:-1], b"XXXXXXXX" + image[8:], image[:4096]):
        d = modeling.build_layered_model(make_cfg(2, 64, 128, True, "exact"))
        d.load_packed(bad)
        with pytest.raises(StnerfError):
            d._ensure_native(torch.device("cuda", 0))
    nt = modeling.build_layered_model(make_cfg(2, 64, 128, False, "exact"))        # performer nets without the time input
    nt.load_packed(image)
    with pytest.raises(StnerfError):
        nt._ensure_native(torch.device("cuda", 0))
    # a stale cache (other checkpoint contents) is ignored and rewritten
    sd2 = synthetic_state_dict(2, True, seed=22)
    torch.save({"model": sd2}, pt)
    e = modeling.build_layered_model(make_cfg(2, 64, 128, True, "exact"))
    assert CK.load_checkpoint_cached(e, pt) == "checkpoint"
    assert not torch.equal(render(e)[0], ref[0])
