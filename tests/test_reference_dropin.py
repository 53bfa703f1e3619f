"""This repository against the UNMODIFIED reference, through what the reference produced for the same configs, weights
and clouds (tests/golden/reference_dropin.json, written by tests/golden/make_dropin_golden.py):
  * the hand-written config dataclasses equal the parsed reference config files
  * anchors equal the reference's TargetAssigner output bit for bit
  * the mirror network has the reference's state-dict keys/shapes/weights and gives the same detections on the oracle
  * the fused engine plans the mirror exactly as it plans the reference network
  * the reference's own builders construct VoxelNet on top of the CUDA drop-in `spconv` (needs the reference tree)
"""
import dataclasses
import subprocess
import sys

import numpy as np
import pytest
import torch

import golden_util as gu
from b2second import config, loader, models, refcompat, synth

GOLDEN = gu.load_json("reference_dropin.json")


def forward(net, max_voxels, pts, golden):
    """net on the voxelized cloud; the voxelizer must reproduce the reference's network input first."""
    res = net.voxel_generator.generate(pts, max_voxels)
    assert gu.voxels_json(res) == golden["voxels"]
    coords = np.pad(res["coordinates"], ((0, 0), (1, 0)))
    ex = {"anchors": torch.from_numpy(net.anchors()[None].copy()), "voxels": torch.from_numpy(res["voxels"]),
          "num_points": torch.from_numpy(res["num_points_per_voxel"]), "coordinates": torch.from_numpy(coords)}
    with torch.no_grad():
        o_m = net(ex)[0]
    d = golden["detections"]
    o_r = {"box3d_lidar": torch.tensor(d["box3d_lidar"], dtype=torch.float32).reshape(-1, 7),
           "scores": torch.tensor(d["scores"], dtype=torch.float32),
           "label_preds": torch.tensor(d["label_preds"], dtype=o_m["label_preds"].dtype)}
    assert o_r["box3d_lidar"].shape == o_m["box3d_lidar"].shape and o_r["box3d_lidar"].shape[0] > 0
    return o_r, o_m


@pytest.mark.parametrize("name", sorted(config.BUILTIN))
def test_builtin_config_equals_reference_file(name):
    parsed = GOLDEN["configs"][name]
    builtin = config.get_config(name)
    assert set(parsed) == set(builtin.__dataclass_fields__)
    for f in builtin.__dataclass_fields__:
        assert gu.jsonable(getattr(builtin, f)) == parsed[f], f


@pytest.mark.parametrize("name", ["car.fhd", "all.fhd", "pointpillars.car.xyres_16", "nuscenes.all.pp.largea"])
def test_mirror_equals_reference_network(oracle, name):
    ref = GOLDEN["networks"][name]
    mine = models.build_network(name, oracle).eval()
    models.synthetic_weights_(mine, name)
    sd_r, sd_m = ref["state_dict"]["tensors"], mine.state_dict()
    assert set(sd_m) <= set(sd_r)
    assert all(k.split(".")[0].startswith("rpn_") for k in set(sd_r) - set(sd_m))   # training metric buffers only
    for k in sd_m:
        assert [gu.digest(sd_m[k])["dtype"], list(sd_m[k].shape)] == sd_r[k], k
    assert gu.state_dict_json(sd_m)["weights_sha1"] == ref["state_dict"]["weights_sha1"]   # same synthetic weights
    # reference checkpoints load unchanged: every reference key, training-metric buffers included
    ckpt = {k: sd_m[k] if k in sd_m else torch.zeros(shape, dtype=getattr(torch, dtype))
            for k, (dtype, shape) in sd_r.items()}
    fresh = models.build_network(name, oracle).eval()
    fresh.load_reference_state_dict(ckpt)
    assert gu.state_dict_json(fresh.state_dict())["weights_sha1"] == ref["state_dict"]["weights_sha1"]
    assert gu.digest(mine.anchors()) == ref["anchors"]
    if name != "car.fhd":
        return                                                   # forward equality: one config is enough here
    b = config.get_config(name)
    o_r, o_m = forward(mine, b.max_voxels, synth.kitti_cloud(4, 12000, b.point_cloud_range), ref["forward"])
    assert torch.allclose(o_r["box3d_lidar"], o_m["box3d_lidar"], atol=1e-6)
    assert torch.equal(o_r["label_preds"], o_m["label_preds"])


@pytest.mark.parametrize("name", sorted(config.BUILTIN))
def test_engine_plan_from_reference_network_equals_plan_from_mirror(oracle, name):
    """b2second.spec reads a network through the reference's attribute names only, so the fused engine plans the
    UNMODIFIED reference VoxelNet (second_builder.build) exactly as it plans the mirror: same layer list, folded
    BN constants, NMS / direction parameters, RPN weights and anchors -- for all five BASELINE configs."""
    from b2second import spec, tc
    ref = GOLDEN["plans"][name]
    mine = models.build_network(name, oracle).eval()
    models.synthetic_weights_(mine, name)
    cfg = config.get_config(name)
    s_mine = spec.spec_from_module(mine, max_voxels=cfg.max_voxels)
    a, b = ref["signature"], s_mine.signature()
    assert set(a) == set(b)
    for k in a:
        assert a[k] == gu.sha_json(b[k]), "spec field %s differs between the reference network and the mirror" % k
    fm = cfg.feature_map_size
    assert gu.digest(spec.anchors_for(s_mine, (fm[1], fm[2]))) == ref["anchors"]
    # the RPN launch program is planned from the module tree, too
    H, W = 64, 48
    p_mine = tc.plan_rpn(mine.rpn, H, W)
    assert len(ref["rpn_plan"]["ops"]) == len(p_mine["ops"])
    assert ref["rpn_plan"]["buffers"] == gu.jsonable(p_mine["buffers"])
    for i, (o1, o2) in enumerate(zip(ref["rpn_plan"]["ops"], p_mine["ops"])):
        assert o1 == gu.sha_json(o2), "RPN op %d differs" % i


@pytest.mark.parametrize("name,agnostic", [("all.fhd", False), ("nuscenes.all.pp.largea", True)])
def test_multiclass_nms_branch_mirror_equals_reference(oracle, name, agnostic):
    """the per-class NMS branch of predict() (voxelnet.py:458-547; off in the five BASELINE configs, SURVEY §8(f)3):
    the UNMODIFIED reference network with use_multi_class_nms switched on vs the mirror, on the CPU oracle."""
    ref = GOLDEN["multiclass"]["%s-%s" % (name, "agnostic" if agnostic else "per_class")]
    b = dataclasses.replace(config.get_config(name), use_multi_class_nms=True, nms_class_agnostic=agnostic)
    mine = models.build_network(b, oracle).eval()
    models.synthetic_weights_(mine, name)
    pts = synth.nuscenes_cloud(1, 40000) if "nuscenes" in name else synth.kitti_cloud(4, 12000, b.point_cloud_range)
    o_r, o_m = forward(mine, b.max_voxels, pts, ref)
    assert len(set(o_r["label_preds"].tolist())) > 1                      # more than one class produced detections
    assert torch.allclose(o_r["box3d_lidar"], o_m["box3d_lidar"], atol=1e-6)
    assert torch.equal(o_r["label_preds"], o_m["label_preds"]) and torch.allclose(o_r["scores"], o_m["scores"])


@pytest.mark.skipif(not refcompat.reference_available(), reason="reference tree not present")
def test_reference_builds_on_cuda_dropin_in_subprocess():
    """`import spconv` == second.pytorch_b200/spconv; the reference's second_builder constructs VoxelNet on it."""
    code = r"""
import sys
sys.path.insert(0, %r)
from b2second import refcompat, loader, config
refcompat.install(loader.PRODUCT_DIR)
import spconv
assert not getattr(spconv, "__oracle__", False) and spconv.__version__.endswith("b2second")
for f in ("car.fhd.config", "car.lite.config", "pointpillars/car/xyres_16.config"):
    cfg = refcompat.load_config(f)
    net = refcompat.build_network(cfg.model.second)
    mods = [m for m in net.modules() if isinstance(m, spconv.SparseConvolution)]
    print(f, type(net).__module__, len(net.state_dict()), len(mods))
    assert type(net).__module__ == "second.pytorch.models.voxelnet"
print("OK")
""" % loader.PRODUCT_DIR
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
    assert "car.fhd.config second.pytorch.models.voxelnet 149 14" in r.stdout
