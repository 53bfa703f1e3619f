"""Record what the UNMODIFIED reference produces for the drop-in tests (tests/test_reference_dropin.py) and the input
restatement tests (tests/test_inputs.py), so that those tests run without the reference tree.

Needs a checkout of the reference (second.pytorch) at $B2S_REFERENCE_ROOT; its own builders, config files, anchor
generator, point-cloud crop and NuScenes sweep loader run here on the CPU oracle ``spconv`` package, with the seeded
synthetic weights of ``b2second.models.synthetic_weights_`` and the seeded clouds of ``b2second.synth``.  Tensors are
stored as digests (dtype, shape, sha1), detections as exact float lists.  Usage:
    B2S_REFERENCE_ROOT=<second.pytorch checkout> python tests/golden/make_dropin_golden.py
writes tests/golden/reference_dropin.json and tests/golden/reference_inputs.json.
"""
import dataclasses
import json
import os
import re
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(REPO, "second.pytorch_b200"))
sys.path.insert(0, os.path.join(REPO, "tests"))

import golden_util as gu  # noqa: E402
from b2second import config, models, refcompat, spec, synth, tc  # noqa: E402

# (config, use_multi_class_nms agnostic) cases of the per-class NMS branch
MULTICLASS = [("all.fhd", False), ("nuscenes.all.pp.largea", True)]
NETWORKS = ["car.fhd", "all.fhd", "pointpillars.car.xyres_16", "nuscenes.all.pp.largea"]
PLAN_HW = (64, 48)


def reference_net(name, edit=None):
    cfgp = refcompat.load_config(config.REFERENCE_FILES[name])
    if edit is not None:
        edit(cfgp.model.second)
    net = refcompat.build_network(cfgp.model.second).eval()
    models.synthetic_weights_(net, name)
    return net, refcompat.generate_anchors(net, cfgp.model.second)


def forward(net, anchors, pts, max_voxels):
    import torch
    res = net.voxel_generator.generate(pts, max_voxels)
    coords = np.pad(res["coordinates"], ((0, 0), (1, 0)))
    ex = {"anchors": torch.from_numpy(anchors[None].copy()), "voxels": torch.from_numpy(res["voxels"]),
          "num_points": torch.from_numpy(res["num_points_per_voxel"]), "coordinates": torch.from_numpy(coords)}
    with torch.no_grad():
        out = net(ex)[0]
    return {"voxels": gu.voxels_json(res), "detections": gu.detections_json(out)}


def dropin():
    out = {"configs": {}, "networks": {}, "plans": {}, "multiclass": {}}
    for name in sorted(config.BUILTIN):
        path = os.path.join(refcompat.REFERENCE_ROOT, "second", "configs", config.REFERENCE_FILES[name])
        out["configs"][name] = gu.jsonable(config.ModelConfig.from_file(path, name))
    for name in NETWORKS:
        ref, anchors = reference_net(name)
        rec = {"state_dict": gu.state_dict_json(ref.state_dict()), "anchors": gu.digest(anchors)}
        if name == "car.fhd":    # forward equality: one config
            b = config.get_config(name)
            rec["forward"] = forward(ref, anchors, synth.kitti_cloud(4, 12000, b.point_cloud_range), b.max_voxels)
        out["networks"][name] = rec
    for name in sorted(config.BUILTIN):
        ref, _ = reference_net(name)
        cfg = config.get_config(name)
        s = spec.spec_from_module(ref, max_voxels=cfg.max_voxels)
        fm = cfg.feature_map_size
        plan = tc.plan_rpn(ref.rpn, *PLAN_HW)
        out["plans"][name] = {"signature": {k: gu.sha_json(v) for k, v in s.signature().items()},
                              "anchors": gu.digest(spec.anchors_for(s, (fm[1], fm[2]))),
                              "rpn_plan": {"buffers": gu.jsonable(plan["buffers"]),
                                           "ops": [gu.sha_json(op) for op in plan["ops"]]}}
    for name, agnostic in MULTICLASS:
        def edit(m):
            for cs in m.target_assigner.class_settings:
                cs.use_multi_class_nms = True
            m.nms_class_agnostic = agnostic
        ref, anchors = reference_net(name, edit)
        assert ref._multiclass_nms and ref._nms_class_agnostic == agnostic
        b = dataclasses.replace(config.get_config(name), use_multi_class_nms=True, nms_class_agnostic=agnostic)
        pts = synth.nuscenes_cloud(1, 40000) if "nuscenes" in name else synth.kitti_cloud(4, 12000, b.point_cloud_range)
        rec = forward(ref, anchors, pts, b.max_voxels)
        assert len(set(rec["detections"]["label_preds"])) > 1
        out["multiclass"]["%s-%s" % (name, "agnostic" if agnostic else "per_class")] = rec
    return out


def inputs():
    import test_inputs as ti
    from second.core import box_np_ops
    P2, rect, Trv2c, shape = ti.kitti_calib()
    pts = ti.raw_kitti_cloud(0, 20000)
    crop = {"points": gu.digest(pts), "kept": gu.digest(box_np_ops.remove_outside_points(pts, rect, Trv2c, P2, shape))}
    # the dataset file imports scikit-image (kitti_common.py) and fire (nuscenes_dataset.py) at top level; the sweep
    # loader never uses them
    for mod in ("skimage", "skimage.io", "fire"):
        if mod not in sys.modules:
            try:
                __import__(mod)
            except ImportError:
                sys.modules[mod] = types.ModuleType(mod)
    if not hasattr(sys.modules["skimage"], "io"):
        sys.modules["skimage"].io = sys.modules["skimage.io"]
    from second.data.nuscenes_dataset import NuScenesDataset
    sweeps, rots, trans, lags = ti.sweep_case(1)
    ts = 1.5e15
    with tempfile.TemporaryDirectory() as tmp:
        paths = []
        for i, p in enumerate(sweeps):
            f = os.path.join(tmp, "s%d.bin" % i)
            p.tofile(f)
            paths.append(f)
        info = {"token": "t", "lidar_path": paths[0], "timestamp": ts,
                "sweeps": [{"lidar_path": paths[i], "timestamp": ts - lags[i] * 1e6, "sweep2lidar_rotation": rots[i],
                            "sweep2lidar_translation": trans[i]} for i in range(1, len(sweeps))]}
        ds = object.__new__(NuScenesDataset)
        ds._nusc_infos = [info]
        merged = ds.get_sensor_data(0)["lidar"]["points"]
    sweep = {"timestamp": ts, "sweeps": [gu.digest(s) for s in sweeps], "merged": gu.digest(merged.astype(np.float32))}
    return {"crop": crop, "sweep_merge": sweep}


def main():
    import torch
    if not refcompat.reference_available():
        raise SystemExit("set B2S_REFERENCE_ROOT to a checkout of the reference (second.pytorch)")
    refcompat.install(os.path.join(REPO, "oracle", "spconv_cpu"))
    torch.set_num_threads(8)
    for fname, fn in (("reference_dropin.json", dropin), ("reference_inputs.json", inputs)):
        text = json.dumps(fn(), indent=1, sort_keys=True)
        # innermost lists (shapes, box rows, score lists) on one line each
        text = re.sub(r"\[\s+([^\[\]{}]*?)\s+\]", lambda m: "[" + " ".join(m.group(1).split()) + "]", text)
        with open(os.path.join(HERE, fname), "w") as f:
            f.write(text + "\n")
        print(fname, os.path.getsize(os.path.join(HERE, fname)), "bytes")


if __name__ == "__main__":
    main()
