"""helpers shared by the golden-fixture tests (CPU oracle path and GPU product path)."""
import dataclasses
import glob
import hashlib
import json
import os

import numpy as np

from b2second import config, synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def digest(a):
    """dtype, shape and sha1 of a tensor or array: equal digests <=> equal arrays (bit for bit)."""
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.ascontiguousarray(a)
    return {"dtype": a.dtype.name, "shape": list(a.shape), "sha1": hashlib.sha1(a.tobytes()).hexdigest()}


def jsonable(x):
    """the plain-JSON form of a config, spec signature or launch plan; tensors and arrays become digests, so
    jsonable(a) == jsonable(b) <=> a == b field by field (torch.equal for tensors)."""
    if hasattr(x, "detach") or isinstance(x, np.ndarray):
        return digest(x)
    if dataclasses.is_dataclass(x) and not isinstance(x, type):
        return jsonable(dataclasses.asdict(x))
    if isinstance(x, dict):
        return {str(k): jsonable(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [jsonable(v) for v in x]
    if isinstance(x, np.generic):
        return x.item()
    if x is None or isinstance(x, (bool, int, float, str)):
        return x
    raise TypeError("no JSON form for %r" % type(x))


def sha_json(x):
    """sha1 of the canonical JSON form of x: compares a whole spec field or launch op in 40 characters."""
    return hashlib.sha1(json.dumps(jsonable(x), sort_keys=True).encode()).hexdigest()


TRAINING_BUFFERS = ("rpn_acc", "rpn_precision", "rpn_recall", "rpn_metrics", "rpn_cls_loss", "rpn_loc_loss",
                    "rpn_total_loss")


def state_dict_json(sd):
    """{"tensors": {key: [dtype, shape]}, "weights_sha1": sha1 over (key, dtype, shape, bytes) of every entry in key
    order, the reference's training-metric buffers left out}."""
    h = hashlib.sha1()
    for k in sorted(sd):
        if k.split(".")[0] not in TRAINING_BUFFERS:
            h.update(json.dumps([k, digest(sd[k])]).encode())
    return {"tensors": {k: [digest(v)["dtype"], list(v.shape)] for k, v in sd.items()}, "weights_sha1": h.hexdigest()}


def load_json(name):
    with open(os.path.join(GOLDEN_DIR, name)) as f:
        return json.load(f)


def detections_json(out):
    """the detections of one frame (box3d_lidar / scores / label_preds) as exact JSON lists."""
    return {k: np.asarray(out[k]).tolist() for k in ("box3d_lidar", "scores", "label_preds")}


def voxels_json(res):
    """digests of a voxelizer result (the network input, so a forward comparison starts from the same data)."""
    return {k: digest(res[k]) for k in ("voxels", "coordinates", "num_points_per_voxel")}


def cases():
    """(config name, seed, num_points, fixture path); fixtures named <config>.seed<S>.n<P>[.mv<max_voxels>].npz"""
    import re
    out = []
    for p in sorted(glob.glob(os.path.join(GOLDEN_DIR, "*.npz"))):
        m = re.match(r"^(.*)\.seed(\d+)\.n(\d+)(?:\.mv(\d+))?$", os.path.basename(p)[:-4])
        out.append((m.group(1), int(m.group(2)), int(m.group(3)), p))
    return out


def max_voxels_of(fix, name):
    """the voxel cap the fixture was generated with (older fixtures: the config's own)."""
    return int(fix["max_voxels"]) if "max_voxels" in fix else config.get_config(name).max_voxels


def sha(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


def make_cloud(name, seed, n):
    cfg = config.get_config(name)
    if "nuscenes" in name:
        return synth.nuscenes_cloud(seed, n)
    return synth.kitti_cloud(seed, n, cfg.point_cloud_range)


def assert_detections_close(got, fix, box_tol=1e-4, score_tol=1e-5):
    gb = np.asarray(got["box3d_lidar"], dtype=np.float32)
    gs = np.asarray(got["scores"], dtype=np.float32)
    gl = np.asarray(got["label_preds"]).astype(np.int64)
    rb, rs, rl = fix["box3d_lidar"], fix["scores"], fix["label_preds"]
    assert gb.shape == rb.shape, "detection count differs: got %d, golden %d" % (gb.shape[0], rb.shape[0])
    np.testing.assert_allclose(gs, rs, rtol=0, atol=score_tol)
    # detections arrive in descending score order; among (numerically) EQUAL scores the order is whatever torch.topk /
    # the sort produced -- unspecified upstream -- so rows inside a run of tied scores are matched by nearest centre
    order = np.arange(len(rs))
    i = 0
    while i < len(rs):
        j = i + 1
        while j < len(rs) and abs(float(rs[j]) - float(rs[i])) <= 2 * score_tol:
            j += 1
        if j - i > 1:
            free = list(range(i, j))
            for a in range(i, j):
                k = min(free, key=lambda q: float(np.abs(gb[q, :3] - rb[a, :3]).sum()))
                free.remove(k)
                order[a] = k
        i = j
    gb, gs, gl = gb[order], gs[order], gl[order]
    # labels: argmax over class logits; only decided where the top-2 logit margin is above fp32 noise
    decided = np.asarray(fix["label_margin"]) > 1e-3 if "label_margin" in fix else np.ones(rl.shape, bool)
    np.testing.assert_array_equal(gl[decided], rl[decided])
    # The bar (BASELINE.json north_star) is 1e-4 on the box REGRESSION outputs.  The decode
    # (box_torch_ops.py:56-102) multiplies them by the anchor: x = xt*diag + xa, z = zt*h + za, w = exp(wt)*wa ...,
    # so a decoded coordinate may move by 1e-4 * max(1, diag, h) of its own box (NuScenes buses: diag ~ 12 m),
    # plus 2e-5 relative for fp32 rounding of the decoded magnitude (|x| ~ 70 m).
    scale = np.maximum(1.0, np.maximum(np.hypot(rb[:, 3], rb[:, 4]), rb[:, 5]))[:, None]
    err = np.abs(gb[:, :6] - rb[:, :6])
    bound = 2e-5 * np.abs(rb[:, :6]) + box_tol * scale
    bad = err > bound
    assert not bad.any(), "decoded boxes differ: %d elements, worst %g (bound %g)" % (
        int(bad.sum()), float((err - bound).max() + bound[np.unravel_index(np.argmax(err - bound), err.shape)]),
        float(bound[np.unravel_index(np.argmax(err - bound), err.shape)]))
    # angles are compared modulo 2*pi (direction fix-up adds multiples of the period)
    d = np.abs(gb[:, 6] - rb[:, 6])
    d = np.minimum(d, np.abs(d - 2 * np.pi))
    assert d.max(initial=0.0) < box_tol * 10, "yaw mismatch %g" % d.max()
