"""On-GPU input path (SURVEY.md §8(f)1): NuScenes sweep merge and KITTI camera-FOV crop.
CPU: the oracle restatement (oracle/py/inputs_ref.py) and the host-side calibration algebra (b2second.inputs) against
what the UNMODIFIED reference functions returned on the same inputs (tests/golden/reference_inputs.json).  GPU: the
CUDA kernels against the oracle, bit for bit."""
import os
import sys

import numpy as np
import pytest
import torch

import golden_util as gu
from conftest import REPO
from b2second import inputs, synth

sys.path.insert(0, os.path.join(REPO, "oracle", "py"))
import inputs_ref  # noqa: E402


def kitti_calib():
    """KITTI-like calibration (values of a typical sequence): P2 [4,4], rect [4,4], Trv2c [4,4], image shape."""
    P2 = np.array([[721.5377, 0.0, 609.5593, 44.85728], [0.0, 721.5377, 172.854, 0.2163791],
                   [0.0, 0.0, 1.0, 0.002745884], [0.0, 0.0, 0.0, 1.0]])
    rect = np.eye(4)
    rect[:3, :3] = np.array([[0.9999239, 0.00983776, -0.00744505], [-0.0098698, 0.9999421, -0.00427846],
                             [0.00740253, 0.00435161, 0.9999631]])
    Trv2c = np.eye(4)
    Trv2c[:3, :] = np.array([[0.00753374, -0.9999714, -0.00061660, -0.00406977],
                             [0.01480249, 0.00072807, -0.9998902, -0.07631618],
                             [0.9998621, 0.00752379, 0.01480755, -0.2717806]])
    return P2, rect, Trv2c, np.array([375, 1242])


def raw_kitti_cloud(seed, n):
    """a 360-degree cloud (the FOV crop has something to remove): forward KITTI-like cloud mirrored to the back."""
    c = synth.kitti_cloud(seed, n, (0, -40, -3, 70.4, 40, 1))
    back = c.copy()
    back[:, 0] = -back[:, 0]
    rng = np.random.default_rng(seed)
    allp = np.concatenate([c, back], 0)
    return allp[rng.permutation(allp.shape[0])].astype(np.float32)


def sweep_case(seed, n_sweeps=4, n=3000):
    rng = np.random.default_rng(seed)
    sweeps, rots, trans, lags = [], [], [], []
    for i in range(n_sweeps):
        p = rng.uniform(-50, 50, (n + 17 * i, 5)).astype(np.float32)
        p[:, 3] = rng.uniform(0, 255, p.shape[0])
        a = rng.uniform(-0.05, 0.05, 3)
        cx, sx, cy, sy, cz, sz = np.cos(a[0]), np.sin(a[0]), np.cos(a[1]), np.sin(a[1]), np.cos(a[2]), np.sin(a[2])
        R = (np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
             @ np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]]))
        sweeps.append(p)
        rots.append(R)
        trans.append(rng.uniform(-3, 3, 3))
        lags.append(0.05 * i + 1e-4 * rng.uniform())
    return sweeps, rots, trans, lags


@pytest.fixture(scope="module")
def ref_inputs():
    """what the reference's own functions returned on the inputs below (tests/golden/make_dropin_golden.py)"""
    return gu.load_json("reference_inputs.json")


def test_crop_restatement_equals_reference_remove_outside_points(ref_inputs):
    """box_np_ops.remove_outside_points of the reference, on the same cloud and calibration."""
    P2, rect, Trv2c, shape = kitti_calib()
    pts = raw_kitti_cloud(0, 20000)
    assert gu.digest(pts) == ref_inputs["crop"]["points"], "synthetic cloud generator drifted"
    planes = inputs.frustum_planes(rect, Trv2c, P2, shape)
    got = inputs_ref.crop_convex_np(pts, planes)
    assert 0 < got.shape[0] < pts.shape[0] // 2 + 100
    assert gu.digest(got) == ref_inputs["crop"]["kept"]


def test_sweep_merge_restatement_equals_reference_dataset_code(ref_inputs):
    """the reference's own NuScenesDataset.get_sensor_data on these sweeps written to disk."""
    sweeps, rots, trans, lags = sweep_case(1)
    assert [gu.digest(p) for p in sweeps] == ref_inputs["sweep_merge"]["sweeps"]
    ts = ref_inputs["sweep_merge"]["timestamp"]
    true_lags = [0.0] + [ts / 1e6 - (ts - lags[i] * 1e6) / 1e6 for i in range(1, len(sweeps))]
    got = inputs_ref.merge_sweeps_np(sweeps, rots, trans, true_lags)
    assert got.dtype == np.float32 and gu.digest(got) == ref_inputs["sweep_merge"]["merged"]


@pytest.mark.gpu
def test_crop_kernel_matches_oracle_and_fills_frame_slots():
    P2, rect, Trv2c, shape = kitti_calib()
    planes = inputs.frustum_planes(rect, Trv2c, P2, shape)
    clouds = [raw_kitti_cloud(s, n) for s, n in ((1, 20000), (2, 300), (3, 29000))]
    refs = [inputs_ref.crop_convex_np(c, planes) for c in clouds]
    out, offs = inputs.crop_convex(torch.from_numpy(clouds[0]).cuda(), planes)
    n0 = int(offs[1].item())
    assert n0 == refs[0].shape[0] and np.array_equal(out[:n0].cpu().numpy(), refs[0])
    # three frames appended back to back into one buffer, offsets chained on the device
    cap = sum(r.shape[0] for r in refs) + 10
    buf = torch.zeros(cap, 4, device="cuda")
    offsets = torch.zeros(4, dtype=torch.int32, device="cuda")
    crop = inputs.ConvexCrop(60000, "cuda")
    keep = [crop.crop_into(torch.from_numpy(c).cuda(), planes, buf, offsets, b) for b, c in enumerate(clouds)]
    o = offsets.cpu().tolist()
    assert o == np.cumsum([0] + [r.shape[0] for r in refs]).tolist()
    assert np.array_equal(buf[:o[3]].cpu().numpy(), np.concatenate(refs, 0))
    # overflow: the tail is dropped, never written past the buffer, and reported
    small = torch.zeros(refs[0].shape[0] - 5, 4, device="cuda")
    st = torch.zeros(1, dtype=torch.int32, device="cuda")
    offsets.zero_()
    crop.crop_into(torch.from_numpy(clouds[0]).cuda(), planes, small, offsets, 0, st)
    assert int(offsets[1].item()) == small.shape[0] and int(st.item()) == 2
    assert np.array_equal(small.cpu().numpy(), refs[0][:small.shape[0]])
    del keep


@pytest.mark.gpu
def test_sweep_merge_kernel_matches_oracle():
    sweeps, rots, trans, lags = sweep_case(2, n_sweeps=10, n=30000)
    ref = inputs_ref.merge_sweeps_np(sweeps, rots, trans, lags)
    got = inputs.merge_sweeps([torch.from_numpy(s).cuda() for s in sweeps], rots, trans, lags).cpu().numpy()
    assert got.shape == ref.shape == (sum(s.shape[0] for s in sweeps), 4)
    assert np.array_equal(got[:, 3], ref[:, 3])
    same = got[:, :3] == ref[:, :3]
    # float64 dot product rounded to float32: a BLAS that fuses multiply-add may differ in the last float64 bit, which
    # can flip a float32 rounding only at an exact tie -- allow a handful of 1-ulp differences, nothing else
    assert same.mean() > 0.99999
    assert float(np.abs(got[:, :3] - ref[:, :3]).max()) <= 4e-6


@pytest.mark.gpu
def test_engine_takes_raw_clouds_with_fov_crop_and_sweeps(product):
    """net(example) with raw 360-degree KITTI clouds + crop planes == net(example) with the clouds cropped on the host;
    net(example) with NuScenes sweeps == net(example) with the cloud merged on the host."""
    from b2second import config, fastpath, models
    P2, rect, Trv2c, shape = kitti_calib()
    planes = inputs.frustum_planes(rect, Trv2c, P2, shape)
    name = "car.fhd"
    net = models.build_network(config.get_config(name), product).eval()
    models.synthetic_weights_(net, name, seed=0)
    net = fastpath.accelerate(net.cuda(), max_points=60000)
    clouds = [raw_kitti_cloud(s, 20000) for s in (4, 5)]
    anchors = torch.from_numpy(net.anchors()[None]).cuda()
    a = net({"points": [torch.from_numpy(c).cuda() for c in clouds], "crop_planes": planes, "anchors": anchors})
    b = net({"points": [torch.from_numpy(inputs_ref.crop_convex_np(c, planes)) for c in clouds], "anchors": anchors})
    for x, y in zip(a, b):
        assert x["box3d_lidar"].shape[0] > 0
        assert torch.equal(x["box3d_lidar"], y["box3d_lidar"]) and torch.equal(x["scores"], y["scores"])
    name = "nuscenes.all.pp.largea"
    net = models.build_network(config.get_config(name), product).eval()
    models.synthetic_weights_(net, name, seed=0)
    net = fastpath.accelerate(net.cuda(), max_points=120000)
    full = synth.nuscenes_cloud(3, 100000)
    # split the synthetic 10-sweep cloud back into "sweeps" in a shifted frame, so that merging restores it
    parts = np.array_split(full, 5)
    rng = np.random.default_rng(0)
    rots, trans, lags, sweeps = [], [], [], []
    for i, p in enumerate(parts):
        ang = 0.01 * i
        R = np.array([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1.0]])
        t = rng.uniform(-1, 1, 3) * (i > 0)
        q = np.zeros((p.shape[0], 5), np.float32)
        q[:, :3] = ((p[:, :3].astype(np.float64) - t) @ R).astype(np.float32)      # inverse transform (approximately)
        sweeps.append(q)
        rots.append(R)
        trans.append(t)
        lags.append(0.05 * i)
    merged = inputs_ref.merge_sweeps_np(sweeps, rots, trans, lags)
    anchors = torch.from_numpy(net.anchors()[None]).cuda()
    a = net({"sweeps": [{"sweeps": [torch.from_numpy(s).cuda() for s in sweeps], "rotations": rots, "translations": trans,
                         "time_lags": lags}], "anchors": anchors})[0]
    b = net({"points": [torch.from_numpy(merged)], "anchors": anchors})[0]
    assert a["box3d_lidar"].shape[0] > 0
    torch.testing.assert_close(a["box3d_lidar"], b["box3d_lidar"], rtol=1e-5, atol=1e-4)
    assert torch.equal(a["label_preds"], b["label_preds"])
