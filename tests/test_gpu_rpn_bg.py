"""The background-tile path of the dense RPN (csrc/rpn_bg.cu and the work / background lists of k_conv3x3_tc2 in
csrc/conv_tc2.cu), one launch at a time and in the engine at the bench batch.

1. k_conv3x3_tc2 with lists, against the same launch without them: work tiles bit-identical (and within the float64
   bars of tests/test_tc_error_model.py), background tiles bit-equal to a SYNTHETIC random field -- so a copy from the
   wrong row, column, frame or channel chunk cannot match by accident -- and everything else (halo, channels past Cout of
   a wider record, tiles in neither list) still the NaN sentinel.  List entries past each count hold tile ids the launch
   must not touch.
2. b2s_rpn_bg_fill at every channel width its chunk arithmetic covers, and separate fill + work-list launch against the
   fused fill.
3. b2s_rpn_bg_plan against its numpy restatement (tests/test_host_rpn_plan.py) past one 1024-tile compaction pass.
4. The engine with the skip on (fused and separate fill) and off at the bench batch: bit-identical heads and detections.
5. B2S_CONV_V2=0 (the 3x3 layers on k_conv_tc) runs the engine without background tiles."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import golden_util as gu
from test_gpu_tc_forms import F16_NAN, _check_split, _report, _sentinel
from test_host_rpn_plan import bg_plan_numpy
from test_tc_error_model import DENSE_MAX_REL, DENSE_RMS_REL, dense_operands, dense_planes, dense_terms, epilogue, rel_errors

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
FORM = (3, 3, 1, 1, 128, 128, 1, 2, True, True)        # the one form that takes tile lists
TILE = 16


def _tiles(B, H, W):
    th, tw = -(-H // TILE), -(-W // TILE)
    return th, tw, B * th * tw


def _pixel_tiles(B, H, W):
    """[B, H, W] id of the 16x16 tile each pixel belongs to: (b * tiles_h + th) * tiles_w + tw."""
    th, tw, _ = _tiles(B, H, W)
    b = torch.arange(B, device="cuda")[:, None, None]
    h = (torch.arange(H, device="cuda") // TILE)[None, :, None]
    w = (torch.arange(W, device="cuda") // TILE)[None, None, :]
    return (b * th + h) * tw + w


def _list(ids, nt):
    """device list buffer of nt entries: `ids` first, then every other tile id -- what a launch that reads past the
    count would wrongly process; and the count."""
    ids = np.asarray(ids, dtype=np.int64)
    rest = np.setdiff1d(np.arange(nt), ids)
    buf = torch.from_numpy(np.concatenate([ids, rest]).astype(np.int32)).cuda()
    return buf, torch.tensor([len(ids)], dtype=torch.int32, device="cuda")


def _field(shape, seed):
    """a synthetic empty-frame response: random finite fp16 hi and lo planes (not a hi/lo split of anything)."""
    g = torch.Generator().manual_seed(seed)
    return ((torch.randn(shape, generator=g) * 4).half().cuda(), (torch.randn(shape, generator=g) * 1e-3).half().cuda())


def _expected(pix, field, ostride, cout, work_src=None):
    """int16 image of an output plane [B, H+2, W+2, ostride] given the class of every image pixel `pix` [B, H, W]:
    work pixels (1) from `work_src` [B, H, W, cout], background pixels (2) from field[h+1, w+1, :cout], everything else
    (class 0, halo, channels past cout) the NaN sentinel."""
    B, H, W = pix.shape
    exp = torch.full((B, H + 2, W + 2, ostride), F16_NAN, dtype=torch.int16, device="cuda")
    inner = exp[:, 1:-1, 1:-1, :cout]
    if work_src is not None:
        inner[pix == 1] = work_src.view(torch.int16)[pix == 1]
    f = field[1:-1, 1:-1, :cout].view(torch.int16)[None].expand(B, H, W, cout)
    inner[pix == 2] = f[pix == 2]
    return exp


def _compare(got, exp, pix, what):
    """bit equality of an output plane with its expected image; a mismatch is reported per region."""
    bad = got.view(torch.int16) != exp
    if not bool(bad.any()):
        return
    cls = torch.full(bad.shape[:3], -1, dtype=torch.int64, device="cuda")
    cls[:, 1:-1, 1:-1] = pix
    counts = {name: int((bad & (cls == c)[..., None]).sum()) for name, c in (("work", 1), ("background", 2),
                                                                            ("neither", 0), ("halo", -1))}
    pytest.fail("%s: %d elements differ %s" % (what, int(bad.sum()), counts))


# ---------------------------------------------------------------- 1. k_conv3x3_tc2 with lists
GEOMS = {"fhd": (2, 200, 176), "lite": (3, 160, 132), "odd": (2, 40, 21), "one-tile": (1, 16, 16),
         "fhd-b8": (8, 200, 176)}
CASES = ([("fhd", r) for r in ("planner", "no-work", "no-bg", "three-work", "last-row", "shuffled", "half-bg",
                               "cout64")]
         + [("lite", r) for r in ("planner", "half-bg", "no-work", "cout64")]
         + [("odd", r) for r in ("planner", "last-row", "three-work", "half-bg")]
         + [("one-tile", r) for r in ("no-work", "no-bg")]
         + [("fhd-b8", r) for r in ("planner", "three-work", "shuffled")])


class Dense:
    """operands of one 3x3 128 -> Cout layer with ReLU on B x H x W, the output of its list-free launch (NaN sentinel
    planes of out_stride = Cout + 8 channels) and its float64 reference [B, H, W, Cout]."""

    def __init__(self, product, B, H, W, cout):
        self.L, self.lib = product._lib, product._lib.load()
        self.B, self.H, self.W, self.cout, self.ostride = B, H, W, cout, cout + 8
        x, w, scale, shift = dense_operands(FORM, B, H, W, cout, seed=B * 1000 + H + W + cout)
        self.x_hi, self.x_lo, self.w_hi, self.w_lo, ws = [t.cuda() if torch.is_tensor(t) else t
                                                          for t in dense_planes(x, w, 128)]
        self.scale_k, self.shift = (scale / ws).cuda(), shift.cuda()
        self.o_hi, self.o_lo = self.launch()
        ref = epilogue(sum(dense_terms(self.x_hi, self.x_lo, self.w_hi, self.w_lo, FORM, cout).values()),
                       self.scale_k, self.shift, True)
        self.ref = ref.permute(0, 2, 3, 1).contiguous()

    def planes(self):
        shape = (self.B, self.H + 2, self.W + 2, self.ostride)
        return _sentinel(shape, torch.float16), _sentinel(shape, torch.float16)

    def launch(self, work=None, bg=None, field=(None, None), out=None):
        """one b2s_conv2d_tc_ex launch; work / bg = (list, count) device pairs; returns the output planes."""
        L = self.L
        o_hi, o_lo = out if out is not None else self.planes()
        work, n_work = work if work is not None else (None, None)
        bg, n_bg = bg if bg is not None else (None, None)
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        L.check(self.lib.b2s_conv2d_tc_ex(
            L.ptr(self.x_hi), L.ptr(self.x_lo), self.B, self.H, self.W, 128, L.ptr(self.w_hi), L.ptr(self.w_lo), 3, 3,
            1, 1, self.cout, 128, L.ptr(self.scale_k), L.ptr(self.shift), 1, self.H, self.W, L.ptr(o_hi), L.ptr(o_lo),
            self.H, self.W, 1, self.ostride, 1, 0, 0, L.ptr(work), L.ptr(n_work), L.ptr(bg), L.ptr(n_bg),
            L.ptr(field[0]), L.ptr(field[1]), L.ptr(status), L.stream()), "b2s_conv2d_tc_ex")
        torch.cuda.synchronize()
        assert int(status.item()) == 0
        return o_hi, o_lo

    def inner(self, t):
        return t[:, 1:-1, 1:-1, :self.cout]


@pytest.fixture(scope="module")
def dense(product):
    """Dense per (B, H, W, Cout), built once and checked against float64 when first used."""
    cache = {}

    def get(B, H, W, cout):
        key = (B, H, W, cout)
        if key not in cache:
            d = Dense(product, B, H, W, cout)
            mask = torch.zeros(d.o_hi.shape, dtype=torch.bool, device="cuda")
            mask[:, 1:-1, 1:-1, :cout] = True
            for t in (d.o_hi, d.o_lo):
                assert bool((t.view(torch.int16)[~mask] == F16_NAN).all()), "list-free launch wrote halo / channels"
            got = d.inner(d.o_hi).double() + d.inner(d.o_lo).double()
            _report("conv3x3 no lists B%d %dx%d cout %d" % key, *rel_errors(got, d.ref), DENSE_MAX_REL, DENSE_RMS_REL)
            _check_split(d.inner(d.o_hi), d.inner(d.o_lo))
            cache[key] = d
        return cache[key]

    yield get
    cache.clear()
    torch.cuda.empty_cache()


def _occupancy(rng, B, H, W):
    """0.2 % random pixels plus blobs touching the top, right and bottom-left border; frame 1 of three or more empty."""
    occ = (rng.random((B, H, W)) < 0.002).astype(np.uint8)
    occ[0, :3, W // 3:W // 3 + 5] = 1
    occ[0, H // 2:H // 2 + 4, W - 2:] = 1
    occ[B - 1, H - 2:, :4] = 1
    if B >= 3:
        occ[1] = 0
    return occ


def _lists(regime, B, H, W, rng):
    """(work tile ids, background tile ids) of a list regime, as numpy arrays."""
    th, tw, nt = _tiles(B, H, W)
    ids = np.arange(nt)
    if regime in ("planner", "shuffled", "half-bg", "cout64"):
        flags = bg_plan_numpy(_occupancy(rng, B, H, W), 2)[1].reshape(-1)
        work, bg = ids[flags != 0], ids[flags == 0]
        assert len(work) > 0 and len(bg) > 0
    elif regime == "no-work":
        work, bg = ids[:0], ids
    elif regime == "no-bg":
        work, bg = ids, ids[:0]
    elif regime == "three-work":
        work = np.sort(rng.choice(nt, 3, replace=False))
        bg = np.setdiff1d(ids, work)
    elif regime == "last-row":
        last = (ids // tw) % th == th - 1
        work, bg = ids[last], ids[~last]
    else:
        raise ValueError(regime)
    if regime == "shuffled":
        work, bg = rng.permutation(work), rng.permutation(bg)
    if regime == "half-bg":
        bg = bg[::2]
    return np.ascontiguousarray(work), np.ascontiguousarray(bg)


@pytest.mark.timeout(300)
@pytest.mark.parametrize("geom,regime", CASES, ids=["%s-%s" % c for c in CASES])
def test_conv3x3_tile_lists(dense, geom, regime):
    """work tiles bit-identical to the list-free launch, background tiles = the field, all else the sentinel.  Regimes:
    planner lists (random occupancy, blobs on the border), no work, no background, three work tiles, only the last tile
    row (half tiles), shuffled lists, half of the background listed, Cout = 64 with n_pad = 128."""
    B, H, W = GEOMS[geom]
    cout = 64 if regime == "cout64" else 128
    d = dense(B, H, W, cout)
    rng = np.random.default_rng(len(geom) * 100 + len(regime))
    work, bg = _lists(regime, B, H, W, rng)
    _, _, nt = _tiles(B, H, W)
    field = _field((H + 2, W + 2, cout), seed=nt + len(regime))
    o_hi, o_lo = d.launch(_list(work, nt), _list(bg, nt), field)
    cls = torch.zeros(nt, dtype=torch.int64, device="cuda")
    cls[torch.from_numpy(work).long().cuda()] = 1
    cls[torch.from_numpy(bg).long().cuda()] = 2
    pix = cls[_pixel_tiles(B, H, W)]
    if regime == "half-bg":
        assert bool((pix == 0).any())
    what = "%s %s B%d %dx%d" % (geom, regime, B, H, W)
    _compare(o_hi, _expected(pix, field[0], d.ostride, cout, d.inner(d.o_hi)), pix, what + " hi")
    _compare(o_lo, _expected(pix, field[1], d.ostride, cout, d.inner(d.o_lo)), pix, what + " lo")
    if len(work):
        m = pix == 1
        got = d.inner(o_hi)[m].double() + d.inner(o_lo)[m].double()
        _report("conv3x3 %s work tiles" % what, *rel_errors(got, d.ref[m]), DENSE_MAX_REL, DENSE_RMS_REL)
        _check_split(d.inner(o_hi)[m], d.inner(o_lo)[m])


# ---------------------------------------------------------------- 2. b2s_rpn_bg_fill
@pytest.mark.timeout(120)
@pytest.mark.parametrize("B,H,W", [(2, 160, 132), (3, 40, 21)])
@pytest.mark.parametrize("C", [8, 64, 128, 256])
def test_bg_fill_copies_listed_tiles_only(product, C, B, H, W):
    """b2s_rpn_bg_fill into a record of C + 8 channels: the listed tiles (half of them, shuffled) get field[h+1, w+1, :C],
    partial tiles only their in-image pixels, everything else keeps the sentinel."""
    L, lib = product._lib, product._lib.load()
    th, tw, nt = _tiles(B, H, W)
    rng = np.random.default_rng(C + H)
    bg = rng.permutation(nt)[:(nt + 1) // 2]
    field = _field((H + 2, W + 2, C), seed=C * 7 + W)
    ostride = C + 8
    o_hi = _sentinel((B, H + 2, W + 2, ostride), torch.float16)
    o_lo = _sentinel(o_hi.shape, torch.float16)
    lst, cnt = _list(bg, nt)
    L.check(lib.b2s_rpn_bg_fill(L.ptr(lst), L.ptr(cnt), B, H, W, C, L.ptr(field[0]), L.ptr(field[1]), L.ptr(o_hi),
                                L.ptr(o_lo), ostride, L.stream()), "b2s_rpn_bg_fill")
    torch.cuda.synchronize()
    cls = torch.zeros(nt, dtype=torch.int64, device="cuda")
    cls[torch.from_numpy(bg).long().cuda()] = 2
    pix = cls[_pixel_tiles(B, H, W)]
    what = "bg_fill C%d B%d %dx%d" % (C, B, H, W)
    _compare(o_hi, _expected(pix, field[0], ostride, C), pix, what + " hi")
    _compare(o_lo, _expected(pix, field[1], ostride, C), pix, what + " lo")


@pytest.mark.timeout(300)
@pytest.mark.parametrize("geom", ["lite", "fhd"])
def test_separate_fill_equals_fused_fill(dense, product, geom):
    """b2s_rpn_bg_fill followed by a work-list launch without a background list (B2S_RPN_BG_FILL=separate) writes the
    same bits as one launch whose epilogue warps fill."""
    L, lib = product._lib, product._lib.load()
    B, H, W = GEOMS[geom]
    d = dense(B, H, W, 128)
    work, bg = _lists("planner", B, H, W, np.random.default_rng(5))
    _, _, nt = _tiles(B, H, W)
    field = _field((H + 2, W + 2, 128), seed=11)
    wl, bl = _list(work, nt), _list(bg, nt)
    fused = d.launch(wl, bl, field)
    sep = d.planes()
    L.check(lib.b2s_rpn_bg_fill(L.ptr(bl[0]), L.ptr(bl[1]), B, H, W, 128, L.ptr(field[0]), L.ptr(field[1]),
                                L.ptr(sep[0]), L.ptr(sep[1]), d.ostride, L.stream()), "b2s_rpn_bg_fill")
    sep = d.launch(wl, None, (None, None), out=sep)
    for a, b in zip(fused, sep):
        assert torch.equal(a.view(torch.int16), b.view(torch.int16))


# ---------------------------------------------------------------- 3. b2s_rpn_bg_plan at scale
PLAN_GEOMS = [(8, 200, 176), (32, 200, 176), (16, 160, 132), (2, 5, 7)]
PATTERNS = ["empty", "full", "random", "corners", "last-frame"]


def _pattern(name, B, H, W, rng):
    occ = np.zeros((B, H, W), np.uint8)
    if name == "full":
        occ[:] = 1
    elif name == "random":
        occ = (rng.random((B, H, W)) < 0.002).astype(np.uint8)
    elif name == "corners":
        occ[:, 0, 0] = occ[:, 0, -1] = occ[:, -1, 0] = occ[:, -1, -1] = 1
    elif name == "last-frame":
        occ[-1] = rng.random((H, W)) < 0.002
        occ[-1, H // 2, W // 2] = 1
    return occ


def _plan(product, occ, nl):
    L, lib = product._lib, product._lib.load()
    B, H, W = occ.shape
    _, _, nt = _tiles(B, H, W)
    bufs = {"flags": torch.full((max(nl, 1), nt), -1, dtype=torch.int32, device="cuda"),
            "work": torch.full((max(nl, 1), nt), -1, dtype=torch.int32, device="cuda"),
            "bg": torch.full((max(nl, 1), nt), -1, dtype=torch.int32, device="cuda"),
            "counts": torch.full((max(nl, 1), 2), -1, dtype=torch.int32, device="cuda")}
    scratch = torch.zeros(2, B, H, W, dtype=torch.uint8, device="cuda")
    rc = lib.b2s_rpn_bg_plan(L.ptr(torch.from_numpy(occ).cuda()), B, H, W, nl, L.ptr(scratch), L.ptr(bufs["flags"]),
                             L.ptr(bufs["work"]), L.ptr(bufs["bg"]), L.ptr(bufs["counts"]), L.stream())
    torch.cuda.synchronize()
    return rc, {k: v.cpu().numpy() for k, v in bufs.items()}


@pytest.mark.timeout(180)
@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("B,H,W", PLAN_GEOMS)
def test_bg_plan_matches_numpy(product, B, H, W, pattern):
    """flags, counts and both lists of every layer; 1144 and 4576 tiles take two and five 1024-tile compaction passes,
    5 x 7 is smaller than one tile."""
    occ = _pattern(pattern, B, H, W, np.random.default_rng(B * H + len(pattern)))
    _, _, nt = _tiles(B, H, W)
    for nl in (1, 6, 32):
        rc, got = _plan(product, occ, nl)
        assert rc == 0
        ref = bg_plan_numpy(occ, nl)
        for l in range(nl):
            f = ref[l].reshape(-1)
            nw = int(f.sum())
            assert np.array_equal(got["flags"][l], f), (nl, l)
            assert tuple(got["counts"][l]) == (nw, nt - nw), (nl, l)
            assert np.array_equal(got["work"][l, :nw], np.nonzero(f)[0]), (nl, l)
            assert np.array_equal(got["bg"][l, :nt - nw], np.nonzero(f == 0)[0]), (nl, l)
            assert (got["work"][l, nw:] == -1).all() and (got["bg"][l, nt - nw:] == -1).all(), (nl, l)
        if pattern == "empty":
            assert (got["counts"][:, 0] == 0).all()
        if pattern == "full":
            assert (got["counts"][:, 1] == 0).all()
        if pattern == "last-frame":
            assert (got["flags"][:, :nt - nt // B] == 0).all() and (got["counts"][:, 0] > 0).all()


@pytest.mark.timeout(60)
@pytest.mark.parametrize("nl", [0, 33])
def test_bg_plan_refuses_layer_counts_outside_1_to_32(product, nl):
    rc, got = _plan(product, np.ones((2, 40, 21), np.uint8), nl)
    assert rc == -2
    assert (got["counts"] == -1).all() and (got["flags"] == -1).all()


# ---------------------------------------------------------------- 4. the engine at bench scale
def _border_cloud(name):
    """points along the four edges of the point-cloud range: data in the outermost BEV pixels only."""
    from b2second import config
    r = config.get_config(name).point_cloud_range
    rng = np.random.default_rng(7)
    xs = np.arange(r[0] + 0.1, r[3] - 0.1, 0.2)
    ys = np.arange(r[1] + 0.1, r[4] - 0.1, 0.2)
    pts = [np.stack([xs, np.full_like(xs, r[1] + 0.1)], 1), np.stack([xs, np.full_like(xs, r[4] - 0.1)], 1),
           np.stack([np.full_like(ys, r[0] + 0.1), ys], 1), np.stack([np.full_like(ys, r[3] - 0.1), ys], 1)]
    xy = np.concatenate(pts, 0)
    z = rng.uniform(-1.5, -0.5, (xy.shape[0], 1))
    refl = rng.uniform(0.0, 1.0, (xy.shape[0], 1))
    return np.concatenate([xy, z, refl], 1).astype(np.float32)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("name,B", [("car.fhd", 32), ("car.lite", 8)])
def test_engine_background_skip_is_bit_identical_at_scale(product, monkeypatch, name, B):
    """B - 2 real clouds, one empty frame, one frame with data at the BEV border; the skip with the fused fill (CUDA
    graph), with b2s_rpn_bg_fill, and off: bit-identical heads, candidate counts and detections."""
    from b2second import config, models
    from b2second.engine import InferenceEngine
    net = models.build_network(config.get_config(name), product).eval()
    models.synthetic_weights_(net, name, seed=0)
    net = net.cuda()
    clouds = [gu.make_cloud(name, s, 12000 + 400 * s) for s in range(B - 2)]
    clouds.insert(B // 2, np.zeros((0, 4), np.float32))
    clouds.append(_border_cloud(name))
    clouds = [torch.from_numpy(c).cuda() for c in clouds]
    res = {}
    for mode, fill in (("1", "fused"), ("1", "separate"), ("0", "fused")):
        monkeypatch.setenv("B2S_RPN_BG", mode)
        monkeypatch.setenv("B2S_RPN_BG_FILL", fill)
        eng = InferenceEngine(net, batch_size=B, max_points=30000, use_cuda_graph=(fill == "fused"))
        assert bool(eng.bg_idx) == (mode == "1")
        eng.infer(clouds)
        res[mode, fill] = (eng.detections(), eng.tc_heads.clone(), eng.cand_count.clone(), int(eng.status[0].item()),
                           eng.bg_counts.clone() if eng.bg_idx else None, getattr(eng, "bg_tiles", 0))
        del eng
        torch.cuda.empty_cache()
    off = res["0", "fused"]
    assert off[3] == 0
    assert off[0][B // 2]["box3d_lidar"].shape[0] == 0 and sum(d["box3d_lidar"].shape[0] for d in off[0]) > 0
    for key in (("1", "fused"), ("1", "separate")):
        on = res[key]
        assert on[3] == 0, key
        skipped = on[4][:, 1].float() / on[5]
        print("%s B%d %s: skipped tile share per layer %s" % (name, B, key, [round(float(s), 3) for s in skipped]))
        assert float(skipped.min()) > 0.3, skipped
        assert torch.equal(on[1], off[1]), key
        assert torch.equal(on[2], off[2]), key
        for a, b in zip(on[0], off[0]):
            for k in ("box3d_lidar", "scores", "label_preds"):
                assert torch.equal(a[k], b[k]), (key, k)


# ---------------------------------------------------------------- 5. B2S_CONV_V2=0
_V2_RUN = """
import numpy as np, torch
import golden_util as gu
from b2second import config, loader, models
from b2second.engine import InferenceEngine
name = "car.fhd"
net = models.build_network(config.get_config(name), loader.product_spconv()).eval()
models.synthetic_weights_(net, name, seed=0)
net = net.cuda()
eng = InferenceEngine(net, batch_size=3, max_points=30000, use_cuda_graph=False)
clouds = [gu.make_cloud(name, 0, 20000), np.zeros((0, 4), np.float32), gu.make_cloud(name, 1, 29000)]
eng.infer([torch.from_numpy(c).cuda() for c in clouds])
torch.cuda.synchronize()
np.savez(OUT, heads=eng.tc_heads.cpu().numpy(), status=eng.status.cpu().numpy(), bg_layers=np.array(len(eng.bg_idx)),
         v2=np.array([op["v2"] for op in eng.tc_plan]))
"""


def _run_fresh(code, env, timeout=600):
    boot = "import sys; sys.path[:0] = %r\n" % [HERE, REPO, os.path.join(REPO, "second.pytorch_b200")]
    r = subprocess.run([sys.executable, "-c", boot + code], capture_output=True, text=True, timeout=timeout, env=env,
                       cwd=REPO)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.timeout(900)
def test_engine_with_conv_v2_off_runs_without_background_tiles(tmp_path):
    """B2S_CONV_V2=0 is read once per process by the library: each engine runs in a fresh interpreter.  With the switch
    the six 3x3 layers run on k_conv_tc, which takes no tile lists, so the plan marks no op v2 and tracks no background
    layer; its heads are within 1e-4 of the default build's (two kernels: not bit-identical)."""
    base = {k: v for k, v in os.environ.items() if k != "B2S_CONV_V2"}
    out = {}
    for v2 in ("0", None):
        path = str(tmp_path / ("v2_%s.npz" % v2))
        _run_fresh("OUT = %r\n" % path + _V2_RUN, dict(base, B2S_CONV_V2=v2) if v2 else base)
        out[v2] = np.load(path)
    off, on = out["0"], out[None]
    assert int(off["status"][0]) == 0 and int(on["status"][0]) == 0
    assert int(off["bg_layers"]) == 0 and not off["v2"].any()
    assert int(on["bg_layers"]) == 6 and int(on["v2"].sum()) == 6
    diff = float(np.abs(off["heads"].astype(np.float64) - on["heads"]).max())
    print("ERR B2S_CONV_V2=0 vs default heads: max abs diff %.2e (bar 1e-4)" % diff)
    assert diff <= 1e-4
    assert not np.array_equal(off["heads"], on["heads"]), "B2S_CONV_V2=0 did not change the kernel"
