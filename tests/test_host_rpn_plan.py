"""Host logic of the tensor-core RPN: b2second.tc.plan_rpn turns every BASELINE config's RPNV2 (stride-1/2 blocks,
k = 1/2/4 ConvTranspose2d or strided-Conv2d deblocks, channel concat, 1x1 heads; rpn.py:264-299,469-497) into a
program of b2s_conv2d_tc_ex launches.  Here the program is INTERPRETED on the CPU with torch.conv2d using exactly
the op fields the CUDA entry point receives (kernel, stride, pad, GEMM grid, output sub-grid, channel offset), and
compared with the torch modules -- so the planner and the op semantics are pinned without a GPU."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from b2second import config, loader, models, tc


def interpret(plan, x):
    """x [B, C, H, W] fp32 -> packed heads [B, S, Hh, Wh], executing the ops with plain torch."""
    B = x.shape[0]
    bufs = {"in": x}
    for name, (h, w, c) in plan["buffers"].items():
        bufs[name] = torch.zeros(B, c, h, w)
    hd = plan["heads"]
    bufs["heads"] = torch.zeros(B, hd["stride"], hd["H"], hd["W"])
    for op in plan["ops"]:
        src = bufs[op["src"]]
        assert src.shape[1] == op["cin"] and tuple(src.shape[2:]) == (op["Hin"], op["Win"])
        # fp16 hi/lo planes of the power-of-two pre-scaled weights; op["scale"] carries the inverse scale
        w = (op["w_hi"].float() + op["w_lo"].float())[:, :op["cout"]]      # [taps, cout, cin]
        w = w.reshape(op["kh"], op["kw"], op["cout"], op["cin"]).permute(2, 3, 0, 1)
        y = F.conv2d(src, w, stride=op["stride"], padding=op["pad"])
        assert tuple(y.shape[2:]) == (op["Hg"], op["Wg"])
        if op["scale"] is not None:
            y = y * op["scale"].view(1, -1, 1, 1)
        if op["shift"] is not None:
            y = y + op["shift"].view(1, -1, 1, 1)
        if op["relu"]:
            y = torch.relu(y)
        dst = bufs[op["dst"]]
        assert tuple(dst.shape[2:]) == (op["Hout"], op["Wout"])
        c0 = op["dst_coff"]
        dst[:, c0:c0 + op["cout"], op["off_h"]::op["out_mul"], op["off_w"]::op["out_mul"]] = y
    return bufs["heads"]


@pytest.mark.parametrize("name", list(config.BUILTIN))
def test_rpn_program_semantics_on_cpu(name):
    sp = loader.oracle_spconv()
    cfg = config.get_config(name)
    net = models.build_network(cfg, sp).eval()
    models.synthetic_weights_(net, name, seed=0)
    rpn = net.rpn
    assert tc.supported(rpn)
    H, W = 32, 48
    cin = rpn.blocks[0][1].in_channels
    torch.manual_seed(1)
    x = torch.relu(torch.randn(2, cin, H, W)) * (torch.rand(2, 1, H, W) < 0.2)
    with torch.no_grad():
        feat = rpn.backbone(x)
        heads = [rpn.conv_box(feat), rpn.conv_cls(feat)] + ([rpn.conv_dir_cls(feat)] if rpn._use_direction_classifier else [])
        ref = torch.cat(heads, 1)
        plan = tc.plan_rpn(rpn, H, W)
        got = interpret(plan, x)
    n = ref.shape[1]
    assert tuple(got.shape[2:]) == tuple(ref.shape[2:])
    err = float((got[:, :n] - ref).abs().max())
    assert err <= 2e-5 * max(1.0, float(ref.abs().max())), err
    assert plan["heads"]["offsets"][-1] == n


@pytest.mark.parametrize("name", list(config.BUILTIN))
def test_rpn_program_structure(name):
    sp = loader.oracle_spconv()
    cfg = config.get_config(name)
    net = models.build_network(cfg, sp).eval()
    _, fH, fW = cfg.feature_map_size
    # the BEV map the RPN sees: feature map x the config's downsample factor
    f = cfg.rpn_downsample_factor if hasattr(cfg, "rpn_downsample_factor") else None
    H = int(round(fH * (f if f else np.prod(cfg.rpn_layer_strides) / (cfg.rpn_upsample_strides[-1] if cfg.rpn_upsample_strides else 1))))
    W = int(round(fW * (f if f else np.prod(cfg.rpn_layer_strides) / (cfg.rpn_upsample_strides[-1] if cfg.rpn_upsample_strides else 1))))
    plan = tc.plan_rpn(net.rpn, H, W, dry=True)
    assert (plan["heads"]["H"], plan["heads"]["W"]) == (fH, fW)
    seen = {}
    for op in plan["ops"]:
        assert op["cin"] % 32 == 0 and op["n_pad"] in (32, 64, 128) and op["cout"] <= op["n_pad"] and op["cout"] % 4 == 0
        assert op["kh"] * op["kw"] == op["taps"] <= 16 and op["stride"] in (1, 2, 4) and op["pad"] in (0, 1)
        assert (op["Hg"] - 1) * op["out_mul"] + op["off_h"] < op["Hout"]
        assert (op["Wg"] - 1) * op["out_mul"] + op["off_w"] < op["Wout"]
        if op["kind"] == "deblock" and op["out_mul"] > 1:
            seen.setdefault((op["dst_coff"], op["out_mul"]), set()).add((op["off_h"], op["off_w"]))
    for (coff, s), offs in seen.items():
        assert offs == {(a, c) for a in range(s) for c in range(s)}, "ConvTranspose2d sub-grids must tile the output"
    # every channel of the concat buffer is written exactly once per sub-grid position
    if "cat" in plan["buffers"]:
        ccat = plan["buffers"]["cat"][2]
        cover = np.zeros(ccat, np.int64)
        for op in plan["ops"]:
            if op["dst"] == "cat" and (op["off_h"], op["off_w"]) == (0, 0):
                cover[op["dst_coff"]:op["dst_coff"] + op["cout"]] += 1
        assert (cover == 1).all()


def bg_plan_numpy(occ, num_layers, tile=16):
    """numpy restatement of b2s_rpn_bg_plan (csrc/rpn_bg.cu): per layer the [B, tiles_h, tiles_w] flags (1 = the tile
    has a pixel whose receptive field holds data) after dilating the data mask by one pixel per layer."""
    B, H, W = occ.shape
    th, tw = -(-H // tile), -(-W // tile)
    cur = occ.astype(bool)
    flags = []
    for l in range(num_layers):
        pad = np.pad(cur, ((0, 0), (1, 1), (1, 1)), constant_values=False)
        out = np.zeros_like(cur)
        for dy in range(3):
            for dx in range(3):
                out |= pad[:, dy:dy + H, dx:dx + W]
        # partial last tiles: the pixels past the image are False
        full = np.pad(out, ((0, 0), (0, th * tile - H), (0, tw * tile - W)), constant_values=False)
        flags.append(full.reshape(B, th, tile, tw, tile).any(axis=(2, 4)).astype(np.int32))
        cur = out
    return flags


@pytest.mark.parametrize("name", ["car.fhd", "car.lite"])
def test_background_tiles_hold_the_empty_frame_response(name):
    """The theory behind the RPN background-tile skip (csrc/rpn_bg.cu), checked against the torch modules: wherever
    the planner says a 16x16 output tile of layer l is background, the dense fp32 computation on the data yields
    exactly what it yields on an EMPTY frame at the same pixels -- in the interior (a constant) and along the image
    border (where the zero padding is felt)."""
    sp = loader.oracle_spconv()
    net = models.build_network(config.get_config(name), sp).eval()
    models.synthetic_weights_(net, name, seed=0)
    rpn = net.rpn
    H, W = 72, 88
    plan = tc.plan_rpn(rpn, H, W)
    idx = tc.background_layers(plan)
    assert len(idx) >= 4
    cin = plan["in_channels"]
    torch.manual_seed(3)
    occ = torch.zeros(2, H, W, dtype=torch.bool)
    occ[0, 20:30, 40:52] = True                       # a blob in the middle, far from the border
    occ[1, 0:5, 10:20] = True                         # blobs touching the border
    occ[1, 60:64, 0:3] = True
    occ[1, 35, 80] = True
    x = torch.relu(torch.randn(2, cin, H, W)) * occ[:, None].float()
    flags = bg_plan_numpy(occ.numpy(), len(idx))
    mods = [m for m in rpn.blocks[0].children()]
    cur, empty, li, i = x, torch.zeros(1, cin, H, W), 0, 0
    with torch.no_grad():
        while i < len(mods) and li < len(idx):
            m = mods[i]
            step = 4 if isinstance(m, torch.nn.ZeroPad2d) else 3
            for mm in mods[i:i + step]:
                cur, empty = mm(cur), mm(empty)
            i += step
            f = flags[li]
            n_bg = n_border = 0
            for b in range(2):
                for th in range(f.shape[1]):
                    for tw in range(f.shape[2]):
                        if f[b, th, tw]:
                            continue
                        n_bg += 1
                        n_border += th == 0 or tw == 0 or th == f.shape[1] - 1 or tw == f.shape[2] - 1
                        sl = (slice(None), slice(th * 16, (th + 1) * 16), slice(tw * 16, (tw + 1) * 16))
                        assert torch.equal(cur[b][sl], empty[0][sl]), (li, b, th, tw)
            assert n_bg > 0 and n_border > 0                # incl. border tiles, which hold a non-constant field
            assert int(f.sum()) > 0
            li += 1
    # the empty-frame response is a constant in the interior and differs near the border from layer 2 on
    inner = empty[0, :, 8:-8, 8:-8]
    assert float((inner - inner[:, :1, :1]).abs().max()) == 0.0
    assert float((empty[0, :, 0, 0] - inner[:, 0, 0]).abs().max()) > 0.0


@pytest.mark.parametrize("switch,want", [(None, 6), ("1", 6), ("0", 0)])
def test_conv_v2_switch_reaches_the_plan(monkeypatch, switch, want):
    """B2S_CONV_V2=0 sends the 3x3 stride-1 layers to k_conv_tc, which refuses tile lists (conv_tc.cu): the plan must
    then mark no op v2 and track no background layer, or the engine would pass lists the library rejects."""
    if switch is None:
        monkeypatch.delenv("B2S_CONV_V2", raising=False)
    else:
        monkeypatch.setenv("B2S_CONV_V2", switch)
    net = models.build_network(config.get_config("car.fhd"), loader.oracle_spconv()).eval()
    plan = tc.plan_rpn(net.rpn, 200, 176, dry=True)
    assert sum(op["v2"] for op in plan["ops"]) == want
    assert len(tc.background_layers(plan)) == want


def test_fused_tail_is_taken_exactly_where_the_program_has_that_shape():
    """b2s_rpn_tail_tc replaces the last two ops only for a single k = s = 1 deblock 128 -> 128 feeding <= 32 packed head
    channels (car.fhd, car.lite); the dispatch is host logic (b2second.tc.fusable_tail) and pinned here for every BASELINE config."""
    sp = loader.oracle_spconv()
    want = {"car.fhd": True, "car.lite": True}        # all.fhd packs 104 head channels, the pillar RPNs are multi-scale
    for name in config.BUILTIN:
        cfg = config.get_config(name)
        net = models.build_network(cfg, sp).eval()
        plan = tc.plan_rpn(net.rpn, 32, 48)
        assert tc.fusable_tail(plan) == want.get(name, False), name
        if tc.fusable_tail(plan):
            d, h = plan["ops"][-2], plan["ops"][-1]
            # what the fused kernel is handed: the deblock as a 1x1 conv [1][128][128], the heads padded to 32 rows
            assert tuple(d["w_hi"].shape) == (1, 128, 128) and tuple(h["w_hi"].shape) == (1, 32, 128)
            assert d["shift"] is not None and h["shift"] is not None and h["cout"] % 4 == 0
            assert plan["heads"]["stride"] >= h["cout"]
