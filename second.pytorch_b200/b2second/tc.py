"""Host side of the tensor-core kernels (csrc/conv_tc.cu, conv_tc2.cu, sparse_conv_tc.cu): 3xF16 weight
preparation and the RPN layer plan.

RPNV2 for the sparse-conv configs (second/pytorch/models/rpn.py:467-497 with layer_strides [1], upsample
strides [1]) is: 6 x [Conv3x3 pad1 + BN + ReLU] -> deblock ConvTranspose2d(k=1,s=1) + BN + ReLU -> three 1x1
heads.  Each becomes one b2s_conv2d_tc launch on NHWC halo-padded fp16 hi/lo planes; the three heads are one launch
writing a packed 32-float record per pixel (box | cls | dir | pad) that b2s_decode_filter_strided reads.
"""
import os

import numpy as np
import torch
from torch import nn


def pow2_scale(w):
    """power of two s with max|w| * s in (2^12, 2^13]: fp16 keeps 11 significant bits down to 2^-14, so after this
    scaling the lo plane of every weight above 2^-17 of the largest one is a NORMAL fp16 (full 22-bit split);
    2^13 leaves three binades of head-room below the fp16 maximum.  The kernels multiply by 1/s in the epilogue."""
    m = float(w.detach().abs().max()) if w.numel() else 0.0
    if not np.isfinite(m) or m <= 0.0:
        return 1.0
    return float(2.0 ** (13 - int(np.ceil(np.log2(m)))))


def split_f16(t, scale=1.0):
    """fp32 tensor -> (hi, lo) torch.float16 planes of t*scale: hi = fp16(t*scale), lo = fp16(t*scale - hi)
    (3xF16 split, csrc/tc_common.cuh; the device-side counterpart is b2s_split_f16)."""
    t = t.detach().float().contiguous() * float(scale)
    hi = t.clamp(-65504.0, 65504.0).half()
    lo = (t - hi.float()).clamp(-65504.0, 65504.0).half()
    return hi.contiguous(), lo.contiguous()


def merge_f16(hi, lo):
    return hi.float() + lo.float()


SPARSE_TC_CIN = (8, 16, 32, 64)      # 3 or 4 input features are zero-padded to 8 (one 16-byte row chunk)
SPARSE_TC_COUT = (16, 32, 64)
SPARSE_BLOCK_K = 64                  # fp16 channels per 128-byte K block


def sparse_tc_cin(cin):
    """channel count the tensor-core sparse kernel sees for a layer with `cin` inputs (None: not covered)."""
    if cin in SPARSE_TC_CIN:
        return cin
    if cin < 8:
        return 8
    return None


def pack_sparse_weights(w):
    """spconv weight [K, Cin, Cout] -> the K-major B operand b2s_sparse_conv_tc expects (fp32, before the split).
    Cin is zero-padded to sparse_tc_cin(Cin).  Cin = 64: [K, Cout, 64].  Cin < 64: PACK = 64/Cin kernel offsets
    share one 128-byte K block, rows packed [ceil(K/PACK), Cout, 64] with column (offset-in-pack * Cin + cin) and
    zero columns past K."""
    K, cin0, cout = w.shape
    cin = sparse_tc_cin(cin0)
    assert cin is not None, "Cin %d is not covered by the tensor-core sparse kernel" % cin0
    wt = torch.zeros(K, cout, cin, dtype=torch.float32, device=w.device)
    wt[:, :, :cin0] = w.detach().float().transpose(1, 2)               # [K, Cout, Cin]
    if cin >= SPARSE_BLOCK_K:
        return wt.contiguous()
    pack = SPARSE_BLOCK_K // cin
    nkb = (K + pack - 1) // pack
    out = torch.zeros(nkb * pack, cout, cin, dtype=wt.dtype, device=wt.device)
    out[:K] = wt
    return out.view(nkb, pack, cout, cin).permute(0, 2, 1, 3).reshape(nkb, cout, SPARSE_BLOCK_K).contiguous()


def _fold_bn2d(bn):
    scale = (bn.weight / torch.sqrt(bn.running_var + bn.eps)).detach().float().contiguous()
    shift = (bn.bias - bn.running_mean * scale).detach().float().contiguous()
    return scale, shift


def _pad_rows(w, n_pad):
    """[taps, Cout, Cin] -> [taps, n_pad, Cin] (zero rows)."""
    taps, cout, cin = w.shape
    if cout == n_pad:
        return w.contiguous()
    out = torch.zeros(taps, n_pad, cin, dtype=w.dtype, device=w.device)
    out[:, :cout] = w
    return out.contiguous()


def _n_pad(cout):
    for n in (32, 64, 128):
        if cout <= n:
            return n
    raise ValueError("Cout %d > 128 not supported by the tensor-core RPN" % cout)


def supported(rpn):
    """True when every layer of this RPNV2 maps onto b2s_conv2d_tc_ex (channels % 64 == 0, kernels <= 4x4)."""
    try:
        plan_rpn(rpn, 64, 64, dry=True)
        return True
    except (ValueError, AssertionError):
        return False


def _conv_out(n, k, s, pad):
    return (n + 2 * pad - k) // s + 1


def conv_v2_enabled():
    """the switch the library's dispatch reads (conv_tc.cu, once per process): B2S_CONV_V2 starting with "0" sends the
    3x3 stride-1 layers to k_conv_tc, which takes no tile lists."""
    return not os.environ.get("B2S_CONV_V2", "").startswith("0")


def plan_rpn(rpn, H, W, dry=False):
    """RPNV2 (second/pytorch/models/rpn.py:469-497 blocks, :264-299 deblocks, :386-420 heads) on an H x W BEV map ->
    {"buffers": {name: (h, w, c)}, "ops": [conv op dicts in execution order], "heads": {...}}.

    Every op is one b2s_conv2d_tc_ex launch: conv k x k / stride / pad, or one (a, c) sub-grid of a k = s
    ConvTranspose2d; output channels are cut into slices of <= 128 (the kernel's n_pad) and `torch.cat` of the
    deblock outputs is a channel offset into the shared "cat" buffer."""
    bufs, ops = {}, []
    use_v2 = conv_v2_enabled()

    def emit(kind, src, dst, w_t_co_ci, kh, kw, stride, pad, scale, shift, relu, hin, win, hg, wg, hout, wout,
             out_mul=1, off=(0, 0), dst_coff=0, planes=2, padded=True):
        taps, cout, cin = w_t_co_ci.shape
        assert taps == kh * kw and cin % 64 == 0, "input channels must be multiples of 64"
        for c0 in range(0, cout, 128):
            c1 = min(cout, c0 + 128)
            n_pad = _n_pad(c1 - c0)
            d = {"kind": kind, "src": src, "dst": dst, "kh": kh, "kw": kw, "taps": taps, "stride": stride, "pad": pad,
                 "cin": cin, "cout": c1 - c0, "n_pad": n_pad, "relu": relu, "Hin": hin, "Win": win, "Hg": hg, "Wg": wg,
                 "Hout": hout, "Wout": wout, "out_mul": out_mul, "off_h": off[0], "off_w": off[1],
                 "dst_coff": dst_coff + c0, "planes": planes, "padded": padded,
                 "shift": None if shift is None else shift[c0:c1].float().contiguous(),
                 # the weights-stationary N=256 kernel takes this op (conv_tc.cu dispatch)
                 "v2": (use_v2 and kh == 3 and kw == 3 and stride == 1 and pad == 1 and n_pad == 128 and planes == 2
                        and padded and out_mul == 1)}
            if not dry:
                # weights pre-scaled by a power of two (exact), undone by the epilogue scale
                wp = _pad_rows(w_t_co_ci[:, c0:c1].float(), n_pad)
                ws = pow2_scale(wp)
                d["w_hi"], d["w_lo"] = split_f16(wp, ws)
                d["w_scale"] = ws
                base = torch.ones(c1 - c0, dtype=torch.float32, device=wp.device) if scale is None \
                    else scale[c0:c1].float()
                d["scale"] = (base / ws).contiguous()
            ops.append(d)

    cur, h, w = "in", H, W
    ups = []                                   # (buffer, channels) of each deblock output, in order
    up_start = rpn._upsample_start_idx
    cat_hw = None
    up_filters = [list(db.children())[0].out_channels for db in rpn.deblocks]
    for bi, block in enumerate(rpn.blocks):
        mods = list(block.children())
        i, li = 0, 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, nn.ZeroPad2d):
                assert tuple(m.padding) == (1, 1, 1, 1)
                conv, bn, relu = mods[i + 1], mods[i + 2], mods[i + 3]
                assert conv.padding == (0, 0)
                i += 4
            else:
                conv, bn, relu = mods[i], mods[i + 1], mods[i + 2]
                assert conv.padding == (1, 1)
                i += 3
            assert isinstance(conv, nn.Conv2d) and conv.kernel_size == (3, 3) and conv.bias is None
            assert conv.stride[0] == conv.stride[1] and conv.stride[0] in (1, 2, 4)
            assert isinstance(bn, nn.BatchNorm2d) and isinstance(relu, nn.ReLU)
            st = conv.stride[0]
            wt = conv.weight.detach()                                   # [Cout, Cin, 3, 3]
            wt = wt.permute(2, 3, 0, 1).reshape(9, wt.shape[0], wt.shape[1])   # [tap=ky*3+kx, Cout, Cin]
            sc, sh = _fold_bn2d(bn)
            ho, wo = _conv_out(h, 3, st, 1), _conv_out(w, 3, st, 1)
            dst = "b%d%s" % (bi, "ab"[li % 2])
            bufs[dst] = (ho, wo, wt.shape[1])
            emit("block", cur, dst, wt, 3, 3, st, 1, sc, sh, True, h, w, ho, wo, ho, wo)
            cur, h, w = dst, ho, wo
            li += 1
        j = bi - up_start
        if j >= 0:
            up, bn, relu = list(rpn.deblocks[j].children())
            assert up.bias is None and isinstance(bn, nn.BatchNorm2d)
            sc, sh = _fold_bn2d(bn)
            coff = sum(up_filters[:j])
            k = up.kernel_size[0]
            assert up.kernel_size == (k, k) and up.stride == (k, k) and k in (1, 2, 4)
            if isinstance(up, nn.ConvTranspose2d):
                hu, wu = h * k, w * k
                if cat_hw is None:
                    cat_hw = (hu, wu)
                assert cat_hw == (hu, wu), "deblock outputs must share one resolution"
                wt = up.weight.detach()                                  # [Cin, Cout, k, k]
                for a in range(k):
                    for c in range(k):
                        emit("deblock", cur, "cat", wt[:, :, a, c].t().unsqueeze(0).contiguous(), 1, 1, 1, 0, sc, sh, True,
                             h, w, h, w, hu, wu, out_mul=k, off=(a, c), dst_coff=coff)
            else:                                                        # Conv2d(k, stride k): upsample_stride < 1
                hu, wu = _conv_out(h, k, k, 0), _conv_out(w, k, k, 0)
                if cat_hw is None:
                    cat_hw = (hu, wu)
                assert cat_hw == (hu, wu), "deblock outputs must share one resolution"
                wt = up.weight.detach()                                  # [Cout, Cin, k, k]
                wt = wt.permute(2, 3, 0, 1).reshape(k * k, wt.shape[0], wt.shape[1])
                emit("deblock", cur, "cat", wt, k, k, k, 0, sc, sh, True, h, w, hu, wu, hu, wu, dst_coff=coff)
            ups.append(up_filters[j])
    if ups:
        bufs["cat"] = (cat_hw[0], cat_hw[1], sum(ups))
        cur, h, w = "cat", cat_hw[0], cat_hw[1]
    # heads: box | cls | dir packed into one record per pixel, bias as shift
    heads = [rpn.conv_box, rpn.conv_cls] + ([rpn.conv_dir_cls] if rpn._use_direction_classifier else [])
    wt = torch.cat([hd.weight.detach()[:, :, 0, 0] for hd in heads], 0).unsqueeze(0)     # [1, sum Cout, Cin]
    bias = torch.cat([hd.bias.detach() for hd in heads], 0).float().contiguous()
    pad = (-wt.shape[1]) % 4
    if pad:
        wt = torch.cat([wt, torch.zeros(1, pad, wt.shape[2], device=wt.device, dtype=wt.dtype)], 1)
        bias = torch.cat([bias, torch.zeros(pad, device=bias.device)])
    stride_s = max(32, wt.shape[1])
    emit("heads", cur, "heads", wt.contiguous(), 1, 1, 1, 0, None, bias, False, h, w, h, w, h, w, planes=1, padded=False)
    offs = np.cumsum([0] + [hd.weight.shape[0] for hd in heads]).tolist()
    return {"buffers": bufs, "ops": ops, "in_channels": ops[0]["cin"],
            "heads": {"offsets": offs, "stride": stride_s, "H": h, "W": w}}


def fusable_tail(plan):
    """True when the program ends with ONE k = s = 1 deblock 128 -> 128 (+BN+ReLU) whose output only feeds the packed heads
    (<= 32 channels): the shape b2s_rpn_tail_tc runs as a single kernel (car.fhd, car.lite; all.fhd packs 104 head
    channels, the multi-scale RPNs concatenate several deblocks)."""
    ops = plan["ops"]
    if len(ops) < 2:
        return False
    d, h = ops[-2], ops[-1]
    return bool(h["kind"] == "heads" and d["kind"] == "deblock" and h["src"] == d["dst"]
                and sum(1 for o in ops if o["dst"] == d["dst"]) == 1
                and (d["kh"], d["kw"], d["stride"], d["out_mul"], d["dst_coff"]) == (1, 1, 1, 1, 0)
                and d["cin"] == 128 and d["cout"] == 128 and d["relu"] and d["planes"] == 2
                and h["cin"] == 128 and h["n_pad"] == 32 and h["planes"] == 1 and not h["relu"])


def background_layers(plan):
    """indices of the leading ops of an RPN program that form a chain of 3x3 stride-1 pad-1 128-out layers starting at
    the BEV input (the ops the weights-stationary kernel takes): background tiles are only tracked through those."""
    idx, src = [], "in"
    for i, op in enumerate(plan["ops"]):
        if op["v2"] and op["src"] == src and op["dst_coff"] == 0 and op["cout"] == op["n_pad"]:
            idx.append(i)
            src = op["dst"]
        else:
            break
    return idx
