"""Error model of the 3xF16 tensor-core kernels, and the accuracy bars the per-form GPU tests hold them to.

Every fp32 operand x travels as two fp16 planes hi = fp16(x), lo = fp16(x - hi); the kernels issue hi*hi + lo*hi + hi*lo
per product with fp32 accumulation (include/b2second.h).  Emulated here in float64 on the SAME shapes and data the
GPU tests use (tests/test_gpu_tc_forms.py imports the constants, shapes and generators from this file):

  * all three products: the only error left is the dropped lo*lo term, ~2^-22 relative -- far under the bars;
  * one cross term dropped, or hi*hi only (plain fp16): ~2^-11 relative -- far over them.

So a bar that passes the first and fails the others can tell a correct kernel from one that lost a product.  The GPU
kernel adds fp32 accumulation and epilogue rounding on top of the emulated error (DESIGN.md §4: max-rel ~1e-6), which
is what the head-room between the emulated three-product error and the bar is for."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

# |err| <= MAX_REL * max|ref| and rms(err) <= RMS_REL * rms(ref) over the region a launch writes; ref is float64 on the
# operands the kernel receives (hi + lo of inputs and weights, fp32 scale and shift)
DENSE_MAX_REL, DENSE_RMS_REL = 4e-6, 2e-6
SPARSE_MAX_REL, SPARSE_RMS_REL = 4e-6, 2e-6
MARGIN = 10.0                      # the emulated three-product error sits this far under a bar, a dropped term this far over

CONFIGS = ("car.fhd", "all.fhd", "car.lite", "pointpillars.car.xyres_16", "nuscenes.all.pp.largea")
FORM_KEYS = ("kh", "kw", "stride", "pad", "cin", "n_pad", "out_mul", "planes", "padded", "v2")
AWKWARD = (3, 13, 21)              # B, Hg, Wg: three frames, a grid that is no multiple of the 8 / 16-pixel tiles
# product terms: hh = x_hi*w_hi, lh = x_lo*w_hi, hl = x_hi*w_lo, ll = x_lo*w_lo (the one the kernels drop)
VARIANTS = {"three products": ("hh", "lh", "hl"), "x_lo*w_hi dropped": ("hh", "hl"),
            "x_hi*w_lo dropped": ("hh", "lh"), "hi*hi only": ("hh",)}


def _net(name):
    from b2second import config, loader, models
    net = models.build_network(config.get_config(name), loader.oracle_spconv()).eval()
    models.synthetic_weights_(net, name, seed=0)
    return net


def bev_hw(name, net=None):
    """H, W of the BEV map the RPN of config `name` runs on."""
    from b2second import loader, spec
    s = spec.spec_from_module(net if net is not None else _net(name), None)
    shape = list(s.sparse_shape)
    ops = loader.oracle_spconv().ops
    for ls in ([] if s.is_pillars else s.layers):
        if not ls["subm"]:
            shape = ops.get_conv_output_size(shape, ls["kernel_size"], ls["stride"], ls["padding"], ls["dilation"])
    return shape[1], shape[2]


def plan_forms():
    """{form: first op of that form in config order} over tc.plan_rpn of every config at its real BEV size; the op dict
    gains "config" and "out_stride" (channels per pixel of the buffer it writes)."""
    from b2second import tc
    forms = {}
    for name in CONFIGS:
        net = _net(name)
        H, W = bev_hw(name, net)
        plan = tc.plan_rpn(net.rpn, H, W, dry=True)
        for op in plan["ops"]:
            f = tuple(op[k] for k in FORM_KEYS)
            if f not in forms:
                stride = plan["heads"]["stride"] if op["dst"] == "heads" else plan["buffers"][op["dst"]][2]
                forms[f] = dict(op, config=name, out_stride=stride)
    return forms


def form_geometry(form, Hg, Wg):
    """(Hin, Win, Hout, Wout) of a launch of `form` on an Hg x Wg GEMM grid."""
    kh, kw, stride, pad, _, _, out_mul, _, _, _ = form
    if out_mul > 1:                                       # ConvTranspose2d(k = s) sub-grid: 1x1 on the input grid
        return Hg, Wg, Hg * out_mul, Wg * out_mul
    if pad == 1:                                          # 3x3 pad 1, stride 1 or 2 (after ZeroPad2d)
        return Hg * stride, Wg * stride, Hg, Wg
    # Conv2d(k, stride k) / 1x1: the input may carry k-1 trailing pixels the conv never reads
    return Hg * stride + (kh - 1), Wg * stride + (kw - 1), Hg, Wg


def form_seed(form):
    return sum((i + 1) * int(v) for i, v in enumerate(form))


def log_uniform(g, shape, lo=-10.0, hi=8.0, zero_frac=0.0):
    """values of magnitude 2^U(lo, hi), random sign, and a fraction of exact zeros (fp32, CPU)."""
    mag = torch.exp2(torch.rand(shape, generator=g, dtype=torch.float64) * (hi - lo) + lo)
    sign = torch.where(torch.rand(shape, generator=g) < 0.5, -1.0, 1.0).double()
    keep = (torch.rand(shape, generator=g) >= zero_frac).double()
    return (mag * sign * keep).float()


def dense_operands(form, B, Hin, Win, cout, seed):
    """CPU operands of one dense launch: x [B, Cin, Hin, Win] spanning 2^-10 .. 2^8 (negatives, zeros: sparse BEV maps),
    w [taps, Cout, Cin], per-channel scale / shift (the shift puts many outputs near the ReLU kink)."""
    kh, kw, _, _, cin = form[:5]
    g = torch.Generator().manual_seed(seed)
    x = log_uniform(g, (B, cin, Hin, Win), zero_frac=0.3)
    w = torch.randn(kh * kw, cout, cin, generator=g) * (2.0 / (kh * kw * cin)) ** 0.5
    scale = torch.rand(cout, generator=g) + 0.5
    shift = torch.randn(cout, generator=g) * 0.5
    return x, w, scale, shift


def dense_planes(x, w, n_pad):
    """the kernel's operands: NHWC halo-padded hi/lo input planes, [taps, n_pad, Cin] weight planes pre-scaled by
    tc.pow2_scale, and that scale."""
    from b2second import tc
    hi, lo = tc.split_f16(F.pad(x.permute(0, 2, 3, 1), (0, 0, 1, 1, 1, 1)))
    wp = tc._pad_rows(w, n_pad)
    ws = tc.pow2_scale(wp)
    w_hi, w_lo = tc.split_f16(wp, ws)
    return hi, lo, w_hi, w_lo, ws


def dense_terms(x_hi, x_lo, w_hi, w_lo, form, cout):
    """float64 products {hh, lh, hl, ll} [B, Cout, Hg, Wg] of the GEMM grid (before scale / shift); x_* are the padded
    NHWC planes, w_* the [taps, n_pad, Cin] planes."""
    kh, kw, stride, pad = form[:4]
    xs = {"h": x_hi[:, 1:-1, 1:-1].permute(0, 3, 1, 2).double(), "l": x_lo[:, 1:-1, 1:-1].permute(0, 3, 1, 2).double()}
    ws = {}
    for n, t in (("h", w_hi), ("l", w_lo)):
        ws[n] = t[:, :cout].double().reshape(kh, kw, cout, -1).permute(2, 3, 0, 1).contiguous()
    return {a + b: F.conv2d(xs[a], ws[b], stride=stride, padding=pad) for a in "hl" for b in "hl"}


def epilogue(v, scale_k, shift, relu, dim=1):
    shape = [1] * v.dim()
    shape[dim] = -1
    y = v * scale_k.double().view(shape) + shift.double().view(shape)
    return torch.relu(y) if relu else y


def rel_errors(got, ref):
    """(max err / max|ref|, rms err / rms ref) in float64."""
    d = (got.double() - ref.double()).abs()
    return (float(d.max() / ref.abs().max().clamp_min(1e-300)),
            float(d.pow(2).mean().sqrt() / ref.pow(2).mean().sqrt().clamp_min(1e-300)))


# ---------------------------------------------------------------- sparse
SPARSE_CIN, SPARSE_COUT = (3, 4, 8, 16, 32, 64), (16, 32, 64)


def sparse_widths():
    """every (Cin, Cout) the tensor-core sparse kernel is built for (3 / 4 input features are padded to 8)."""
    from b2second import tc
    return [(ci, co) for ci in SPARSE_CIN for co in SPARSE_COUT
            if tc.sparse_tc_cin(ci) in tc.SPARSE_TC_CIN and co in tc.SPARSE_TC_COUT]


def sparse_operands(cin, cout, K, n_out, rows_in, seed, fill=0.45):
    """CPU operands of one sparse launch: features [rows_in, Cin] spanning 2^-10 .. 2^8, a neighbour table [n_out, K]
    (each entry an input row with probability `fill`, else -1; for odd K the centre is row o mod rows_in, as in a
    SubM table), weights [K, Cin, Cout], scale, shift."""
    g = torch.Generator().manual_seed(seed)
    feats = log_uniform(g, (rows_in, cin))
    nbr = torch.randint(0, rows_in, (n_out, K), generator=g, dtype=torch.int32)
    nbr[torch.rand(n_out, K, generator=g) >= fill] = -1
    if K % 2 == 1 and K > 1:
        nbr[:, K // 2] = (torch.arange(n_out) % rows_in).int()
    w = torch.randn(K, cin, cout, generator=g) * (2.0 / (K * cin * fill)) ** 0.5
    scale = torch.rand(cout, generator=g) + 0.5
    shift = torch.randn(cout, generator=g) * 0.5
    return feats, nbr, w, scale, shift


def sparse_terms(f_hi, f_lo, w_hi, w_lo, nbr):
    """float64 products {hh, lh, hl, ll} [n_out, Cout] of the gather-GEMM over nbr (f_* [rows_in, Cin], w_* [K, Cin,
    Cout], any device)."""
    n_out, K = nbr.shape
    idx = nbr.long().clamp_min(0)
    ok = (nbr >= 0).double().unsqueeze(-1)
    out = {}
    for a, fa in (("h", f_hi), ("l", f_lo)):
        gathered = fa.double()[idx] * ok                                   # [n_out, K, Cin]
        for b, wb in (("h", w_hi), ("l", w_lo)):
            out[a + b] = torch.einsum("okc,kcd->od", gathered, wb.double())
    return out


# ---------------------------------------------------------------- the checks
def _assert_bars(terms, scale_k, shift, relu, max_bar, rms_bar, what, dim=1):
    ref = epilogue(sum(terms.values()), scale_k, shift, relu, dim)
    errs = {}
    for name, keys in VARIANTS.items():
        errs[name] = rel_errors(epilogue(sum(terms[k] for k in keys), scale_k, shift, relu, dim), ref)
    mx, rms = errs["three products"]
    assert mx * MARGIN <= max_bar and rms * MARGIN <= rms_bar, "%s: three products %s vs bars" % (what, errs)
    for name, (mx, rms) in errs.items():
        if name != "three products":
            assert mx >= MARGIN * max_bar and rms >= MARGIN * rms_bar, "%s: %s not caught: %s" % (what, name, errs)


FORMS = plan_forms()
# the forms tests/test_gpu_tc_forms.py launches one by one, as (kh, kw, stride, pad, cin, n_pad, out_mul, planes, padded, v2)
KNOWN_FORMS = [
    (1, 1, 1, 0, 64, 128, 1, 2, True, False), (1, 1, 1, 0, 128, 32, 1, 1, False, False),
    (1, 1, 1, 0, 128, 128, 1, 2, True, False), (1, 1, 1, 0, 128, 128, 2, 2, True, False),
    (1, 1, 1, 0, 256, 128, 1, 1, False, False), (1, 1, 1, 0, 256, 128, 1, 2, True, False),
    (1, 1, 1, 0, 256, 128, 4, 2, True, False), (1, 1, 1, 0, 384, 32, 1, 1, False, False),
    (1, 1, 1, 0, 384, 128, 1, 1, False, False), (2, 2, 2, 0, 128, 128, 1, 2, True, False),
    (3, 3, 1, 1, 64, 64, 1, 2, True, False), (3, 3, 1, 1, 128, 64, 1, 2, True, False),
    (3, 3, 1, 1, 128, 128, 1, 2, True, True), (3, 3, 1, 1, 256, 128, 1, 2, True, True),
    (3, 3, 2, 1, 64, 64, 1, 2, True, False), (3, 3, 2, 1, 64, 128, 1, 2, True, False),
    (3, 3, 2, 1, 128, 128, 1, 2, True, False), (4, 4, 4, 0, 64, 128, 1, 2, True, False)]


def form_id(f):
    return "k%dx%d-s%d-p%d-c%d-n%d-m%d-pl%d-%s" % (f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7], "v2" if f[9] else "v1")


def test_plan_forms_are_the_known_set():
    """the planner emits exactly the forms the per-form GPU tests launch: a new form fails here until it is tested."""
    assert set(FORMS) == set(KNOWN_FORMS), "untested: %s; gone: %s" % (set(FORMS) - set(KNOWN_FORMS),
                                                                        set(KNOWN_FORMS) - set(FORMS))
    for f, op in FORMS.items():
        assert op["cout"] <= op["n_pad"] and op["out_stride"] >= op["dst_coff"] + op["cout"]


@pytest.mark.parametrize("form", KNOWN_FORMS, ids=form_id)
def test_dense_bars_separate_correct_from_dropped_terms(form):
    op = FORMS[form]
    B, Hg, Wg = AWKWARD
    Hin, Win, _, _ = form_geometry(form, Hg, Wg)
    x, w, scale, shift = dense_operands(form, B, Hin, Win, op["cout"], seed=form_seed(form))
    x_hi, x_lo, w_hi, w_lo, ws = dense_planes(x, w, op["n_pad"])
    terms = dense_terms(x_hi, x_lo, w_hi, w_lo, form, op["cout"])
    assert terms["hh"].shape == (B, op["cout"], Hg, Wg)
    _assert_bars(terms, scale / ws, shift, op["relu"], DENSE_MAX_REL, DENSE_RMS_REL, str(form))


@pytest.mark.parametrize("cin,cout", sparse_widths())
@pytest.mark.parametrize("K", [27, 3])
def test_sparse_bars_separate_correct_from_dropped_terms(cin, cout, K):
    from b2second import tc
    feats, nbr, w, scale, shift = sparse_operands(cin, cout, K, 1000, 1100, seed=cin * 100 + cout + K)
    ws = tc.pow2_scale(w)
    f_hi, f_lo = tc.split_f16(feats)
    w_hi, w_lo = tc.split_f16(w, ws)
    terms = sparse_terms(f_hi, f_lo, w_hi, w_lo, nbr)
    _assert_bars(terms, scale / ws, shift, True, SPARSE_MAX_REL, SPARSE_RMS_REL, "sparse %d->%d K=%d" % (cin, cout, K))


def test_split_planes_are_exact_and_tight():
    """hi + lo keeps 22 significant bits of an fp32 value, down to the fp16 subnormal step 2^-24 of the lo plane (below
    2^-3 an unscaled activation loses bits there -- why the references use hi + lo, not the fp32 value), and
    |lo| <= ulp(hi) / 2."""
    from b2second import tc
    g = torch.Generator().manual_seed(0)
    x = log_uniform(g, (4096,), lo=-10.0, hi=8.0) * 1.0001
    hi, lo = tc.split_f16(x)
    err = (hi.double() + lo.double() - x.double()).abs()
    assert bool((err <= torch.clamp(x.double().abs() * 2.0 ** -22, min=2.0 ** -25)).all())
    assert bool((lo.double().abs() <= half_ulp(hi)).all())


def half_ulp(hi):
    """ulp(hi) / 2 of fp16 values, float64 (2^-25 for zero and subnormals)."""
    m, e = torch.frexp(hi.double())
    h = torch.exp2(e.double() - 12.0)
    return torch.where((hi.double().abs() < 2.0 ** -14), torch.full_like(h, 2.0 ** -25), h)
