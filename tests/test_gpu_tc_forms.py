"""One launch per tensor-core kernel form against float64, and the sparse rulebook chain the engine builds against the
CPU oracle.

Each reference is float64 on the operands the kernel receives (hi + lo planes of inputs and weights, the fp32 scale and
shift), so the only differences left are the kernel's own: the dropped lo*lo term, fp32 accumulation and rounding.  The
bars come from tests/test_tc_error_model.py, which shows on CPU that they pass the three-product split with a 10x
margin and fail a kernel that loses one product by 10x.  Every output buffer starts as NaN: whatever a launch must not
write (halo, other sub-grid pixels, channels outside its slice of the record, rows past the live count) must still hold
that bit pattern afterwards."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from test_tc_error_model import (AWKWARD, DENSE_MAX_REL, DENSE_RMS_REL, FORMS, KNOWN_FORMS, SPARSE_MAX_REL,
                                 SPARSE_RMS_REL, dense_operands, dense_planes, dense_terms, epilogue, form_geometry,
                                 form_id, form_seed, half_ulp, rel_errors, sparse_operands, sparse_terms, sparse_widths)

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
F16_NAN = 0x7E00


def _lib(product):
    return product._lib, product._lib.load()


def _sentinel(shape, dtype):
    return torch.full(shape, float("nan"), dtype=dtype, device="cuda")


def _untouched(buf, mask):
    """every element of `buf` outside `mask` still holds the NaN sentinel bit pattern."""
    if buf.dtype == torch.float16:
        return bool((buf.view(torch.int16)[~mask] == F16_NAN).all())
    return bool(torch.isnan(buf[~mask]).all())


def _check_split(hi, lo):
    """|lo| <= ulp(hi)/2: hi is the fp16 rounding of the value and lo the rounding of the rest."""
    assert bool((lo.double().abs() <= half_ulp(hi)).all()), "lo plane larger than half an ulp of hi"


def _report(what, mx, rms, max_bar, rms_bar):
    print("ERR %-58s max %.2e (%5.1fx under)  rms %.2e (%5.1fx under)" % (what, mx, max_bar / max(mx, 1e-30), rms,
                                                                          rms_bar / max(rms, 1e-30)))
    assert mx <= max_bar and rms <= rms_bar, "%s: max %.3g (bar %.3g), rms %.3g (bar %.3g)" % (what, mx, max_bar, rms,
                                                                                              rms_bar)


# ---------------------------------------------------------------- a. dense forms
def run_dense_form(product, form, B, Hg, Wg, real):
    """one b2s_conv2d_tc_ex launch of `form` on a B x Hg x Wg grid; real=True: the channel slice, record width and
    sub-grid of the planner's op, else a channel offset and record width of our own and the last sub-grid position."""
    L, lib = _lib(product)
    kh, kw, stride, pad, cin, n_pad, out_mul, planes, padded, v2 = form
    op = FORMS[form]
    cout = op["cout"]
    if real:
        Hin, Win, Hout, Wout = op["Hin"], op["Win"], op["Hout"], op["Wout"]
        off_h, off_w, coff, ostride = op["off_h"], op["off_w"], op["dst_coff"], op["out_stride"]
    else:
        Hin, Win, Hout, Wout = form_geometry(form, Hg, Wg)
        off_h, off_w = out_mul - 1, out_mul // 2
        step = 8 if planes == 2 else 4                    # 16 bytes
        coff, ostride = op["dst_coff"] + step, op["out_stride"] + 2 * step
    x, w, scale, shift = dense_operands(form, B, Hin, Win, cout, seed=form_seed(form) + B + Hg)
    x_hi, x_lo, w_hi, w_lo, ws = [t.cuda() if torch.is_tensor(t) else t for t in dense_planes(x, w, n_pad)]
    scale_k, shift = (scale / ws).cuda(), shift.cuda()
    p = 1 if padded else 0
    if planes == 2:
        o_hi = _sentinel((B, Hout + 2 * p, Wout + 2 * p, ostride), torch.float16)
        o_lo = _sentinel(o_hi.shape, torch.float16)
    else:
        o_hi, o_lo = _sentinel((B, Hout + 2 * p, Wout + 2 * p, ostride), torch.float32), None
    esz = o_hi.element_size()
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    L.check(lib.b2s_conv2d_tc_ex(
        L.ptr(x_hi), L.ptr(x_lo), B, Hin, Win, cin, L.ptr(w_hi), L.ptr(w_lo), kh, kw, stride, pad, cout, n_pad,
        L.ptr(scale_k), L.ptr(shift), 1 if op["relu"] else 0, Hg, Wg, o_hi.data_ptr() + esz * coff,
        None if o_lo is None else o_lo.data_ptr() + esz * coff, Hout, Wout, p, ostride, out_mul, off_h, off_w,
        None, None, None, None, None, None, L.ptr(status), L.stream()), "b2s_conv2d_tc_ex")
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    rows = p + off_h + out_mul * torch.arange(Hg, device="cuda")
    cols = p + off_w + out_mul * torch.arange(Wg, device="cuda")
    mask = torch.zeros(o_hi.shape, dtype=torch.bool, device="cuda")
    mask[:, rows[:, None], cols[None, :], coff:coff + cout] = True
    for buf in (o_hi, o_lo):
        if buf is not None:
            assert _untouched(buf, mask), "%s wrote outside its pixels / channels" % form_id(form)
    pick = (lambda t: t[:, rows[:, None], cols[None, :], coff:coff + cout].permute(0, 3, 1, 2))
    got = pick(o_hi).double() + (pick(o_lo).double() if o_lo is not None else 0.0)
    assert bool(torch.isfinite(got).all()), "%s left target pixels unwritten" % form_id(form)
    if o_lo is not None:
        _check_split(pick(o_hi), pick(o_lo))
    terms = dense_terms(x_hi, x_lo, w_hi, w_lo, form, cout)
    ref = epilogue(sum(terms.values()), scale_k, shift, op["relu"])
    return rel_errors(got, ref)


@pytest.mark.timeout(300)
@pytest.mark.parametrize("grid", ["real", "awkward", "one-wide"])
@pytest.mark.parametrize("form", KNOWN_FORMS, ids=form_id)
def test_dense_form_matches_float64(product, form, grid):
    """every form tc.plan_rpn emits (tests/test_tc_error_model.py keeps that list complete): at its config's real grid
    (B = 1), on B = 3 x 13 x 21, and on a one-pixel-wide grid."""
    op = FORMS[form]
    B, Hg, Wg = {"real": (1, op["Hg"], op["Wg"]), "awkward": AWKWARD, "one-wide": (2, 9, 1)}[grid]
    mx, rms = run_dense_form(product, form, B, Hg, Wg, grid == "real")
    _report("dense %s %s B%d %dx%d" % (form_id(form), grid, B, Hg, Wg), mx, rms, DENSE_MAX_REL, DENSE_RMS_REL)


# ---------------------------------------------------------------- c. fused tail
@pytest.mark.timeout(180)
@pytest.mark.parametrize("cout2", [4, 20, 32])
def test_fused_tail_matches_float64_and_two_launches(product, cout2):
    """b2s_rpn_tail_tc with a record wider than the heads and a partial last 128-pixel tile (3 x 7 x 13 = 273 pixels):
    bit-identical to the two b2s_conv2d_tc_ex launches, each layer within the bars of its float64 reference."""
    L, lib = _lib(product)
    form1 = (1, 1, 1, 0, 128, 128, 1, 2, True, False)
    B, H, W = 3, 7, 13
    ostride = cout2 + 12
    x, w1, scale1, shift1 = dense_operands(form1, B, H, W, 128, seed=cout2)
    x_hi, x_lo, w1_hi, w1_lo, ws1 = [t.cuda() if torch.is_tensor(t) else t for t in dense_planes(x, w1, 128)]
    scale1_k, shift1 = (scale1 / ws1).cuda(), shift1.cuda()
    g = torch.Generator().manual_seed(100 + cout2)
    w2 = torch.randn(1, cout2, 128, generator=g) * 0.1
    bias2 = (torch.randn(cout2, generator=g) * 0.5).cuda()
    _, _, w2_hi, w2_lo, ws2 = dense_planes(x[:, :, :1, :1], w2, 32)
    w2_hi, w2_lo = w2_hi.cuda(), w2_lo.cuda()
    scale2_k = (torch.ones(cout2) / ws2).cuda()
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    # two launches: deblock into halo-padded hi/lo planes, heads into a packed fp32 record
    y_hi = torch.zeros(B, H + 2, W + 2, 128, dtype=torch.float16, device="cuda")
    y_lo = torch.zeros_like(y_hi)
    two = _sentinel((B, H, W, ostride), torch.float32)
    L.check(lib.b2s_conv2d_tc(L.ptr(x_hi), L.ptr(x_lo), B, H, W, 128, L.ptr(w1_hi), L.ptr(w1_lo), 1, 128, 128,
                              L.ptr(scale1_k), L.ptr(shift1), 1, L.ptr(y_hi), L.ptr(y_lo), 1, 128, L.ptr(status),
                              L.stream()), "b2s_conv2d_tc")
    L.check(lib.b2s_conv2d_tc(L.ptr(y_hi), L.ptr(y_lo), B, H, W, 128, L.ptr(w2_hi), L.ptr(w2_lo), 1, cout2, 32,
                              L.ptr(scale2_k), L.ptr(bias2), 0, L.ptr(two), None, 0, ostride, L.ptr(status),
                              L.stream()), "b2s_conv2d_tc")
    one = _sentinel((B, H, W, ostride), torch.float32)
    L.check(lib.b2s_rpn_tail_tc(L.ptr(x_hi), L.ptr(x_lo), B, H, W, 128, L.ptr(w1_hi), L.ptr(w1_lo), 128,
                                L.ptr(scale1_k), L.ptr(shift1), L.ptr(w2_hi), L.ptr(w2_lo), cout2, 32, L.ptr(scale2_k),
                                L.ptr(bias2), L.ptr(one), ostride, L.ptr(status), L.stream()), "b2s_rpn_tail_tc")
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    assert torch.equal(one[..., :cout2], two[..., :cout2]), "fused tail differs from the two-launch path"
    assert bool(torch.isnan(one[..., cout2:]).all()) and bool(torch.isnan(two[..., cout2:]).all())
    # deblock layer vs float64 on its operands, then the heads vs float64 on the deblock output they received
    y = (y_hi[:, 1:-1, 1:-1].double() + y_lo[:, 1:-1, 1:-1].double()).permute(0, 3, 1, 2)
    ref1 = epilogue(sum(dense_terms(x_hi, x_lo, w1_hi, w1_lo, form1, 128).values()), scale1_k, shift1, True)
    _report("tail deblock cout2=%d" % cout2, *rel_errors(y, ref1), DENSE_MAX_REL, DENSE_RMS_REL)
    _check_split(y_hi[:, 1:-1, 1:-1], y_lo[:, 1:-1, 1:-1])
    form2 = (1, 1, 1, 0, 128, 32, 1, 1, False, False)
    ref2 = epilogue(sum(dense_terms(y_hi, y_lo, w2_hi, w2_lo, form2, cout2).values()), scale2_k, bias2, False)
    _report("tail heads cout2=%d" % cout2, *rel_errors(one[..., :cout2].permute(0, 3, 1, 2), ref2), DENSE_MAX_REL,
            DENSE_RMS_REL)


# ---------------------------------------------------------------- d. sparse
def run_sparse(product, feats, nbr, w, scale, shift, relu=True, expect_status=0):
    """b2s_sparse_conv_tc_plan over `nbr` with rows_in = feats rows, feature / output records wider than 2*C (NaN in
    the gaps), a row capacity past the live count; returns (got, ref) float64 [n_out, Cout] after checking the
    sentinels and the split."""
    from b2second import tc
    L, lib = _lib(product)
    rows_in, cin = feats.shape
    n_out, K = nbr.shape
    cout = w.shape[2]
    cin_tc = tc.sparse_tc_cin(cin)
    assert lib.b2s_sparse_conv_tc_supported(cin_tc, cout)
    ws = tc.pow2_scale(w)
    wh, wl = tc.split_f16(w, ws)                                         # [K, Cin, Cout]
    w_hi = tc.pack_sparse_weights(wh.float().cuda()).half()             # packing only moves / zero-pads: exact
    w_lo = tc.pack_sparse_weights(wl.float().cuda()).half()
    f_hi, f_lo = tc.split_f16(feats.cuda())
    in_stride = 2 * cin_tc + 8
    fbuf = _sentinel((max(rows_in, 1), in_stride), torch.float16)
    fbuf[:, :cin_tc] = 0
    fbuf[:, cin_tc + 8:] = 0
    fbuf[:rows_in, :cin] = f_hi
    fbuf[:rows_in, cin_tc + 8:cin_tc + 8 + cin] = f_lo
    cap = n_out + 5
    nbr_cap = torch.full((cap, K), -1, dtype=torch.int32, device="cuda")
    nbr_cap[:n_out] = nbr.cuda()
    n_dev = torch.tensor([n_out], dtype=torch.int32, device="cuda")
    out_stride = 2 * cout + 8
    obuf = _sentinel((cap, out_stride), torch.float16)
    scale_k, shift_d = (scale / ws).cuda(), shift.cuda()
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    esz = 2
    L.check(lib.b2s_sparse_conv_tc_plan(
        L.ptr(fbuf), fbuf.data_ptr() + esz * (cin_tc + 8), in_stride, rows_in, cin_tc, L.ptr(w_hi), L.ptr(w_lo),
        L.ptr(nbr_cap), K, L.ptr(n_dev), cap, None, None, L.ptr(scale_k), L.ptr(shift_d), 1 if relu else 0,
        L.ptr(obuf), obuf.data_ptr() + esz * (cout + 8), out_stride, cout, L.ptr(status), L.stream()),
        "b2s_sparse_conv_tc_plan")
    torch.cuda.synchronize()
    assert int(status.item()) == expect_status
    mask = torch.zeros(obuf.shape, dtype=torch.bool, device="cuda")
    mask[:n_out, :cout] = True
    mask[:n_out, cout + 8:] = True
    assert _untouched(obuf, mask), "sparse conv wrote outside its rows / channels"
    o_hi, o_lo = obuf[:n_out, :cout], obuf[:n_out, cout + 8:]
    assert bool(torch.isfinite(o_hi).all() and torch.isfinite(o_lo).all()), "rows left unwritten"
    _check_split(o_hi, o_lo)
    got = o_hi.double() + o_lo.double()
    ref = epilogue(sum(sparse_terms(f_hi, f_lo, wh.cuda(), wl.cuda(), nbr.cuda()).values()), scale_k, shift_d, relu)
    return got, ref


def _sparse_synthetic(product, cin, cout, K, n_out, rows_in):
    feats, nbr, w, scale, shift = sparse_operands(cin, cout, K, n_out, rows_in, seed=cin * 100 + cout + K + n_out)
    got, ref = run_sparse(product, feats, nbr, w, scale, shift)
    _report("sparse %d->%d K=%d n_out=%d rows_in=%d" % (cin, cout, K, n_out, rows_in), *rel_errors(got, ref),
            SPARSE_MAX_REL, SPARSE_RMS_REL)


@pytest.mark.timeout(180)
@pytest.mark.parametrize("cin,cout", sparse_widths())
def test_sparse_widths_match_float64(product, cin, cout):
    """every (Cin, Cout) the kernel is built for, K = 27, 1000 output rows over 1100 input rows."""
    _sparse_synthetic(product, cin, cout, 27, 1000, 1100)


@pytest.mark.timeout(180)
@pytest.mark.parametrize("cin,cout", [(64, 64), (16, 32), (4, 16)])
@pytest.mark.parametrize("n_out", [1, 127, 128, 129, 8200])
def test_sparse_row_counts_match_float64(product, cin, cout, n_out):
    """partial and exactly full 128-row tiles, and more than one 8192-row chunk."""
    _sparse_synthetic(product, cin, cout, 27, n_out, n_out + 37)


@pytest.mark.timeout(180)
@pytest.mark.parametrize("cin,cout", [(64, 64), (16, 32)])
def test_sparse_k3_matches_float64(product, cin, cout):
    """K = 3, the (3,1,1)/(2,1,1) layer; 16 channels: one packed K block holding three of its four offsets."""
    _sparse_synthetic(product, cin, cout, 3, 3000, 2000)


def _random_coords(rng, shape, batch, n):
    D, H, W = shape
    flat = rng.choice(batch * D * H * W, size=n, replace=False)
    b, r = np.divmod(flat, D * H * W)
    z, r = np.divmod(r, H * W)
    y, x = np.divmod(r, W)
    return torch.from_numpy(np.stack([b, z, y, x], 1).astype(np.int32))


@pytest.mark.timeout(180)
@pytest.mark.parametrize("cin,cout,ksize,stride,padding", [
    (16, 32, [3, 3, 3], [2, 2, 2], [1, 1, 1]), (32, 64, [3, 3, 3], [2, 2, 2], [1, 1, 1]),
    (64, 64, [3, 3, 3], [2, 2, 2], [0, 1, 1]), (3, 16, [3, 3, 3], [2, 2, 2], [1, 1, 1]),
    (64, 64, [3, 1, 1], [2, 1, 1], [0, 0, 0]), (16, 32, [3, 1, 1], [2, 1, 1], [0, 0, 0])])
def test_sparse_strided_rulebooks_match_float64(product, cin, cout, ksize, stride, padding):
    """the strided geometries of the five configs on real rulebooks (b2s_rulebook_conv), plus one packed K = 3 case."""
    rng = np.random.default_rng(cin + cout + ksize[1])
    shape, batch = (11, 40, 36), 2
    idx = _random_coords(rng, shape, batch, 6000)
    g = torch.Generator().manual_seed(cin + cout)
    feats = sparse_operands(cin, cout, 1, 1, idx.shape[0], seed=cin)[0]
    x = product.SparseConvTensor(feats.cuda(), idx.cuda(), shape, batch)
    rb = product.ops.build_rulebook(x, ksize, stride, padding, [1, 1, 1], False)
    K = int(np.prod(ksize))
    assert rb.num_out > 128
    w = torch.randn(K, cin, cout, generator=g) * (2.0 / (K * cin)) ** 0.5
    scale, shift = torch.rand(cout, generator=g) + 0.5, torch.randn(cout, generator=g) * 0.5
    got, ref = run_sparse(product, feats, rb.nbr[:rb.num_out].cpu(), w, scale, shift)
    _report("sparse %d->%d k%s s%s p%s rulebook" % (cin, cout, ksize, stride, padding), *rel_errors(got, ref),
            SPARSE_MAX_REL, SPARSE_RMS_REL)


@pytest.mark.timeout(120)
def test_sparse_fp16_range_guard_raises_status(product):
    """an output beyond the fp16 range is clamped to 65504 and reported (B2S_STATUS_F16_RANGE), never inf."""
    from b2second import tc
    L, lib = _lib(product)
    n, K, cin, cout = 300, 27, 64, 64
    f_hi, f_lo = tc.split_f16(torch.full((n, cin), 30.0, device="cuda"))
    w = torch.full((K, cin, cout), 8.0)                               # 27 * 64 * 30 * 8 = 414720 > 65504
    ws = tc.pow2_scale(w)
    w_hi, w_lo = tc.split_f16(tc.pack_sparse_weights(w.cuda()), ws)
    nbr = torch.arange(n, dtype=torch.int32, device="cuda")[:, None].repeat(1, K)
    n_dev = torch.tensor([n], dtype=torch.int32, device="cuda")
    scale = torch.full((cout,), 1.0 / ws, device="cuda")
    o_hi = torch.zeros(n, cout, dtype=torch.float16, device="cuda")
    o_lo = torch.zeros_like(o_hi)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    shift = torch.zeros(cout, device="cuda")
    L.check(lib.b2s_sparse_conv_tc_plan(L.ptr(f_hi), L.ptr(f_lo), cin, n, cin, L.ptr(w_hi), L.ptr(w_lo), L.ptr(nbr), K,
                                        L.ptr(n_dev), n, None, None, L.ptr(scale), L.ptr(shift), 0, L.ptr(o_hi), L.ptr(o_lo),
                                        cout, cout, L.ptr(status), L.stream()), "b2s_sparse_conv_tc_plan")
    torch.cuda.synchronize()
    assert int(status.item()) & 16
    assert bool(torch.isfinite(o_hi.float()).all() and torch.isfinite(o_lo.float()).all())
    assert float(o_hi.float().max()) == 65504.0


# ---------------------------------------------------------------- e. the engine's rulebook chain
def _nbr_from_pairs(pairs, num, n_out):
    K = pairs.shape[0]
    nbr = torch.full((n_out, K), -1, dtype=torch.int32)
    for k in range(K):
        m = int(num[k])
        nbr[pairs[k, 1, :m].long(), k] = pairs[k, 0, :m]
    return nbr


def _row_mask(nbr):
    return ((nbr >= 0).long() << torch.arange(nbr.shape[1])).sum(1)


def _chain_coords(rng, shape, batch, n, empty_frame):
    """random cells plus cells on all six faces of the grid in every non-empty frame."""
    D, H, W = shape
    pts = set()
    frames = [b for b in range(batch) if b != empty_frame]
    for b in frames:
        for _ in range(n):
            pts.add((b, int(rng.integers(D)), int(rng.integers(H)), int(rng.integers(W))))
        for _ in range(6):
            z, y, x = int(rng.integers(D)), int(rng.integers(H)), int(rng.integers(W))
            pts.update({(b, 0, y, x), (b, D - 1, y, x), (b, z, 0, x), (b, z, H - 1, x), (b, z, y, 0), (b, z, y, W - 1)})
    order = rng.permutation(len(pts))                                    # voxelizer rows are not sorted
    arr = np.array(sorted(pts), dtype=np.int32)[order]
    return torch.from_numpy(arr)


class _Chain:
    """b2s_rulebook_conv / b2s_rulebook_subm_ranked calls the way the engine makes them (one shared workspace)."""

    def __init__(self, product, batch, shapes):
        self.L, self.lib = _lib(product)
        self.B = batch
        ws = max(self.lib.b2s_rulebook_conv_workspace_bytes(batch, self.L.i3(s)) for s in shapes)
        self.ws, self.ws_bytes = torch.empty(max(ws, 1), dtype=torch.uint8, device="cuda"), ws
        self.status = torch.zeros(1, dtype=torch.int32, device="cuda")

    def conv(self, coors, n_dev, in_shape, out_shape, k, s, p, cap_out, hash_in=None):
        L = self.L
        coors_out = torch.full((cap_out, 4), -7, dtype=torch.int32, device="cuda")
        n_out = torch.zeros(1, dtype=torch.int32, device="cuda")
        nbr = torch.full((cap_out, int(np.prod(k))), -7, dtype=torch.int32, device="cuda")
        row_mask = torch.full((cap_out,), -7, dtype=torch.int32, device="cuda")
        keys, vals, hcap = hash_in if hash_in is not None else (None, None, 0)
        L.check(self.lib.b2s_rulebook_conv(
            L.ptr(coors), L.ptr(n_dev), coors.shape[0], self.B, L.i3(in_shape), L.i3(out_shape), L.i3(k), L.i3(s),
            L.i3(p), L.i3([1, 1, 1]), L.ptr(keys), L.ptr(vals), hcap, L.ptr(coors_out), L.ptr(n_out), cap_out,
            L.ptr(nbr), None, None, 0, L.ptr(self.ws), self.ws_bytes, L.ptr(row_mask), L.ptr(self.status),
            L.stream()), "b2s_rulebook_conv")
        return coors_out, n_out, nbr, row_mask

    def subm_ranked(self, coors, n_dev, shape):
        L = self.L
        cap = coors.shape[0]
        nbr = torch.full((cap, 27), -7, dtype=torch.int32, device="cuda")
        row_mask = torch.full((cap,), -7, dtype=torch.int32, device="cuda")
        L.check(self.lib.b2s_rulebook_subm_ranked(
            L.ptr(coors), L.ptr(n_dev), cap, self.B, L.i3(shape), L.i3([3, 3, 3]), L.i3([1, 1, 1]), L.ptr(self.ws),
            self.ws_bytes, L.ptr(nbr), L.ptr(row_mask), L.stream()), "b2s_rulebook_subm_ranked")
        return nbr, row_mask

    def hash(self, coors, n_dev, shape):
        from b2second.engine import _pow2_at_least
        L = self.L
        hcap = _pow2_at_least(2 * coors.shape[0])
        keys = torch.empty(hcap, dtype=torch.int64, device="cuda")
        vals = torch.empty(hcap, dtype=torch.int32, device="cuda")
        L.check(self.lib.b2s_hash_build(L.ptr(coors), L.ptr(n_dev), coors.shape[0], L.i3(shape), L.ptr(keys),
                                        L.ptr(vals), hcap, L.ptr(self.status), L.stream()), "b2s_hash_build")
        return keys, vals, hcap


def _check_level(oracle, coors_out, n_out, nbr, row_mask, in_idx, B, in_shape, k, s, p, subm=False):
    """a rulebook against oracle get_indice_pairs: output coordinates bit-exact and in order, the same neighbour
    table, row_mask = OR of (nbr >= 0) << k; entries past the live rows untouched."""
    out_idx, pairs, num = oracle.ops.get_indice_pairs(in_idx, B, in_shape, k, s, p, 1, subm=subm)
    n = int(n_out.item()) if n_out is not None else in_idx.shape[0]
    assert n == out_idx.shape[0]
    if coors_out is not None:
        assert torch.equal(coors_out[:n].cpu(), out_idx), "output coordinates differ from the oracle (value or order)"
        assert bool((coors_out[n:] == -7).all())
    ref = _nbr_from_pairs(pairs, num, n)
    got = nbr[:n].cpu()
    assert torch.equal(got, ref), "neighbour table differs in %d entries" % int((got != ref).sum())
    assert torch.equal(row_mask[:n].cpu().long() & 0x7FFFFFF, _row_mask(ref))
    return out_idx


CHAINS = {  # level-0 shape, first strided conv (k, s, p), second strided conv on the level in between
    "k3s2p1-then-k311": ((9, 40, 42), ([3, 3, 3], [2, 2, 2], [1, 1, 1]), ([3, 1, 1], [2, 1, 1], [0, 0, 0])),
    "k3s2p011-then-k3s2p1": ((11, 30, 45), ([3, 3, 3], [2, 2, 2], [0, 1, 1]), ([3, 3, 3], [2, 2, 2], [1, 1, 1])),
}


@pytest.mark.timeout(180)
@pytest.mark.parametrize("batch", [1, 3])
@pytest.mark.parametrize("chain", sorted(CHAINS))
def test_rulebook_chain_matches_oracle(product, oracle, chain, batch):
    """strided conv without an output hash -> SubM by rank on the same workspace -> strided conv on that level without
    an input hash, as the engine builds levels >= 1.  Output widths 21 / 23 are no multiple of 32: occupancy words
    straddle rows, and (B = 3, frame 1 empty) frames."""
    shape0, (k1, s1, p1), (k2, s2, p2) = CHAINS[chain]
    ops = oracle.ops
    shape1 = ops.get_conv_output_size(shape0, k1, s1, p1, [1, 1, 1])
    shape2 = ops.get_conv_output_size(shape1, k2, s2, p2, [1, 1, 1])
    rng = np.random.default_rng(batch * 10 + len(chain))
    idx0 = _chain_coords(rng, shape0, batch, 900, empty_frame=1 if batch == 3 else None)
    ch = _Chain(product, batch, [shape1, shape2])
    c0 = idx0.cuda()
    n0 = torch.tensor([idx0.shape[0]], dtype=torch.int32, device="cuda")
    cap1 = idx0.shape[0] * 8 + 11
    c1, n1, nbr1, rm1 = ch.conv(c0, n0, shape0, shape1, k1, s1, p1, cap1)
    nbr_s, rm_s = ch.subm_ranked(c1, n1, shape1)
    torch.cuda.synchronize()
    idx1 = _check_level(oracle, c1, n1, nbr1, rm1, idx0, batch, shape0, k1, s1, p1)
    if batch == 3:
        assert not bool((idx1[:, 0] == 1).any()) and bool((idx1[:, 0] == 2).any())
    _check_level(oracle, None, n1, nbr_s, rm_s, idx1, batch, shape1, [3, 3, 3], [1, 1, 1], [1, 1, 1], subm=True)
    c2, n2, nbr2, rm2 = ch.conv(c1, n1, shape1, shape2, k2, s2, p2, int(n1.item()) * 4 + 11)
    torch.cuda.synchronize()
    _check_level(oracle, c2, n2, nbr2, rm2, idx1, batch, shape1, k2, s2, p2)
    assert int(ch.status.item()) == 0


def probe_vs_scatter_main():
    """run with B2S_RB_SCATTER=0 (read once per process): the strided table by hash probes (k_conv_nbr) where an input
    hash is given, by the input-side scatter where it is not -- in either call order -- must agree with the oracle."""
    from b2second import loader
    assert os.environ.get("B2S_RB_SCATTER") == "0"
    product, oracle = loader.product_spconv(), loader.oracle_spconv()
    for chain in sorted(CHAINS):
        shape0, (k1, s1, p1), _ = CHAINS[chain]
        shape1 = oracle.ops.get_conv_output_size(shape0, k1, s1, p1, [1, 1, 1])
        for batch in (1, 3):
            rng = np.random.default_rng(batch + 5)
            idx0 = _chain_coords(rng, shape0, batch, 900, empty_frame=1 if batch == 3 else None)
            ch = _Chain(product, batch, [shape1])
            c0 = idx0.cuda()
            n0 = torch.tensor([idx0.shape[0]], dtype=torch.int32, device="cuda")
            cap1 = idx0.shape[0] * 8 + 11
            res = []
            for hashed in (False, True, False):
                h = ch.hash(c0, n0, shape0) if hashed else None
                res.append(ch.conv(c0, n0, shape0, shape1, k1, s1, p1, cap1, hash_in=h))
                torch.cuda.synchronize()
                _check_level(oracle, *res[-1], idx0, batch, shape0, k1, s1, p1)
            for r in res[1:]:
                assert all(torch.equal(a, b) for a, b in zip(res[0], r))
            assert int(ch.status.item()) == 0
    print("probe == scatter == oracle")


def _run_with_scatter_off(code, timeout=600):
    env = dict(os.environ, B2S_RB_SCATTER="0")
    boot = "import sys; sys.path[:0] = %r\n" % [HERE, REPO, os.path.join(REPO, "second.pytorch_b200")]
    r = subprocess.run([sys.executable, "-c", boot + code], capture_output=True, text=True, timeout=timeout, env=env,
                       cwd=REPO)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


@pytest.mark.timeout(600)
def test_rulebook_probe_path_matches_scatter_path():
    """B2S_RB_SCATTER=0 is cached per process: the comparison runs in a fresh interpreter."""
    out = _run_with_scatter_off("import test_gpu_tc_forms as t; t.probe_vs_scatter_main()")
    assert "probe == scatter == oracle" in out


_ENGINE_RUN = """
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
dets = eng.detections()
np.savez(OUT, **{"%s_%d" % (k, i): d[k].cpu().numpy() for i, d in enumerate(dets)
                 for k in ("box3d_lidar", "scores", "label_preds")}, status=eng.status.cpu().numpy())
"""


@pytest.mark.timeout(900)
def test_engine_probe_rulebooks_give_identical_detections(tmp_path):
    """the engine with B2S_RB_SCATTER=0 (hash probes wherever a level has a hash; levels whose hash the engine skips
    fall back to the scatter) against the default build of the tables: bit-identical detections, B = 3 with an empty
    frame in the middle."""
    outs = []
    for scatter_off in (True, False):
        path = str(tmp_path / ("off.npz" if scatter_off else "on.npz"))
        code = "OUT = %r\n" % path + _ENGINE_RUN
        if scatter_off:
            _run_with_scatter_off(code)
        else:
            r = subprocess.run([sys.executable, "-c", "import sys; sys.path[:0] = %r\n" % [
                HERE, REPO, os.path.join(REPO, "second.pytorch_b200")] + code], capture_output=True, text=True,
                timeout=600, env={k: v for k, v in os.environ.items() if k != "B2S_RB_SCATTER"}, cwd=REPO)
            assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        outs.append(np.load(path))
    a, b = outs
    assert int(a["status"][0]) == 0 and int(b["status"][0]) == 0
    assert sorted(a.files) == sorted(b.files)
    for k in a.files:
        assert np.array_equal(a[k], b[k]), k
    assert a["scores_0"].shape[0] > 0 and a["scores_1"].shape[0] == 0
