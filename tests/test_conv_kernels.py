"""Kernel-level tests of the tensor-core convolutions: the TMA dense conv (sassd_conv2d_f16x3[_occ]), the split-row
sparse conv (sassd_spconv_f16x3), the register-gather conv (sassd_gconv) and the conversions that feed them.

Every output element is held to an fp64 reference through a per-element bound derived from the kernels' arithmetic
(part A, CPU), every launch variant is driven through the C ABI with the test's own descriptor, and every output
buffer sits between guard regions filled with a sentinel, so that what a kernel must leave untouched or write as zero
is checked too.  Part A runs without a GPU; everything else is marked `gpu`.
"""
import ctypes
import os
import subprocess
import sys
from itertools import product

import numpy as np
import pytest
import torch

from tests.kernel_buffers import SENTINEL, Guarded, _p, _stream, pos_zero, untouched

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ------------------------------------------------------------------------------------------------------------------
# A. fp64 reference, per-element error bound, CPU emulation of the kernels' arithmetic
# ------------------------------------------------------------------------------------------------------------------
# Bound: |got - ref| <= TAU * S + TINY, S = |scale| * sum_k |x_k| |w_k| (fp64), TINY = 2^-21 |ref| + 1e-30.
#
# The FP16x3 kernels split each operand into hi = half(v) and lo = half((v - hi) * 2048) (22 significant bits), sum
# hi*hi in one fp32 accumulator and hi*lo + lo*hi in another, and return big + small / 2048.  Every product is exact
# in fp32; what is lost is the lo*lo term and the lo rounding (~2^-22 |x||w| per term, random sign) and the fp32
# rounding of the running sums, which grows with the partial sums, not with the result.  Relative to S these stay
# near 2^-24: emulate_f16x3 below reproduces the arithmetic (sequential fp32 accumulation in the kernels' K order)
# and its largest err / S over test_emulated_error_stays_within_tau's cases, K up to 2880, is 3.9e-7.  TAU = 2^-19
# (1.9e-6) keeps a 4x margin over that for the tensor core's own summation order inside a K = 16 step.  It cannot be
# loosened much: dropping the two cross products (the defect that turns FP16x3 into plain fp16) moves err / S by only
# ~2^-11 / sqrt(K), 29 TAU at the shape test_mutations_are_rejected uses, and it must stay >= 10 TAU.
# TINY absorbs the rounding of the result itself (fp32 store: 2^-24 |ref|; split output hi + lo / 2048: 2^-22 |ref|).
# The 3xTF32 split keeps one significand bit less per operand (hi 11, lo 10 after the sign-free residual), which
# doubles the representation part of the error; the FFMA path has only the fp32 accumulation part.
TAU = 2.0 ** -19
TAU_TF32 = 2 * TAU
TAU_FFMA = TAU

F16_LO_SCALE = 2048.0


def nhwc_taps(x, taps):
    """Yield the per-tap input rows [B*H*W, C] of a 3x3 (zero padding 1) or 1x1 NHWC convolution."""
    B, H, W, C = x.shape
    if taps == 1:
        yield x.reshape(-1, C)
        return
    xp = torch.nn.functional.pad(x, (0, 0, 1, 1, 1, 1))
    for t in range(9):
        dy, dx = t // 3 - 1, t % 3 - 1
        yield xp[:, 1 + dy:1 + dy + H, 1 + dx:1 + dx + W, :].reshape(-1, C)


def table_taps(x, nbr):
    """Yield the per-tap input rows of the neighbour-table conv: row(m, t) = nbr[m, t], -1 = no input (zero)."""
    rows, C = x.shape
    xz = torch.cat([x, torch.zeros((1, C), dtype=x.dtype, device=x.device)])
    idx = torch.where(nbr < 0, torch.full_like(nbr, rows), nbr).long()
    for t in range(nbr.shape[1]):
        yield xz[idx[:, t]]


def conv_ref(xt, w, scale, shift, relu):
    """fp64 out[m, :] = act((sum_t X_t[m] @ W[t]) * scale + shift) and S = |scale| * sum_t |X_t[m]| @ |W[t]|."""
    wd = w.double()
    acc = S = 0
    for t, X in enumerate(xt):
        X = X.double()
        acc = acc + X @ wd[t]
        S = S + X.abs() @ wd[t].abs()
    cout = w.shape[2]
    sc = scale.double() if scale is not None else torch.ones(cout, dtype=torch.float64, device=w.device)
    sh = shift.double() if shift is not None else torch.zeros(cout, dtype=torch.float64, device=w.device)
    ref = acc * sc + sh
    if relu:
        ref = ref.clamp_min(0)
    return ref, S * sc.abs()


def _tiny(ref):
    return 2.0 ** -21 * ref.abs() + 1e-30


def err_ratio(got, ref, S):
    """Largest |got - ref| / S (elements with S > 0) - the number reported next to TAU."""
    err = (got.double() - ref).abs()
    m = S > 0
    return float((err[m] / S[m]).max()) if bool(m.any()) else 0.0


def excess(got, ref, S, tau):
    """max (|got - ref| - TINY) / (tau * S): <= 1 inside the bound, the factor by which a corrupted result misses it."""
    err = (got.double() - ref).abs() - _tiny(ref)
    return float((err.clamp_min(0) / (tau * S + 1e-300)).max())


MAX_RATIO = {}       # kernel family -> (largest err / S seen, tau), printed at the end of the module


def check_bound(got, ref, S, tau, family, what=""):
    ok = (got.double() - ref).abs() <= tau * S + _tiny(ref)
    r = err_ratio(got, ref, S)
    prev = MAX_RATIO.get(family, (0.0, tau))[0]
    MAX_RATIO[family] = (max(prev, r), tau)
    if not bool(ok.all()):
        bad = torch.nonzero(~ok)
        raise AssertionError("%s %s: %d elements outside the bound (tau %.2e), max err/S %.3e, first %s" % (
            family, what, bad.shape[0], tau, r, bad[:4].tolist()))


def f16_split(v):
    """hi / lo planes of fp32 values exactly as tc::split_f16x2 computes them."""
    hi = v.half()
    lo = ((v - hi.float()) * F16_LO_SCALE).half()
    return hi, lo


def emulate_f16x3(xt, w, scale, shift, relu, corrupt=None, accumulators=2):
    """CPU emulation of the FP16x3 kernels on fp32 inputs (xt: per-tap rows, w [taps, cin, cout]): operands split by
    f16_split, hi*hi summed in one fp32 accumulator and the cross products in another (accumulators = 3: one per
    cross product, as the sparse kernel keeps them), K in tap-major order, then big + small / 2048, fp32 scale /
    shift, ReLU.  `corrupt` injects one defect (test_mutations_are_rejected):
      "cross"  the two cross products dropped         "tap"   tap 0 missing at the last pixel
      "chunk"  input channels 64..127 of tap 4 missing "swap"  scale / shift of channels 0 and 1 swapped
      "relu"   ReLU not applied."""
    taps, cin, cout = w.shape
    X = torch.stack([t.float() for t in xt], 1).clone()          # [M, taps, cin]
    if corrupt == "tap":
        X[-1, 0, :] = 0
    if corrupt == "chunk":
        X[:, 4, 64:128] = 0
    X = X.reshape(X.shape[0], -1).numpy()
    Wk = w.float().reshape(-1, cout).numpy()
    xh, xl = (a.numpy().astype(np.float32) for a in f16_split(torch.from_numpy(X)))
    wh, wl = (a.numpy().astype(np.float32) for a in f16_split(torch.from_numpy(Wk)))
    M = X.shape[0]
    big = np.zeros((M, cout), np.float32)
    s1 = np.zeros((M, cout), np.float32)
    s2 = np.zeros((M, cout), np.float32) if accumulators == 3 else s1
    for k in range(X.shape[1]):
        big = big + xh[:, k, None] * wh[None, k, :]
        if corrupt != "cross":
            s1 = s1 + xl[:, k, None] * wh[None, k, :]
            if accumulators == 3:
                s2 = s2 + xh[:, k, None] * wl[None, k, :]
            else:
                s1 = s1 + xh[:, k, None] * wl[None, k, :]
    small = s1 + s2 if accumulators == 3 else s1
    a = (big + small * np.float32(1.0 / F16_LO_SCALE)).astype(np.float64)
    sc = scale.double().numpy().copy() if scale is not None else np.ones(cout)
    sh = shift.double().numpy().copy() if shift is not None else np.zeros(cout)
    if corrupt == "swap":
        sc[[0, 1]] = sc[[1, 0]]
        sh[[0, 1]] = sh[[1, 0]]
    out = (a * sc + sh).astype(np.float32)            # fmaf: exact product in fp64, one rounding to fp32
    if relu and corrupt != "relu":
        out = np.maximum(out, 0)
    return torch.from_numpy(out)


def _emu_case(seed, B, H, W, cin, cout, taps, table_rows=0):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(taps, cin, cout, generator=g) * 0.05
    scale = torch.rand(cout, generator=g) + 0.5
    shift = torch.randn(cout, generator=g) * 0.3
    if table_rows:
        x = torch.randn(table_rows, cin, generator=g)
        nbr = torch.where(torch.rand(table_rows, taps, generator=g) < 0.4,
                          torch.randint(0, table_rows, (table_rows, taps), generator=g), torch.full((table_rows, taps), -1))
        xt = list(table_taps(x.double(), nbr))
    else:
        x = torch.randn(B, H, W, cin, generator=g)
        xt = list(nhwc_taps(x.double(), taps))
    return xt, w, scale, shift


@pytest.mark.parametrize("case", [(1, 9, 17, 128, 32, 9, 0), (1, 5, 7, 320, 64, 9, 0), (1, 8, 16, 256, 256, 1, 0),
                                  (1, 3, 21, 28, 20, 9, 0), (0, 0, 0, 64, 64, 27, 200)],
                         ids=["3x3-128-32", "3x3-320-64", "1x1-256-256", "3x3-28-20", "table-64-64"])
def test_emulated_error_stays_within_tau(case):
    """The emulated FP16x3 arithmetic stays 4x inside TAU (the margin TAU keeps for the hardware's summation order)."""
    B, H, W, cin, cout, taps, rows = case
    xt, w, scale, shift = _emu_case(cin * 7 + cout, B, H, W, cin, cout, taps, rows)
    for relu in (False, True):
        ref, S = conv_ref(xt, w, scale, shift, relu)
        emu = emulate_f16x3([t.float() for t in xt], w, scale, shift, relu, accumulators=3 if rows else 2)
        assert excess(emu, ref, S, TAU / 4) <= 1.0, err_ratio(emu, ref, S)
        # the split output as the next layer reads it (hi + lo / 2048) obeys the same bound
        hi, lo = f16_split(emu)
        assert excess(hi.float() + lo.float() / F16_LO_SCALE, ref, S, TAU / 4) <= 1.0


@pytest.mark.parametrize("corrupt", ["cross", "tap", "chunk", "swap", "relu"])
def test_mutations_are_rejected(corrupt):
    """The bound can fail: each single defect of the emulated kernel misses it by at least 10x.  The map has
    partial tiles in H and W (H % 8 = 1, W % 16 = 1); the missing tap is at the pixel alone in its corner tile."""
    xt, w, scale, shift = _emu_case(3, 1, 9, 17, 128, 32, 9)
    ref, S = conv_ref(xt, w, scale, shift, True)
    x32 = [t.float() for t in xt]
    good = emulate_f16x3(x32, w, scale, shift, True)
    assert excess(good, ref, S, TAU) <= 1.0
    bad = emulate_f16x3(x32, w, scale, shift, True, corrupt=corrupt)
    assert excess(bad, ref, S, TAU) >= 10.0, (corrupt, excess(bad, ref, S, TAU))


def tile_dist_model(coors, n_rows, batch, H, W, fill):
    """numpy model of sassd_mark_conv2d_tiles: per 8x16 tile, the smallest Chebyshev distance from an active cell
    (b, y, x) of rows [0, n_rows) to the tile's rectangle, recorded when it is at most SASSD_TILE_DIST_MAX."""
    th, tw, R = 8, 16, 9
    ty_n, tx_n = (H + th - 1) // th, (W + tw - 1) // tw
    dist = np.full((batch, ty_n, tx_n), fill, np.int64)
    y0 = np.arange(ty_n)[:, None] * th
    x0 = np.arange(tx_n)[None, :] * tw
    for b, _, y, x in coors[:n_rows]:
        dy = np.maximum(np.maximum(y0 - y, y - (y0 + th - 1)), 0)
        dx = np.maximum(np.maximum(x0 - x, x - (x0 + tw - 1)), 0)
        d = np.maximum(dy, dx)
        dist[b] = np.where(d <= R, np.minimum(dist[b], d), dist[b])
    return dist.reshape(-1)


def test_tile_dist_model_matches_definition():
    """The numpy model of the tile distances equals a brute-force pixel-level Chebyshev distance (CPU)."""
    H, W = 19, 37
    coors = np.array([[0, 0, 0, 0], [0, 0, 18, 36], [1, 0, 9, 20], [1, 0, 3, 33]])
    got = tile_dist_model(coors, 4, 2, H, W, 1 << 20).reshape(2, 3, 3)
    for b, ty, tx in product(range(2), range(3), range(3)):
        d = [max(max(ty * 8 - y, y - (ty * 8 + 7), 0), max(tx * 16 - x, x - (tx * 16 + 15), 0))
             for bb, _, y, x in coors if bb == b]
        exp = min(d)
        assert got[b, ty, tx] == (exp if exp <= 9 else 1 << 20)


# ------------------------------------------------------------------------------------------------------------------
# GPU helpers: direct C-ABI launches into guarded buffers (tests/kernel_buffers.py)
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    from sassd_b200 import ops
    ops.require_cuda()
    return torch.device("cuda:0")


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if MAX_RATIO:
        print("\nlargest |err|/S per kernel family:")
        for k, (r, tau) in sorted(MAX_RATIO.items()):
            print("  %-28s %.3e   tau %.3e   (%.2f tau)" % (k, r, tau, r / tau))


def dense_width(cout):
    """Output channels the dense kernel computes and stores: cout rounded up to 32, 64, 128 or 256."""
    return 32 if cout <= 32 else 64 if cout <= 64 else 128 if cout <= 128 else 256


def launch_dense(planes, cin, wpack, scale, shift, cout, taps, relu, mode, dev, n_split=0, tile_order=0,
                 tile_dist=None, reach=0, cvec=None, f32_stride=None, split_ch=None):
    """One sassd_conv2d_f16x3_occ launch with guarded outputs.  mode: "split", "f32" or "both"."""
    from sassd_b200 import lib
    _, B, H, W, cs = planes.shape
    d = lib.Conv2dDesc()
    d.batch, d.H, d.W, d.cin, d.cin_stored = B, H, W, cin, cs
    d.cout, d.taps, d.relu = cout, taps, int(relu)
    d.tile_order, d.n_split = tile_order, n_split
    of = osp = None
    if mode in ("f32", "both"):
        d.out_f32_stride = f32_stride or (cout + 3) // 4 * 4
        of = Guarded((B, H, W, d.out_f32_stride), torch.float32, dev)
    if mode in ("split", "both"):
        d.out_split_ch = split_ch or (cout + 63) // 64 * 64
        osp = Guarded((2, B, H, W, d.out_split_ch), torch.float16, dev)
    rc = lib.load().sassd_conv2d_f16x3_occ(ctypes.byref(d), _p(planes), _p(wpack), _p(scale), _p(shift),
                                           _p(of.t if of else None), _p(osp.t if osp else None), _p(tile_dist), reach,
                                           _p(cvec), None, _stream())
    lib.check(rc, "sassd_conv2d_f16x3_occ")
    torch.cuda.synchronize()
    return of, osp


def split_float(planes):
    return planes[0].float() + planes[1].float() / F16_LO_SCALE


def check_dense_outputs(of, osp, ref, S, cout, family, tau=TAU):
    """Values within the bound, [cout, width) exactly +0, channels beyond the width and the guards untouched, and the
    split output equal to the split of the fp32 output when both exist."""
    n = dense_width(cout)
    if of is not None:
        v = of.t
        st = v.shape[-1]
        check_bound(v[..., :cout].reshape(-1, cout), ref, S, tau, family, "fp32 out")
        assert pos_zero(v[..., cout:min(st, n)]), "fp32 channels [cout, width) not exactly 0"
        assert untouched(v[..., n:]), "fp32 channels beyond the computed width written"
        assert of.guards_intact(), "write outside the fp32 output"
    if osp is not None:
        p = osp.t
        ch = p.shape[-1]
        check_bound(split_float(p)[..., :cout].reshape(-1, cout), ref, S, tau, family, "split out")
        assert pos_zero(p[..., cout:min(ch, n)]), "split channels [cout, width) not exactly 0"
        assert untouched(p[..., n:]), "split channels beyond the computed width written"
        assert osp.guards_intact(), "write outside the split output"
    if of is not None and osp is not None:
        hi, lo = f16_split(of.t[..., :cout])
        assert torch.equal(osp.t[0, ..., :cout].view(torch.int16), hi.view(torch.int16))
        assert torch.equal(osp.t[1, ..., :cout].view(torch.int16), lo.view(torch.int16))


def _dense_inputs(dev, B, H, W, cin, cout, taps, ss, seed):
    from sassd_b200 import ops
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(B, H, W, cin, device=dev, generator=g)
    w = torch.randn(taps, cin, cout, device=dev, generator=g) * (1.0 / (taps * cin) ** 0.5)
    scale = (torch.rand(cout, device=dev, generator=g) + 0.5) if ss in ("both", "scale") else None
    shift = (torch.randn(cout, device=dev, generator=g) * 0.5) if ss in ("both", "shift") else None
    xs = ops.SplitMap.from_float(x)
    # the reference sees exactly the value the split planes carry (hi + lo / 2048), as the kernel does
    xr = split_float(xs.planes)[..., :cin].double()
    return xs, w, scale, shift, xr


# ------------------------------------------------------------------------------------------------------------------
# B. dense TMA conv: variant matrix against fp64, with guarded outputs (D)
# ------------------------------------------------------------------------------------------------------------------
MAPS = {"h1w15": (1, 17, 31), "h7w1": (1, 15, 17), "tile1": (1, 8, 16), "b3": (3, 23, 33), "many": (2, 96, 144)}
OUT_MODES = ("split", "f32", "both")
SS_MODES = ("both", "none", "scale", "shift")


def _dense_cases():
    cases = []
    for i, (cout, taps, cin) in enumerate(product((20, 28, 33, 64, 72, 128, 129, 256), (1, 9), (28, 64, 256, 320))):
        m = list(MAPS)[i % len(MAPS)]
        out, relu, ss = OUT_MODES[i % 3], (i // 3) % 2, SS_MODES[(i // 2) % 4]
        for ns in ((0, 2) if taps == 9 and cout > 128 else (0,)):
            cases.append(pytest.param(m, cin, cout, taps, ns, out, relu, ss,
                                      id="%s-%d-%d-t%d-ns%d-%s-%s-ss_%s" % (m, cin, cout, taps, ns, out,
                                                                           "relu" if relu else "lin", ss)))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("m,cin,cout,taps,n_split,out,relu,ss", _dense_cases())
def test_dense_conv_matrix(dev, m, cin, cout, taps, n_split, out, relu, ss):
    """Every N width (cout 20 .. 256 -> BN 32, 64, 128, 256), 1x1 and 3x3, K-chunk tail / one / many chunks, partial
    tiles in H and W, a single tile, B = 3, more tiles than SMs, whole and half-width units, each output mode: every
    element within the fp64 bound, padding channels exactly 0, nothing written outside.  A launch in another output
    mode gives the same bits."""
    from sassd_b200 import ops
    B, H, W = MAPS[m]
    xs, w, scale, shift, xr = _dense_inputs(dev, B, H, W, cin, cout, taps, ss, hash((m, cin, cout, taps)) % 1000)
    wp = ops.pack_tc(w, ops.PREC_F16X3)
    ref, S = conv_ref(nhwc_taps(xr, taps), w, scale, shift, relu)
    of, osp = launch_dense(xs.planes, cin, wp, scale, shift, cout, taps, relu, out, dev, n_split=n_split)
    check_dense_outputs(of, osp, ref, S, cout, "dense conv2d_tma")
    if out != "both":           # the output mode does not change a bit of what is computed
        of2, osp2 = launch_dense(xs.planes, cin, wp, scale, shift, cout, taps, relu, "both", dev, n_split=n_split)
        if of is not None:
            assert torch.equal(of.t.view(torch.int32), of2.t.view(torch.int32))
        if osp is not None:
            assert torch.equal(osp.t[..., :cout].view(torch.int16), osp2.t[..., :cout].view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize("cout,split_ch,f32_stride", [(20, 40, 24), (20, 64, 40), (72, 80, 76), (129, 136, 132),
                                                      (33, 32 * 3, 64 + 8)])
def test_dense_conv_output_widths(dev, cout, split_ch, f32_stride):
    """Output buffers narrower or wider than the computed width (cout rounded up to 32 / 64 / 128 / 256): channels
    [cout, width) are 0, channels beyond the width are left untouched, nothing beyond the buffer is written."""
    from sassd_b200 import ops
    B, H, W, cin, taps = 1, 17, 31, 64, 9
    xs, w, scale, shift, xr = _dense_inputs(dev, B, H, W, cin, cout, taps, "both", cout)
    wp = ops.pack_tc(w, ops.PREC_F16X3)
    ref, S = conv_ref(nhwc_taps(xr, taps), w, scale, shift, True)
    of, osp = launch_dense(xs.planes, cin, wp, scale, shift, cout, taps, True, "both", dev, split_ch=split_ch,
                           f32_stride=f32_stride)
    check_dense_outputs(of, osp, ref, S, cout, "dense conv2d_tma")


# ------------------------------------------------------------------------------------------------------------------
# C. exact relations between launch variants
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cout", [129, 256])
@pytest.mark.parametrize("m", ["b3", "many"])
def test_dense_nsplit_1_vs_2_bit_identical(dev, m, cout):
    """Half-width units (n_split = 2) run the N = 128 kernel over the same K order as whole tiles: same bits."""
    from sassd_b200 import ops
    B, H, W = MAPS[m]
    xs, w, scale, shift, _ = _dense_inputs(dev, B, H, W, 256, cout, 9, "both", 11)
    wp = ops.pack_tc(w, ops.PREC_F16X3)
    a = launch_dense(xs.planes, 256, wp, scale, shift, cout, 9, True, "both", dev, n_split=1)
    b = launch_dense(xs.planes, 256, wp, scale, shift, cout, 9, True, "both", dev, n_split=2)
    assert torch.equal(a[0].t.view(torch.int32), b[0].t.view(torch.int32))
    assert torch.equal(a[1].t.view(torch.int16), b[1].t.view(torch.int16))


def _scattered(dev, B, H, W, cin, seed, n=40):
    """A split map that is zero except near scattered active cells (clustered in a corner, one in the far corner, the
    last frame empty), with the tile distances sassd_sparse_to_bev_split records."""
    from sassd_b200 import ops
    g = torch.Generator(device=dev).manual_seed(seed)
    coors = torch.zeros((n, 4), dtype=torch.int32, device=dev)
    coors[:, 0] = torch.randint(0, max(B - 1, 1), (n,), device=dev, generator=g)
    coors[:, 2] = torch.randint(0, 12, (n,), device=dev, generator=g)
    coors[:, 3] = torch.randint(0, 20, (n,), device=dev, generator=g)
    coors[n - 1, 2], coors[n - 1, 3] = H - 1, W - 1
    key = (coors[:, 0].long() * H + coors[:, 2].long()) * W + coors[:, 3].long()
    keep = torch.from_numpy(np.unique(key.cpu().numpy(), return_index=True)[1]).to(dev)
    rows = coors[keep].contiguous()
    feat = torch.randn(rows.shape[0], cin, device=dev, generator=g)
    d_rows = torch.tensor([rows.shape[0]], dtype=torch.int32, device=dev)
    planes = torch.zeros((2, B, H, W, cin), dtype=torch.float16, device=dev)
    dist = torch.full((B * ((H + 7) // 8) * ((W + 15) // 16),), 1 << 20, dtype=torch.int32, device=dev)
    from sassd_b200 import lib
    lib.check(lib.load().sassd_sparse_to_bev_split(_p(feat), _p(rows), _p(d_rows), rows.shape[0], cin, 1, H, W, B,
                                                   _p(planes), _p(dist), _stream()), "sassd_sparse_to_bev_split")
    return ops.SplitMap(planes, cin, dist)


@pytest.mark.gpu
@pytest.mark.parametrize("out", OUT_MODES)
@pytest.mark.parametrize("B,H,W", [(3, 40, 52), (4, 200, 176)], ids=["60tiles", "1100tiles"])
def test_dense_tile_order_0_vs_1_bit_identical(dev, B, H, W, out):
    """With tile distances present, tile_order = 1 (computed tiles first, the latency graph's order) stores the same
    bits as round-robin, in every output mode, for maps below and above the 832-tile verdict table."""
    from sassd_b200 import ops
    cin, cout = 64, 256
    x = _scattered(dev, B, H, W, cin, 3)
    g = torch.Generator(device=dev).manual_seed(4)
    w = torch.randn(9, cin, cout, device=dev, generator=g) * 0.1
    scale = torch.rand(cout, device=dev, generator=g) + 0.5
    shift = torch.randn(cout, device=dev, generator=g) * 0.3
    wp = ops.pack_tc(w, ops.PREC_F16X3)
    cvec = ops.conv_constant(None, cin, w, scale, shift, True, cout)
    r = [launch_dense(x.planes, cin, wp, scale, shift, cout, 9, True, out, dev, tile_order=o, tile_dist=x.tile_dist,
                      reach=1, cvec=cvec) for o in (0, 1)]
    for a, b in zip(r[0], r[1]):
        if a is not None:
            assert torch.equal(a.raw, b.raw)


_PAIR_SCRIPT = r"""
import ctypes, sys
sys.path.insert(0, sys.argv[1])
import torch
from sassd_b200 import lib, ops
from tests.test_conv_kernels import MAPS, _dense_inputs, launch_dense
dev = torch.device("cuda:0")
res = {}
for m, cout in [("b3", 129), ("b3", 256), ("many", 256)]:
    B, H, W = MAPS[m]
    xs, w, scale, shift, _ = _dense_inputs(dev, B, H, W, 320, cout, 9, "both", 21)
    of, osp = launch_dense(xs.planes, 320, ops.pack_tc(w, ops.PREC_F16X3), scale, shift, cout, 9, True, "both", dev)
    res["%s-%d" % (m, cout)] = (of.raw.cpu(), osp.raw.cpu(), of.lo, osp.lo)
torch.save(res, sys.argv[2])
"""


@pytest.mark.gpu
def test_dense_cta_pair_vs_single_cta(dev, tmp_path):
    """The opt-in CTA-pair kernel (SASSD_TMA_PAIR=1, read once per process: a fresh one) stores the same bits as the
    single-CTA kernel, and both satisfy the fp64 bound and the output contract."""
    from sassd_b200 import ops
    out = tmp_path / "pair.pt"
    env = dict(os.environ, SASSD_TMA_PAIR="1")
    r = subprocess.run([sys.executable, "-c", _PAIR_SCRIPT, ROOT, str(out)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    pair = torch.load(str(out))
    for m, cout in [("b3", 129), ("b3", 256), ("many", 256)]:
        B, H, W = MAPS[m]
        xs, w, scale, shift, xr = _dense_inputs(dev, B, H, W, 320, cout, 9, "both", 21)
        ref, S = conv_ref(nhwc_taps(xr, 9), w, scale, shift, True)
        of, osp = launch_dense(xs.planes, 320, ops.pack_tc(w, ops.PREC_F16X3), scale, shift, cout, 9, True, "both", dev)
        p_of, p_osp, lo_f, lo_s = pair["%s-%d" % (m, cout)]
        # same layout in both processes: compare the buffers, then check the pair's output like any other
        nf, ns = of.hi - of.lo, osp.hi - osp.lo
        assert torch.equal(p_of[lo_f:lo_f + nf], of.raw[of.lo:of.hi].cpu()), "fp32 output differs (%s %d)" % (m, cout)
        assert torch.equal(p_osp[lo_s:lo_s + ns], osp.raw[osp.lo:osp.hi].cpu()), "split output differs (%s %d)" % (m, cout)
        assert bool((p_of[:lo_f] == SENTINEL).all()) and bool((p_of[lo_f + nf:] == SENTINEL).all())
        assert bool((p_osp[:lo_s] == SENTINEL).all()) and bool((p_osp[lo_s + ns:] == SENTINEL).all())
        check_dense_outputs(of, osp, ref, S, cout, "dense conv2d_tma")


# ------------------------------------------------------------------------------------------------------------------
# E. split-row sparse conv: variant matrix against fp64, guarded outputs (D)
# ------------------------------------------------------------------------------------------------------------------
def sparse_width(cout):
    return 16 if cout <= 16 else 32 if cout <= 32 else 64


def tile_masks(nb, n_rows):
    """What the rulebook kernels record: per 128-row tile, the taps present among rows [0, n_rows)."""
    M, taps = nb.shape
    nt = (M + 127) // 128
    pad = np.full((nt * 128, taps), -1, np.int64)
    pad[:n_rows] = nb[:n_rows]
    present = (pad.reshape(nt, 128, taps) >= 0).any(1)
    return (present * (1 << np.arange(taps))[None, :]).sum(1).astype(np.int32)


def run_sparse(dev, cin_valid, cin_s, cout, taps, rows_cap, in_rows, n_rows, out, ws, masks, seed, relu=True,
               ss="both"):
    """One sassd_spconv_f16x3 launch on random split rows with a random neighbour table (hot rows gathered by many
    outputs, one 128-row tile without any pair); returns (guarded outputs, fp64 ref, S)."""
    from sassd_b200 import lib, ops
    rs = np.random.RandomState(seed)
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(in_rows, cin_valid, device=dev, generator=g)
    w = torch.randn(taps, cin_valid, cout, device=dev, generator=g) * (1.0 / (taps * cin_valid * 0.3) ** 0.5)
    scale = (torch.rand(cout, device=dev, generator=g) + 0.5) if ss in ("both", "scale") else None
    shift = (torch.randn(cout, device=dev, generator=g) * 0.5) if ss in ("both", "shift") else None
    planes = torch.zeros((2, in_rows, cin_s), dtype=torch.float16, device=dev)
    hi, lo = f16_split(x)
    planes[0, :, :cin_valid], planes[1, :, :cin_valid] = hi, lo
    xr = split_float(planes)[:, :cin_valid].double()
    nbr = tm = None
    if taps > 1:
        nb = np.where(rs.rand(rows_cap, taps) < 0.3, rs.randint(0, in_rows, (rows_cap, taps)), -1)
        hot = rs.randint(0, in_rows, 3)
        nb = np.where(rs.rand(rows_cap, taps) < 0.1, hot[rs.randint(0, 3, (rows_cap, taps))], nb)
        if rows_cap > 256:
            nb[128:256] = -1                                   # a tile with no pair at all: act(shift)
        nb = nb.astype(np.int32)
        nbr = torch.from_numpy(nb).to(dev)
        if masks:
            tm = torch.from_numpy(tile_masks(nb, n_rows)).to(dev)
        xt = table_taps(xr, nbr[:n_rows].long())
    else:
        xt = [xr[:n_rows]]
    ref, S = conv_ref(xt, w, scale, shift, relu)
    wp = ops.spconv_pack_cached(w, cin_s)
    d = lib.SpconvDesc()
    d.cin, d.cout, d.taps, d.rows_cap, d.in_rows_cap, d.relu = cin_s, cout, taps, rows_cap, in_rows, int(relu)
    d.out_ch = (cout + 7) // 8 * 8
    osp = Guarded((2, rows_cap, d.out_ch), torch.float16, dev)
    of = None
    if out == "both":
        d.out_f32_stride = (cout + 3) // 4 * 4
        of = Guarded((rows_cap, d.out_f32_stride), torch.float32, dev)
    wsb = torch.empty(lib.load().sassd_spconv_workspace_bytes(), dtype=torch.uint8, device=dev) if ws else None
    d_rows = torch.tensor([n_rows], dtype=torch.int32, device=dev)
    rc = lib.load().sassd_spconv_f16x3(ctypes.byref(d), _p(planes), _p(wp), _p(scale), _p(shift), _p(nbr), _p(tm),
                                       _p(d_rows), _p(osp.t), _p(of.t if of else None), _p(wsb),
                                       0 if wsb is None else wsb.numel(), None, _stream())
    lib.check(rc, "sassd_spconv_f16x3")
    torch.cuda.synchronize()
    return of, osp, ref, S


def check_sparse_outputs(of, osp, ref, S, cout, n_rows):
    n = sparse_width(cout)
    p = osp.t
    check_bound(split_float(p[:, :n_rows])[:, :cout], ref, S, TAU, "sparse spconv_split", "split out")
    assert pos_zero(p[:, :n_rows, cout:n]), "split channels [cout, out_ch) not exactly 0"
    assert untouched(p[:, n_rows:]), "split rows at or beyond d_rows written"
    assert osp.guards_intact(), "write outside the split output"
    if of is not None:
        v = of.t
        check_bound(v[:n_rows, :cout], ref, S, TAU, "sparse spconv_split", "fp32 out")
        assert pos_zero(v[:n_rows, cout:]), "fp32 stride padding not exactly 0"
        assert untouched(v[n_rows:]), "fp32 rows at or beyond d_rows written"
        assert of.guards_intact(), "write outside the fp32 output"
        hi, lo = f16_split(v[:n_rows, :cout])
        assert torch.equal(p[0, :n_rows, :cout].view(torch.int16), hi.view(torch.int16))
        assert torch.equal(p[1, :n_rows, :cout].view(torch.int16), lo.view(torch.int16))


CIN_S = [(4, 8), (16, 16), (32, 32), (64, 64)]


def _sparse_cases():
    cases = []
    drows = ("0", "1", "127", "129", "cap-5")
    for i, ((cv, cs), cout, taps) in enumerate(product(CIN_S, (16, 20, 32, 64), (27, 1))):
        dr = drows[i % 5]
        out = ("split", "both")[i % 2]
        ws, masks = (i // 2) % 2 == 0, (i // 4) % 2 == 0
        if taps == 1:
            ws = masks = False
        mode = "table" if taps > 1 else "rows"
        cases.append(pytest.param(cv, cs, cout, taps, 1000, dr, out, ws, masks,
                                  id="%s-%d_%d-%d-rows1000-d%s-%s-%s-%s" % (mode, cv, cs, cout, dr, out,
                                                                           "ws" if ws else "nows", "mask" if masks else "nomask")))
    return cases


def _n_rows(dr, cap):
    return cap - 5 if dr == "cap-5" else int(dr)


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cin_s,cout,taps,rows_cap,dr,out,ws,masks", _sparse_cases())
def test_sparse_conv_matrix(dev, cin, cin_s, cout, taps, rows_cap, dr, out, ws, masks):
    """Stored cin 8 (4 valid) / 16 / 32 / 64, cout 16 / 20 / 32 / 64 (N width 16, 32, 64; out_ch with padding), table
    (27 taps) and rows (1 tap) mode, d_rows 0 / 1 / 127 / 129 / rows_cap - 5 with in_rows_cap != rows_cap, with and
    without the tap-split workspace and tile masks, split-only and split + fp32 output."""
    n_rows = _n_rows(dr, rows_cap)
    in_rows = rows_cap + 40 if taps == 1 else rows_cap // 2 + 77
    of, osp, ref, S = run_sparse(dev, cin, cin_s, cout, taps, rows_cap, in_rows, n_rows, out, ws, masks, seed=cin * cout + taps)
    check_sparse_outputs(of, osp, ref, S, cout, n_rows)


@pytest.mark.gpu
@pytest.mark.parametrize("ws", [True, False], ids=["ws", "nows"])
@pytest.mark.parametrize("tiles", [1, 73, 74, 75, 160], ids=lambda t: "tiles%d" % t)
def test_sparse_conv_tap_split_boundary(dev, tiles, ws):
    """Layers of up to SPLIT_TILES_MAX = 74 tiles run as a tap split (two CTAs share each tile's chunks, partial sums
    through the workspace), larger ones do not; without the workspace no layer splits.  160 tiles makes CTAs walk
    two tiles.  Same bound and output contract on both sides of the rule."""
    rows_cap = tiles * 128
    of, osp, ref, S = run_sparse(dev, 64, 64, 64, 27, rows_cap, rows_cap + 300, rows_cap - 5, "both", ws, True,
                                 seed=tiles)
    check_sparse_outputs(of, osp, ref, S, 64, rows_cap - 5)


# ------------------------------------------------------------------------------------------------------------------
# F. conversion kernels and the register-gather conv
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cin,cs,d_rows", [(4, 8, 300), (16, 16, 0), (20, 24, 511), (64, 64, None), (3, 16, 1)])
def test_features_to_split_exact(dev, cin, cs, d_rows):
    """fp32 rows -> split rows: bit-exact hi / lo of every value of rows [0, d_rows), padding channels +0, rows at
    or beyond d_rows untouched, nothing outside the planes written."""
    from sassd_b200 import lib
    cap = 512
    g = torch.Generator(device=dev).manual_seed(cin)
    x = torch.randn(cap, cin, device=dev, generator=g) * torch.logspace(-6, 4, cap, device=dev)[:, None]
    out = Guarded((2, cap, cs), torch.float16, dev)
    dr = None if d_rows is None else torch.tensor([d_rows], dtype=torch.int32, device=dev)
    lib.check(lib.load().sassd_features_to_split(_p(x), _p(dr), cap, cin, cs, _p(out.t), _stream()),
              "sassd_features_to_split")
    torch.cuda.synchronize()
    n = cap if d_rows is None else d_rows
    hi, lo = f16_split(x[:n])
    assert torch.equal(out.t[0, :n, :cin].view(torch.int16), hi.view(torch.int16))
    assert torch.equal(out.t[1, :n, :cin].view(torch.int16), lo.view(torch.int16))
    assert pos_zero(out.t[:, :n, cin:])
    assert untouched(out.t[:, n:])
    assert out.guards_intact()


def _bev_rows(B, D, H, W, n, cap, seed):
    """Unique active cells (b, z, y, x) over B frames (the last one empty) including every map edge and corner;
    rows beyond n hold valid but different cells that a correct scatter never writes."""
    rs = np.random.RandomState(seed)
    edge = [(0, 0, 0, 0), (0, D - 1, H - 1, W - 1), (0, 0, 0, W - 1), (0, 0, H - 1, 0), (0, 0, H // 2, 0),
            (0, 0, 0, W // 2), (B - 2, D - 1, H - 1, W // 3), (B - 2, 0, H // 3, W - 1)]
    cells = set(edge)
    while len(cells) < cap:
        cells.add((rs.randint(0, B - 1), rs.randint(0, D), rs.randint(0, H), rs.randint(0, W)))
    allc = np.array(edge + sorted(cells - set(edge)), np.int32)
    return np.concatenate([allc[:len(edge)], rs.permutation(allc[len(edge):])])[:cap]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["split_rows", "sparse_f32"])
def test_bev_scatter_and_tile_dist_exact(dev, kind):
    """dense() of sparse rows into the split BEV map: exactly the active cells of rows [0, d_rows) are written
    (bits of the split rows / of the fp32 split), everything else keeps its prior content; the tile distances equal the
    numpy model of sassd_mark_conv2d_tiles.  Three frames, the last one empty, active cells on every edge."""
    from sassd_b200 import lib
    B, D, H, W, C = 3, 2, 41, 70, 16
    cap, n = 300, 260
    coors = _bev_rows(B, D, H, W, n, cap, 5)
    g = torch.Generator(device=dev).manual_seed(6)
    feat = torch.randn(cap, C, device=dev, generator=g)
    hi, lo = f16_split(feat)
    rows_split = torch.stack([hi, lo]).contiguous()
    bev = Guarded((2, B, H, W, D * C), torch.float16, dev)
    nt = B * ((H + 7) // 8) * ((W + 15) // 16)
    fill = 1 << 20
    dist = torch.full((nt,), fill, dtype=torch.int32, device=dev)
    c_t = torch.from_numpy(coors).to(dev)
    d_rows = torch.tensor([n], dtype=torch.int32, device=dev)
    L = lib.load()
    if kind == "split_rows":
        rc = L.sassd_split_rows_to_bev(_p(rows_split), _p(c_t), _p(d_rows), cap, C, D, H, W, B, _p(bev.t), _p(dist),
                                       _stream())
    else:
        rc = L.sassd_sparse_to_bev_split(_p(feat), _p(c_t), _p(d_rows), cap, C, D, H, W, B, _p(bev.t), _p(dist),
                                         _stream())
    lib.check(rc, kind)
    torch.cuda.synchronize()
    exp = np.full((2, B, H, W, D * C), -1, np.int16)           # int16 -1 == 0xFFFF: the sentinel
    rsn = rows_split.cpu().view(torch.int16).numpy()
    for r in range(n):
        b, z, y, x = coors[r]
        exp[:, b, y, x, z * C:(z + 1) * C] = rsn[:, r]
    assert np.array_equal(bev.t.cpu().view(torch.int16).numpy(), exp)
    assert bev.guards_intact()
    assert np.array_equal(dist.cpu().numpy(), tile_dist_model(coors, n, B, H, W, fill))


_GCONV_CASES = [
    # (mode, B, H, W or rows, cin, cout, taps)
    ("rows", 0, 0, 128, 32, 16, 1), ("rows", 0, 0, 128, 32, 64, 1), ("rows", 0, 0, 128, 64, 256, 1),
    ("rows", 0, 0, 1000, 256, 256, 1), ("rows", 0, 0, 1000, 28, 28, 1), ("rows", 0, 0, 777, 256, 20, 1),
    ("conv2d", 2, 12, 10, 32, 16, 9), ("conv2d", 1, 40, 36, 256, 256, 9), ("conv2d", 1, 40, 36, 320, 256, 9),
    ("conv2d", 1, 40, 36, 256, 28, 9),
    # shapes of the former test_tensor_core_conv_matches_fp64 (B = 2, 24 x 20)
    ("conv2d", 2, 24, 20, 256, 256, 9), ("conv2d", 2, 24, 20, 320, 256, 9), ("conv2d", 2, 24, 20, 256, 28, 9),
    ("conv2d", 2, 24, 20, 28, 28, 1), ("conv2d", 2, 24, 20, 256, 20, 1),
    ("table", 0, 0, 3000, 4, 16, 27), ("table", 0, 0, 3000, 16, 16, 27), ("table", 0, 0, 3000, 16, 32, 27),
    ("table", 0, 0, 3000, 32, 64, 27), ("table", 0, 0, 3000, 64, 64, 27),
]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "f16x3"])
@pytest.mark.parametrize("case", _GCONV_CASES, ids=lambda c: "%s-%s-%d-%d" % (c[0], "x".join(map(str, c[1:4])), c[4], c[5]))
def test_gconv_vs_fp64(dev, case, prec):
    """sassd_gconv (FFMA, 3xTF32 and FP16x3 register-gather kernels) in rows, conv2d and table mode: every element
    within the fp64 bound of its precision; table mode with a real d_rows leaves the rows beyond it untouched."""
    from sassd_b200 import ops
    mode, B, H, Wr, cin, cout, taps = case
    p = {"fp32": ops.PREC_FP32, "tf32x3": ops.PREC_TF32X3, "f16x3": ops.PREC_F16X3}[prec]
    tau = {"fp32": TAU_FFMA, "tf32x3": TAU_TF32, "f16x3": TAU}[prec]
    M = B * H * Wr if mode == "conv2d" else Wr
    g = torch.Generator(device=dev).manual_seed(cin * 1000 + cout + taps)
    x = torch.randn(M, cin, device=dev, generator=g)
    w = torch.randn(taps, cin, cout, device=dev, generator=g) * 0.1
    scale = torch.rand(cout, device=dev, generator=g) + 0.5
    shift = torch.randn(cout, device=dev, generator=g) * 0.1
    relu = mode != "rows"
    nbr = d_rows = None
    n = M
    if mode == "table":
        rs = np.random.RandomState(cin + cout)
        nbr = torch.from_numpy(np.where(rs.rand(M, 27) < 0.3, rs.randint(0, M, (M, 27)), -1).astype(np.int32)).to(dev)
        n = M - 37
        d_rows = torch.tensor([n], dtype=torch.int32, device=dev)
        xt = table_taps(x.double(), nbr[:n].long())
    elif mode == "conv2d":
        xt = nhwc_taps(x.double().view(B, H, Wr, cin), taps)
    else:
        xt = [x.double()]
    ref, S = conv_ref(xt, w, scale, shift, relu)
    out = Guarded((M, (cout + 3) // 4 * 4), torch.float32, dev)
    m = {"rows": ops.GCONV_ROWS, "conv2d": ops.GCONV_CONV2D, "table": ops.GCONV_TABLE}[mode]
    ops.gconv(x, w, scale, shift, out.t, mode=m, taps=taps, cin=cin, cout=cout, relu=relu, nbr=nbr, d_rows=d_rows,
              rows_cap=M, batch=B, H=H, W=Wr, precision=p)
    torch.cuda.synchronize()
    check_bound(out.t[:n, :cout], ref, S, tau, "gconv " + prec)
    assert untouched(out.t[n:]), "rows at or beyond d_rows written"
    assert out.guards_intact()
