"""Kernel-level tests of the detection tail: decode + guided-anchor selection (sassd_decode_select), PSWarp sampling
(sassd_pswarp), rescoring + rotated NMS + gather (sassd_rescore_nms) and the rotated BEV IoU / NMS kernels
(sassd_nms_mask, sassd_nms_sorted, sassd_boxes_iou_bev).

Every kernel is driven through the C ABI with the test's own buffers, capacities, strides and workspaces.  Outputs sit
between sentinel-filled guards (tests/kernel_buffers.py); inputs sit in NaN-filled allocations whose padding channels,
unused columns and rows that must not be read are NaN too, so a read that should not happen turns into a NaN in the
output.  Where the arithmetic is exact the results are compared bit for bit with a numpy fp32 model; elsewhere they are
held to an fp64 reference through a per-element bound derived from the kernels' arithmetic (part B derives the PSWarp
bound and shows on the CPU that it rejects single defects).  The rotated IoU and the NMS mask are compared bit for bit
with the reference CUDA kernel's outputs stored in tests/golden/nms.npz.  Parts marked `gpu` need a CUDA device.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests.kernel_buffers import SENTINEL, Guarded, _p, _stream, untouched
from tests.nms_box_sets import MIX_SIZES, RANDOM_N, THRESHOLDS, GROUPS

FLAG_GUIDED_CAP, FLAG_NMS_CAP, FLAG_DET_CAP = 4, 8, 32
NMS_CAP = 4096
U = 2.0 ** -24                       # unit roundoff of fp32
F32 = np.float32

MAX_RATIO = {}                       # quantity -> largest |err| / bound seen, printed at the end of the module


def record(what, err, bound):
    r = float(np.max(err / bound)) if np.size(err) else 0.0
    MAX_RATIO[what] = max(MAX_RATIO.get(what, 0.0), r)
    return r


def ulp(v):
    return np.spacing(np.abs(np.asarray(v, F32))).astype(np.float64)


def sigmoid64(x):
    return 1.0 / (1.0 + np.exp(-np.asarray(x, np.float64)))


def sigmoid_bound(x):
    """|fp32 sigmoid - fp64 sigmoid| of the kernels' 1 / (1 + expf(-x)): expf within 2 ulp of e = exp(-x) moves the
    result by s (1 - s) * 2 ulp(e) / e, the add and the divide round once each (2^-24 relative); counted as 2^-23 s
    plus the expf term."""
    x = np.asarray(x, np.float64)
    e = np.exp(-x)
    s = 1.0 / (1.0 + e)
    return s * ((1.0 - s) * 2.0 * ulp(e) / e + 2.0 * U) + 1e-45


# ------------------------------------------------------------------------------------------------------------------
# A. sassd_decode_select: numpy fp32 model (exact where the kernel's arithmetic is), capacities, exact edges
# ------------------------------------------------------------------------------------------------------------------
DS_CHUNK = 1024
PI32 = F32(3.14159274101257324)


def head_layout(ncls):
    na = 2 * ncls
    return na * 7, na * 7 + na * ncls, na * 7 + na * ncls + na * 2      # cls_off, dir_off, minimal stride


def anchor_parts(a, H, W):
    rot = a & 1
    t = a >> 1
    return t // (H * W), t % (H * W), rot                             # class, pixel, rotation


def decode_model(head, ncls, anchors, mask, thr):
    """Per frame: the selected anchors in anchor order (mask && max_c sigmoid > thr), their labels, and the decoded
    boxes: x, y, r and the fp32 part of z exactly as the kernel rounds them (numpy fp32 ops are IEEE), w / l / h and
    z in fp64 with their bounds.  anchors [B, Na, 7] (a shared table repeated)."""
    B, H, W, stride = head.shape
    cls_off, dir_off, _ = head_layout(ncls)
    n = ncls * H * W * 2
    a = np.arange(n)
    cls_a, pix, rot = anchor_parts(a, H, W)
    out = []
    for b in range(B):
        hb = head[b].reshape(H * W, stride)
        lg = hb[pix[:, None], cls_off + cls_a[:, None] * 2 * ncls + rot[:, None] * ncls + np.arange(ncls)[None]]
        with np.errstate(invalid="ignore", over="ignore"):
            s = sigmoid64(lg)
            sel = mask[b].astype(bool) & (s.max(1) > float(F32(thr)))
        idx = np.nonzero(sel)[0]
        lab = np.argmax(s[idx], 1) if len(idx) else np.zeros(0, np.int64)   # first maximum on ties
        c, p, r = cls_a[idx], pix[idx], rot[idx]
        e = hb[p[:, None], c[:, None] * 14 + r[:, None] * 7 + np.arange(7)[None]].astype(F32)
        an = anchors[b][idx].astype(F32)
        xa, ya, za, wa, la, ha, ra = (an[:, i] for i in range(7))
        zac = za + ha / F32(2)
        diag = np.sqrt(la * la + wa * wa)
        xg = e[:, 0] * diag + xa
        yg = e[:, 1] * diag + ya
        z0 = e[:, 2] * ha + zac                                        # fp32, before "- hg / 2"
        ex = np.exp(e[:, 3:6].astype(np.float64))
        whl = ex * an[:, 3:6].astype(np.float64)                       # w, l, h in fp64
        # expf within 2 ulp of exp(e), times the anchor size, then one rounding of the product
        whl_bound = 2.0 * ulp(ex) * an[:, 3:6].astype(np.float64) + 0.5 * ulp(whl)
        z = z0.astype(np.float64) - whl[:, 2] / 2.0
        # z inherits hg's error (halved), and "z0 - hg / 2" rounds once more (a full ulp covers a binade edge)
        z_bound = 0.5 * whl_bound[:, 2] + ulp(z)
        rg = e[:, 6] + ra
        d = hb[p[:, None], dir_off + c[:, None] * 4 + r[:, None] * 2 + np.arange(2)[None]]
        dl = d[:, 1] > d[:, 0]                                         # tie -> direction label 0
        rg = np.where((rg > 0) != dl, rg + PI32, rg).astype(F32)
        out.append(dict(index=idx, labels=lab, x=xg.astype(F32), y=yg.astype(F32), r=rg, whl=whl, whl_bound=whl_bound,
                        z=z, z_bound=z_bound))
    return out


DECODE_CASES = {
    # name: (ncls, H, W, B, anchors per frame, extra head channels, thr, frame with every anchor masked out)
    "c1-b1-shared": (1, 13, 45, 1, False, 0, 0.3, None),            # 1170 anchors: 2 chunks, the last partial
    "c3-b3-perframe-pad": (3, 21, 37, 3, True, 5, 0.3, 2),          # 4662 anchors, frame 2 all masked out
    "c1-b3-shared-pad-thr05": (1, 17, 61, 3, False, 3, 0.5, None),  # 4148 anchors, exact 0 logits at thr 0.5
    "c3-b1-perframe-thr05": (3, 9, 40, 1, True, 0, 0.5, None),
}


def make_decode_inputs(case, seed):
    """Head map, anchors and mask of one case, built from per-anchor roles: masked out, below thr or selected (with
    margin in the logit, plus the exact edges), and the selected anchors per frame.  Channels nobody may read are
    NaN: padding channels, every channel of masked-out anchors, codes / direction logits / anchor rows of anchors
    that are not selected (fill_codes writes the codes and direction logits of the emitted ones).  Returns (head
    [B, H*W, stride], anchors [B or 1, Na, 7], mask [B, Na], selected [B, Na], (stride, cls_off, dir_off))."""
    ncls, H, W, B, per_frame, extra, thr, dead = DECODE_CASES[case]
    rs = np.random.RandomState(seed)
    cls_off, dir_off, need = head_layout(ncls)
    stride = need + extra
    n = ncls * H * W * 2
    cls_a, pix, rot = anchor_parts(np.arange(n), H, W)
    lthr = float(np.log(thr / (1 - thr)))
    head = np.full((B, H * W, stride), np.nan, F32)
    mask = (rs.rand(B, n) < 0.85).astype(np.uint8)
    if dead is not None:
        mask[dead] = 0
    psel = [0.08, 0.2, 0.12]
    sel = (rs.rand(B, n) < np.array(psel[:B])[:, None]) & mask.astype(bool)
    edges = [a for a in (0, 1, DS_CHUNK - 1, DS_CHUNK, 2 * DS_CHUNK - 1, 2 * DS_CHUNK, 3 * DS_CHUNK, n - 1) if a < n]
    for b in range(B):
        if b != dead:
            mask[b, edges] = 1
            sel[b, edges] = True
    for b in range(B):
        for a in np.nonzero(mask[b])[0]:
            c, p, r = cls_a[a], pix[a], rot[a]
            lo = cls_off + c * 2 * ncls + r * ncls
            if sel[b, a]:
                top = lthr + rs.uniform(0.3, 3.0)
                lg = top - rs.uniform(0.1, 2.0, ncls)
                lg[rs.randint(ncls)] = top
                kind = rs.rand()
                if kind < 0.05:
                    lg[:] = top                                  # identical class logits: label 0
                elif kind < 0.1 and ncls == 3:
                    lg[1] = lg[2] = top                          # tie between classes 1 and 2: label 1
                    lg[0] = top - 0.5
                elif kind < 0.15 and thr == 0.5 and ncls > 1:
                    lg[0], lg[1] = 0.0, top                      # exact sigmoid 0.5 on a class that loses
            else:
                lg = lthr - rs.uniform(0.3, 3.0, ncls)
                if thr == 0.5 and rs.rand() < 0.3:
                    lg[:rs.randint(1, ncls + 1)] = 0.0           # sigmoid(0) = 0.5 exactly: not > 0.5
            head[b, p, lo:lo + ncls] = lg
    anchors = np.full((B if per_frame else 1, n, 7), np.nan, F32)
    used = sel.any(0) if not per_frame else None
    for f in range(anchors.shape[0]):
        rows = sel[f] if per_frame else used
        idx = np.nonzero(rows)[0]
        k = len(idx)
        an = np.stack([rs.uniform(0, 70.4, k), rs.uniform(-40, 40, k), rs.normal(-1.78, 0.1, k), rs.normal(1.6, 0.1, k),
                       rs.normal(3.9, 0.2, k), rs.normal(1.56, 0.05, k), np.where(rot[idx] == 1, 1.57, 0.0)], 1)
        an[rs.rand(k) < 0.05, 6] = -0.0                              # r = -0.0 anchors
        anchors[f, idx] = an.astype(F32)
    return head, anchors, mask, sel, (stride, cls_off, dir_off)


def fill_codes(head, H, W, sel, k_cap, lay, rs, signed_zero_anchors):
    """Box codes and direction logits of the anchors the kernel emits (the first k_cap selected ones per frame)."""
    dir_off = lay[2]
    B = head.shape[0]
    for b in range(B):
        idx = np.nonzero(sel[b])[0][:k_cap]
        c, p, r = anchor_parts(idx, H, W)
        k = len(idx)
        codes = np.stack([rs.uniform(-1, 1, k), rs.uniform(-1, 1, k), rs.uniform(-1, 1, k), rs.uniform(-1.5, 1.5, k),
                          rs.uniform(-1.5, 1.5, k), rs.uniform(-1.5, 1.5, k), rs.uniform(-1.5, 1.5, k)], 1).astype(F32)
        d = rs.normal(0, 1, (k, 2)).astype(F32)
        tie = rs.rand(k) < 0.1
        d[tie, 1] = d[tie, 0]                                        # tied direction logits: label 0
        z = np.isin(idx, signed_zero_anchors)
        codes[z, 6] = np.where(rs.rand(int(z.sum())) < 0.5, F32(0.0), F32(-0.0))   # r = +0 / -0 with ra = +-0
        for j in range(k):
            head[b, p[j], c[j] * 14 + r[j] * 7:c[j] * 14 + r[j] * 7 + 7] = codes[j]
            head[b, p[j], dir_off + c[j] * 4 + r[j] * 2:dir_off + c[j] * 4 + r[j] * 2 + 2] = d[j]


def bits(a):
    return np.ascontiguousarray(a, F32).view(np.int32)


def check_decode(got, model, k_cap):
    boxes, labels, index = got["boxes"].t.cpu().numpy(), got["labels"].t.cpu().numpy(), got["index"].t.cpu().numpy()
    d_k = got["d_k"].t.cpu().numpy()
    for b, m in enumerate(model):
        k = min(len(m["index"]), k_cap)
        assert d_k[b] == k, "frame %d: d_k %d, expected %d" % (b, d_k[b], k)
        assert np.array_equal(index[b, :k], m["index"][:k]), "frame %d: selected anchors differ" % b
        assert np.array_equal(labels[b, :k], m["labels"][:k]), "frame %d: labels differ" % b
        bx = boxes[b, :k]
        assert np.isfinite(bx).all(), "frame %d: NaN in the boxes (a read that must not happen)" % b
        for col, key in ((0, "x"), (1, "y"), (6, "r")):
            assert np.array_equal(bits(bx[:, col]), bits(m[key][:k])), "frame %d: column %d not bit-exact" % (b, col)
        err = np.abs(bx[:, 3:6].astype(np.float64) - m["whl"][:k])
        for i, name in enumerate("wlh"):
            record("decode " + name, err[:, i], m["whl_bound"][:k, i])
        assert (err <= m["whl_bound"][:k]).all(), "frame %d: w / l / h outside the bound" % b
        ez = np.abs(bx[:, 2].astype(np.float64) - m["z"][:k])
        record("decode z", ez, m["z_bound"][:k])
        assert (ez <= m["z_bound"][:k]).all(), "frame %d: z outside the bound" % b
        for t in (got["boxes"].t, got["labels"].t, got["index"].t):
            assert untouched(t[b, k:]), "frame %d: rows at or beyond d_k written" % b
    for g in ("boxes", "labels", "index", "d_k"):
        assert got[g].guards_intact(), "write outside " + g


@pytest.mark.gpu
@pytest.mark.parametrize("cap", ["roomy", "full", "over"])
@pytest.mark.parametrize("case", list(DECODE_CASES))
def test_decode_select(dev, case, cap):
    """Selection, labels and x / y / r bit-exact with the numpy fp32 model, w / l / h / z within their bounds, d_k
    and the GUIDED_CAP flag: k_cap above the largest frame count, equal to it (no flag), or below it (flag 4, that
    frame keeps its first k_cap selections in anchor order, the others are unchanged).  Rows at or beyond d_k and the
    guards untouched; a second run on the now dirty workspace (the first one's starts as 0xFF) gives the same bytes."""
    ncls, H, W, B, per_frame, _, thr, _ = DECODE_CASES[case]
    seed = sum(map(ord, case))
    head, anchors, mask, sel, lay = make_decode_inputs(case, seed)
    counts = sel.sum(1)
    top = int(counts.max())
    k_cap = {"roomy": top + 37, "full": top, "over": top - 3}[cap]
    if cap == "over":
        assert (np.sort(counts)[:-1] <= k_cap).all(), "only one frame may exceed k_cap"
    rs = np.random.RandomState(seed + 1)
    n = mask.shape[1]
    zero_r = np.nonzero(anchors[0, :, 6] == 0)[0][:40]               # anchors whose r code gets +-0 (with ra = +-0)
    fill_codes(head, H, W, sel, k_cap, lay, rs, zero_r)
    head = head.reshape(B, H, W, -1)
    from sassd_b200 import lib
    L = lib.load()
    hg = Guarded(head.shape, torch.float32, dev)
    hg.t.copy_(torch.from_numpy(head))
    ag = Guarded(anchors.shape, torch.float32, dev)
    ag.t.copy_(torch.from_numpy(anchors))
    m = torch.from_numpy(mask).to(dev)
    ws = torch.full((L.sassd_decode_select_workspace_bytes(B, n),), SENTINEL, dtype=torch.uint8, device=dev)
    runs = []
    for _ in range(2):
        outs = dict(boxes=Guarded((B, k_cap, 7), torch.float32, dev), labels=Guarded((B, k_cap), torch.int32, dev),
                    index=Guarded((B, k_cap), torch.int32, dev), d_k=Guarded((B,), torch.int32, dev))
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        rc = L.sassd_decode_select(_p(hg.t), head.shape[3], B, H, W, ncls, _p(ag.t), int(per_frame), _p(m), n,
                                   ctypes.c_float(thr), _p(outs["boxes"].t), _p(outs["labels"].t), _p(outs["index"].t),
                                   _p(outs["d_k"].t), k_cap, _p(status), _p(ws), ws.numel(), _stream())
        lib.check(rc, "sassd_decode_select")
        torch.cuda.synchronize()
        outs["status"] = int(status.item())
        runs.append(outs)
    an_full = anchors if per_frame else np.repeat(anchors, B, 0)
    model = decode_model(head, ncls, an_full, mask, thr)
    assert [len(x["index"]) for x in model] == list(counts), "the inputs do not select what they were built to"
    got = runs[0]
    assert got["status"] == (FLAG_GUIDED_CAP if cap == "over" else 0), got["status"]
    check_decode(got, model, k_cap)
    if per_frame and B > 1:                 # each frame's table differs: a frame reading another's would be caught
        assert not np.array_equal(anchors[0][np.isfinite(anchors[0][:, 0])][:5], anchors[1][np.isfinite(anchors[1][:, 0])][:5])
    for g in ("boxes", "labels", "index", "d_k"):
        assert torch.equal(runs[0][g].body(), runs[1][g].body()), "second run on the dirty workspace differs: " + g
        assert runs[1][g].guards_intact()
    assert runs[1]["status"] == got["status"]
    if case == "c1-b3-shared-pad-thr05":    # the exact edges are present in this case
        lg = head.reshape(B, -1, head.shape[3])[..., head_layout(1)[0]:head_layout(1)[0] + 2]
        assert (lg == 0).sum() > 10, "no exact-0 logits"


def test_decode_model_exact_edges():
    """CPU check of the model's exact edges: sigmoid(0) = 0.5 is not selected at thr 0.5, identical class logits give
    label 0, tied direction logits do not flip, r = -0.0 stays -0.0 and +0.0 stays +0.0, r > 0 with direction label
    0 flips by fp32(pi)."""
    H, W, ncls = 1, 1, 3
    cls_off, dir_off, stride = head_layout(ncls)
    head = np.zeros((1, H, W, stride), F32)
    head[0, 0, 0, cls_off:cls_off + 3] = [1.0, 1.0, 1.0]          # anchor 0: all classes equal
    head[0, 0, 0, cls_off + 3:cls_off + 6] = [0.0, 0.0, 0.0]      # anchor 1: sigmoid exactly 0.5
    head[0, 0, 0, 6] = -0.0                                       # anchor 0: r code -0
    head[0, 0, 0, dir_off:dir_off + 2] = [0.25, 0.25]             # tie
    anchors = np.zeros((1, 2 * ncls * H * W, 7), F32)
    anchors[0, :, 3:6] = 1.0
    anchors[0, 0, 6] = -0.0
    mask = np.ones((1, 6), np.uint8)
    m = decode_model(head, ncls, anchors, mask, 0.5)[0]
    assert list(m["index"]) == [0] and list(m["labels"]) == [0]
    assert bits(m["r"])[0] == bits(F32(-0.0))
    head[0, 0, 0, 6] = 0.5
    head[0, 0, 0, dir_off:dir_off + 2] = [0.3, 0.2]               # direction label 0 with r > 0: flip
    m = decode_model(head, ncls, anchors, mask, 0.5)[0]
    assert m["r"][0] == F32(0.5) + PI32


# ------------------------------------------------------------------------------------------------------------------
# B. sassd_pswarp: fp64 bilinear reference, derived bound, mutation self-test
# ------------------------------------------------------------------------------------------------------------------
def _f(bits_):
    return float(np.array([bits_], np.uint32).view(F32)[0])


# torch.linspace(-.5, .5, 4) and (-.5, .5, 7) in fp32 as the kernel holds them
LIN4 = np.array([-0.5, _f(0xBE2AAAAA), _f(0x3E2AAAAA), 0.5], F32)
LIN7 = np.array([-0.5, _f(0xBEAAAAAA), _f(0xBE2AAAAA), _f(0xB2800000), _f(0x3E2AAAAA), _f(0x3EAAAAAA), 0.5], F32)
PI_IDX, PJ_IDX = np.arange(28) // 7, np.arange(28) % 7


def _bilinear(fm, ix, iy, ch, clamp=False):
    """Bilinear sample of fm [H, W, C] (fp64) at (ix, iy) [k, 28], channel ch [28]; zero padding (or clamping)."""
    H, W = fm.shape[:2]
    x0, y0 = np.floor(ix), np.floor(iy)
    wx, wy = ix - x0, iy - y0
    x0, y0 = x0.astype(np.int64), y0.astype(np.int64)
    acc = np.zeros(ix.shape)
    absum = np.zeros(ix.shape)
    chb = np.broadcast_to(ch, ix.shape)
    for dy, dx, w in ((0, 0, (1 - wy) * (1 - wx)), (0, 1, (1 - wy) * wx), (1, 0, wy * (1 - wx)), (1, 1, wy * wx)):
        xx, yy = x0 + dx, y0 + dy
        if clamp:
            ok = np.ones(ix.shape, bool)
            xx, yy = np.clip(xx, 0, W - 1), np.clip(yy, 0, H - 1)
        else:
            ok = (xx >= 0) & (xx < W) & (yy >= 0) & (yy < H)
        v = np.where(ok, fm[np.clip(yy, 0, H - 1), np.clip(xx, 0, W - 1), chb], 0.0)
        acc += v * w
        absum += np.abs(v)
    return acc, absum, x0, y0


def _local_gradient(fm, x0, y0, ch):
    """Largest |difference of neighbouring pixels| along x and along y around the sample's cell (rows and columns
    x0 - 1 .. x0 + 2, zero padded): a coordinate error below one pixel cannot move the sample's value by more than
    the coordinate error times it."""
    H, W = fm.shape[:2]
    fp = np.pad(fm, ((3, 3), (3, 3), (0, 0)))
    chb = np.broadcast_to(ch, x0.shape)
    gx = np.zeros(x0.shape)
    gy = np.zeros(x0.shape)
    X = np.clip(x0, -3, W + 1) + 3
    Y = np.clip(y0, -3, H + 1) + 3
    for dy in range(-1, 3):
        for dx in range(-1, 2):
            a = fp[np.clip(Y + dy, 0, H + 5), np.clip(X + dx, 0, W + 5), chb]
            b = fp[np.clip(Y + dy, 0, H + 5), np.clip(X + dx + 1, 0, W + 5), chb]
            gx = np.maximum(gx, np.abs(b - a))
            a = fp[np.clip(Y + dx, 0, H + 5), np.clip(X + dy, 0, W + 5), chb]
            b = fp[np.clip(Y + dx + 1, 0, H + 5), np.clip(X + dy, 0, W + 5), chb]
            gy = np.maximum(gy, np.abs(b - a))
    return gx, gy


def pswarp_ref(fm, boxes, off_x, off_y, sscale):
    """fp64 PSWarp of one frame: fm [H, W, >= 28] fp64, boxes [k, 7] fp32.  Returns (score [k], bound [k]).

    Sampling grid from the fp32 box in fp64 (the normalisation to [-1, 1] and grid_sample's align_corners=True
    un-normalisation cancel exactly), bilinear with zero padding, part p = i * 7 + j reads channel p, mean over 28.
    Bound, first order in the unit roundoff U = 2^-24, from the kernel's arithmetic:
      coordinate error e_ix: cosf / sinf within 2 ulp, one rounding per operation of xx * c + yy * s + xg,
        (x + off) * scale, / (W - 1), * 2 - 1, + 1, / 2, * (W - 1) (each U times the magnitude it rounds);
      value error per part: e_ix * Gx + e_iy * Gy with the local gradients, plus 6 U sum |corner| for the weights,
        products and the three adds of the four weighted corners;
      the warp-shuffle sum of the 28 parts (depth 5: 5 U sum |part|) and the division by 28 (U |score|)."""
    H, W = fm.shape[:2]
    b = boxes.astype(np.float64)
    xg, yg, wg, lg, rg = b[:, 0:1], b[:, 1:2], b[:, 3:4], b[:, 4:5], b[:, 6:7]
    c, s = np.cos(rg), np.sin(rg)
    xx = LIN4[PI_IDX].astype(np.float64)[None] * wg
    yy = LIN7[PJ_IDX].astype(np.float64)[None] * lg
    x = xx * c + yy * s + xg
    y = yy * c - xx * s + yg
    sc = float(F32(sscale))
    X, Y = (x + float(F32(off_x))) * sc, (y + float(F32(off_y))) * sc
    val, absum, x0, y0 = _bilinear(fm, X, Y, np.arange(28))
    score = val.mean(1)
    ec, es = 2 * ulp(c), 2 * ulp(s)
    axx, ayy, ac, as_ = np.abs(xx), np.abs(yy), np.abs(c), np.abs(s)

    def prod(a, t, et):            # error of fl(fl(lin * size) * trig): the lin * size rounding, trig's, the product's
        return a * et + 2 * U * a * t

    def coord_err(e_prod, mag, v, V, off, n1):
        e = e_prod + U * mag + U * np.abs(v)                                  # the two adds
        e = (e + U * np.abs(v + off)) * sc + U * np.abs(V)                    # (v + off) * scale
        gx = 2 * (V / n1) - 1
        # / (W - 1), "* 2 - 1", "+ 1", "/ 2", "* (W - 1)": the roundings of the quotient and of the product are
        # U |V| each, those of the subtraction and the addition (n1 / 2) U |.|
        return e + 2 * U * np.abs(V) + n1 / 2 * U * (np.abs(gx) + np.abs(gx + 1))

    e_ix = coord_err(prod(axx, ac, ec) + prod(ayy, as_, es), axx * ac + ayy * as_, x, X, float(F32(off_x)), W - 1)
    e_iy = coord_err(prod(ayy, ac, ec) + prod(axx, as_, es), ayy * ac + axx * as_, y, Y, float(F32(off_y)), H - 1)
    gx, gy = _local_gradient(fm, x0, y0, np.arange(28))
    per_part = gx * e_ix + gy * e_iy + 6 * U * absum
    bound = (per_part.sum(1) + 5 * U * np.abs(val).sum(1)) / 28 + U * np.abs(score) + 1e-30
    return score, bound


def pswarp_emulate(fm, boxes, off_x, off_y, sscale, corrupt=None):
    """numpy fp32 emulation of pswarp_kernel (one frame).  `corrupt` injects one defect:
      "ij"     part p reads channel j * 4 + i instead of i * 7 + j      "W"      x / W instead of x / (W - 1)
      "clamp"  out-of-range corners clamped instead of zero              "sin"    the sign of sin flipped
      "mean32" the sum divided by 32 instead of 28"""
    H, W = fm.shape[:2]
    f = fm.astype(F32)
    b = boxes.astype(F32)
    xg, yg, wg, lg, rg = b[:, 0:1], b[:, 1:2], b[:, 3:4], b[:, 4:5], b[:, 6:7]
    c, s = np.cos(rg), np.sin(rg)
    if corrupt == "sin":
        s = -s
    xx, yy = LIN4[PI_IDX][None] * wg, LIN7[PJ_IDX][None] * lg
    x = (xx * c + yy * s) + xg
    y = (yy * c - xx * s) + yg
    x = (x + F32(off_x)) * F32(sscale)
    y = (y + F32(off_y)) * F32(sscale)
    nx = F32(W) if corrupt == "W" else F32(W - 1)
    gx = x / nx * F32(2) - F32(1)
    gy = y / F32(H - 1) * F32(2) - F32(1)
    ix = (gx + F32(1)) / F32(2) * F32(W - 1)
    iy = (gy + F32(1)) / F32(2) * F32(H - 1)
    ch = PJ_IDX * 4 + PI_IDX if corrupt == "ij" else np.arange(28)
    val, _, _, _ = _bilinear(f.astype(np.float64), ix.astype(np.float64), iy.astype(np.float64), ch,
                             clamp=corrupt == "clamp")
    return (val.astype(F32).sum(1) / F32(32.0 if corrupt == "mean32" else 28.0)).astype(np.float64)


def _pswarp_case(seed, H=24, W=40, k=400, sscale=2.5, off=(0.0, 40.0)):
    """A rough random map (neighbouring pixels independent) with a smooth ramp, and boxes: inside, partly off and
    fully off the map, rotations 0, +-pi/2, pi, 3.0 and random."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    fm = rs.normal(0, 1, (H, W, 28)) + 0.05 * (xx + 2 * yy)[..., None]
    fm = fm.astype(F32).astype(np.float64)
    px = rs.uniform(-6, W + 6, k)
    py = rs.uniform(-6, H + 6, k)
    rots = np.array([0.0, np.pi / 2, -np.pi / 2, np.pi, 3.0])
    r = np.where(rs.rand(k) < 0.5, rots[rs.randint(0, 5, k)], rs.uniform(-4, 4, k))
    boxes = np.stack([px / sscale - off[0], py / sscale - off[1], rs.normal(-1, 0.1, k), rs.normal(1.6, 0.2, k) * 2,
                      rs.normal(3.9, 0.3, k) * 2, rs.normal(1.5, 0.1, k), r], 1).astype(F32)
    return fm, boxes


def excess_ratio(got, ref, bound):
    return float(np.max(np.abs(got - ref) / bound))


def test_pswarp_emulation_within_bound():
    """The fp32 emulation of the kernel stays inside the derived bound (excess <= 1)."""
    for seed in range(3):
        fm, boxes = _pswarp_case(seed)
        ref, bound = pswarp_ref(fm, boxes, 0.0, 40.0, 2.5)
        assert excess_ratio(pswarp_emulate(fm, boxes, 0.0, 40.0, 2.5), ref, bound) <= 1.0


@pytest.mark.parametrize("corrupt", ["ij", "W", "clamp", "sin", "mean32"])
def test_pswarp_mutations_are_rejected(corrupt):
    """The bound can fail: each single defect of the emulated kernel misses it by at least 10x (factor printed)."""
    fm, boxes = _pswarp_case(7)
    ref, bound = pswarp_ref(fm, boxes, 0.0, 40.0, 2.5)
    good = excess_ratio(pswarp_emulate(fm, boxes, 0.0, 40.0, 2.5), ref, bound)
    bad = excess_ratio(pswarp_emulate(fm, boxes, 0.0, 40.0, 2.5, corrupt=corrupt), ref, bound)
    print("pswarp defect %-7s rejected by %.3g x the bound (defect-free emulation %.3g)" % (corrupt, bad, good))
    assert good <= 1.0 and bad >= 10.0, (corrupt, good, bad)


PSWARP_CASES = {
    # name: (B, H, W, feat_stride, k_cap, d_k per frame, off_x, off_y, scale)
    "mixed": (3, 24, 40, 33, 300, (0, 350, 123), 0.0, 40.0, 2.5),
    "integer": (2, 16, 20, 28, 64, (40, 64), 0.0, 0.0, 1.0),
    "grid_stride": (2, 40, 48, 28, 8192, (8192, 5000), 0.0, 40.0, 2.5),
}


def _pswarp_inputs(case):
    B, H, W, stride, k_cap, dks, ox, oy, sc = PSWARP_CASES[case]
    rs = np.random.RandomState(len(case))
    maps = np.full((B, H, W, stride), np.nan, F32)                   # channels 28 .. stride-1 stay NaN
    boxes = np.full((B, k_cap, 7), np.nan, F32)                      # rows >= d_k stay NaN
    for b in range(B):
        fm, bx = _pswarp_case(100 * b + len(case), H, W, k_cap, sc, (ox, oy))
        maps[b, ..., :28] = fm
        boxes[b] = bx
    if case == "integer":
        # r = 0, w = 2, l = 6 on integer centres: x samples at xg +-1 (integers) and +-1/3, y at yg + -3 .. 3 (all
        # integers up to the 1e-8 rounding of linspace's middle tap); centres at 0 (negative coordinates) and at
        # (W - 2, H - 4) in the last frame, so that samples fall on x = W - 1 and y = H - 1 of the last map, whose
        # out-of-range corner lies in the NaN guard after the allocation
        for b in range(B):
            n_int = 30
            cx = rs.randint(0, W, n_int).astype(F32)
            cy = rs.randint(0, H, n_int).astype(F32)
            cx[:3], cy[:3] = 0, 0
            cx[3:6], cy[3:6] = W - 2, H - 4
            cx[6], cy[6] = W - 1, H - 1
            boxes[b, :n_int] = np.stack([cx, cy, np.zeros(n_int), np.full(n_int, 2.0), np.full(n_int, 6.0),
                                         np.ones(n_int), np.zeros(n_int)], 1)
    for b in range(B):
        k = min(dks[b], k_cap)
        boxes[b, k:] = np.nan
        boxes[b, :, 2] = np.nan                                      # z and h are never read
        boxes[b, :, 5] = np.nan
        # fully off the map: score exactly 0
        boxes[b, 7:10, 0] = -100.0
    return maps, boxes


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PSWARP_CASES))
def test_pswarp_vs_fp64(dev, case):
    """Every score within the derived bound of the fp64 reference (frames with different maps, NaN padding channels
    and NaN guards around map and boxes); boxes fully off the map score exactly 0; d_k = 0, d_k > k_cap (clamped) and
    k_cap = 8192 (the grid-stride loop: 592 CTAs x 8 warps cover 4736 boxes per pass); score rows at or beyond d_k
    and the guards untouched."""
    from sassd_b200 import lib
    B, H, W, stride, k_cap, dks, ox, oy, sc = PSWARP_CASES[case]
    maps, boxes = _pswarp_inputs(case)
    mg = Guarded(maps.shape, torch.float32, dev)
    mg.t.copy_(torch.from_numpy(maps))
    bg = Guarded(boxes.shape, torch.float32, dev)
    bg.t.copy_(torch.from_numpy(boxes))
    d_k = torch.tensor(dks, dtype=torch.int32, device=dev)
    scores = Guarded((B, k_cap), torch.float32, dev)
    rc = lib.load().sassd_pswarp(_p(mg.t), stride, B, H, W, _p(bg.t), _p(d_k), k_cap, ctypes.c_float(ox),
                                 ctypes.c_float(oy), ctypes.c_float(sc), _p(scores.t), _stream())
    lib.check(rc, "sassd_pswarp")
    torch.cuda.synchronize()
    got = scores.t.cpu().numpy()
    for b in range(B):
        k = min(dks[b], k_cap)
        g = got[b, :k].astype(np.float64)
        assert np.isfinite(g).all(), "frame %d: NaN score (a read of a padding channel, guard or unused column)" % b
        ref, bound = pswarp_ref(maps[b, ..., :28].astype(np.float64), boxes[b, :k], ox, oy, sc)
        err = np.abs(g - ref)
        record("pswarp score", err, bound)
        assert (err <= bound).all(), "frame %d: %d scores outside the bound, worst %.3g x" % (
            b, int((err > bound).sum()), float((err / bound).max()))
        if k > 9:
            assert (got[b, 7:10] == 0).all(), "boxes fully off the map must score exactly 0"
        assert untouched(scores.t[b, k:]), "frame %d: score rows at or beyond d_k written" % b
    assert scores.guards_intact()


# ------------------------------------------------------------------------------------------------------------------
# C. sassd_rescore_nms against a model built from verified parts
# ------------------------------------------------------------------------------------------------------------------
SCORE_THR, IOU_THR = 0.3, 0.1
STRAY_LOGIT = 8.0                    # score rows the kernel must not read: above every real logit (<= 4.6)


def greedy_keep(mask, n):
    """The reference host loop (iou3d.cpp) on a suppression bitmask [n, >= ceil(n / 64)] uint64."""
    colb = (n + 63) // 64
    removed = np.zeros(colb, np.uint64)
    keep = []
    for i in range(n):
        if not (int(removed[i >> 6]) >> (i & 63)) & 1:
            keep.append(i)
            removed |= mask[i, :colb]
    return np.array(keep, np.int64)


def bev_of(b7):
    """boxes3d_to_bev_torch in fp32 (half extents from columns 3 and 4)."""
    b7 = b7.astype(F32)
    hl, hw = b7[:, 3] / F32(2), b7[:, 4] / F32(2)
    return np.stack([b7[:, 0] - hl, b7[:, 1] - hw, b7[:, 0] + hl, b7[:, 1] + hw, b7[:, 6]], 1).astype(F32)


def rescore_frame(k, n_pass, seed, ties=True):
    """k candidates, n_pass of them above the score threshold (logits distinct by >= 1e-3 but for tie groups of
    identical logits), boxes in clusters of heavy overlap spread over 40 x 40 m, labels 0..2."""
    rs = np.random.RandomState(seed)
    logits = np.full(k, np.nan, F32)
    passing = np.sort(rs.choice(k, n_pass, replace=False)) if n_pass else np.zeros(0, np.int64)
    fail = np.setdiff1d(np.arange(k), passing)
    logits[fail] = (-1.2 - 1e-3 * rs.permutation(len(fail))).astype(F32)
    grid = -0.5 + 1e-3 * rs.permutation(max(n_pass, 1))[:n_pass]
    logits[passing] = grid.astype(F32)
    if ties and n_pass >= 8:
        # a group of identical logits larger than 64 where possible (crosses a 64-boundary of the sorted order), and
        # a few small groups
        g = rs.choice(passing, min(70, n_pass // 2), replace=False)
        logits[g] = logits[g[0]]
        for _ in range(5):
            g = rs.choice(passing, 3, replace=False)
            logits[g] = logits[g[0]]
    centres = rs.uniform(-20, 20, (max(k // 6, 1), 2))
    ci = rs.randint(0, len(centres), k)
    b7 = np.stack([centres[ci, 0] + rs.normal(0, 0.4, k), centres[ci, 1] + rs.normal(0, 0.4, k), rs.normal(-1, 0.2, k),
                   rs.normal(1.6, 0.1, k), rs.normal(3.9, 0.3, k), rs.normal(1.5, 0.1, k), rs.uniform(-3.2, 3.2, k)],
                  1).astype(F32)
    labels = rs.randint(0, 3, k).astype(np.int32)
    return b7, logits, labels


def rescore_model(dev, b7, logits, labels, det_cap):
    """Expected (det rows [m, 9] with the score column in fp64, score bounds, kept count before the cap, NMS_CAP hit).
    Order: score descending, then candidate index; the first NMS_CAP passing candidates in candidate order survive
    an overflow.  The suppression mask comes from sassd_nms_mask on the fp32 BEV boxes (held bit for bit to the
    reference kernel by part D), the keep list from the reference's greedy loop."""
    from sassd_b200 import lib
    s = sigmoid64(logits)
    passing = np.nonzero(s > float(F32(SCORE_THR)))[0]
    over = len(passing) > NMS_CAP
    passing = passing[:NMS_CAP]
    order = passing[np.lexsort((passing, -s[passing]))]
    n = len(order)
    if n == 0:
        return np.zeros((0, 9)), np.zeros(0), 0, over
    bev = torch.from_numpy(bev_of(b7[order])).to(dev)
    colb = (n + 63) // 64
    mask = torch.zeros((n, colb), dtype=torch.int64, device=dev)
    lib.check(lib.load().sassd_nms_mask(_p(bev), n, ctypes.c_float(IOU_THR), _p(mask), _stream()), "sassd_nms_mask")
    torch.cuda.synchronize()
    keep = greedy_keep(mask.cpu().numpy().view(np.uint64), n)
    src = order[keep][:det_cap]
    rows = np.concatenate([b7[src].astype(np.float64), s[src, None], labels[src, None].astype(np.float64)], 1)
    return rows, sigmoid_bound(logits[src]), len(keep), over


def run_rescore(dev, frames, det_cap, k_cap=None, dk_extra=None, ws=None):
    """frames: list of (b7 [k, 7], logits [k], labels [k]).  Box rows at or beyond each frame's k are NaN and score
    rows there hold STRAY_LOGIT, so a read of them would add the best-scoring candidate (with a NaN box); dk_extra
    {frame: d_k} overrides d_k (above k_cap: the kernel clamps; rows past k_cap are the next frame's)."""
    from sassd_b200 import lib
    L = lib.load()
    B = len(frames)
    k_cap = k_cap or max(max(len(f[1]) for f in frames), 1)
    b7 = np.full((B, k_cap, 7), np.nan, F32)
    sc = np.full((B, k_cap), STRAY_LOGIT, F32)
    lab = np.full((B, k_cap), -1, np.int32)
    dk = np.zeros(B, np.int32)
    for i, (b, s, l) in enumerate(frames):
        b7[i, :len(s)], sc[i, :len(s)], lab[i, :len(s)], dk[i] = b, s, l, len(s)
    for i, v in (dk_extra or {}).items():
        dk[i] = v
    bg, sg, lg = (Guarded(a.shape, torch.float32 if a.dtype == F32 else torch.int32, dev) for a in (b7, sc, lab))
    for g, a in ((bg, b7), (sg, sc), (lg, lab)):
        g.t.copy_(torch.from_numpy(a))
    d_k = torch.from_numpy(dk).to(dev)
    det = Guarded((B, det_cap, 9), torch.float32, dev)
    d_ndet = Guarded((B,), torch.int32, dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    nb = L.sassd_rescore_nms_workspace_bytes(B, k_cap, NMS_CAP)
    if ws is None:
        ws = torch.full((nb,), SENTINEL, dtype=torch.uint8, device=dev)
    rc = L.sassd_rescore_nms(_p(bg.t), _p(sg.t), _p(lg.t), _p(d_k), B, k_cap, ctypes.c_float(SCORE_THR),
                             ctypes.c_float(IOU_THR), NMS_CAP, _p(det.t), _p(d_ndet.t), det_cap, _p(status), _p(ws),
                             ws.numel(), _stream())
    lib.check(rc, "sassd_rescore_nms")
    torch.cuda.synchronize()
    return det, d_ndet, int(status.item()), ws


def check_rescore(dev, frames, det, d_ndet, det_cap):
    nd = d_ndet.t.cpu().numpy()
    got = det.t.cpu().numpy()
    kept = []
    for i, (b7, lg, lab) in enumerate(frames):
        rows, sb, nkeep, _ = rescore_model(dev, b7, lg, lab, det_cap)
        kept.append(nkeep)
        m = len(rows)
        assert nd[i] == m, "frame %d: d_ndet %d, expected %d" % (i, nd[i], m)
        g = got[i, :m]
        assert np.array_equal(bits(g[:, :7]), bits(rows[:, :7].astype(F32))), "frame %d: boxes / order differ" % i
        assert np.array_equal(g[:, 8], rows[:, 8].astype(F32)), "frame %d: labels differ" % i
        err = np.abs(g[:, 7].astype(np.float64) - rows[:, 7])
        record("rescore score", err, sb)
        assert (err <= sb).all(), "frame %d: scores outside the bound" % i
        assert untouched(det.t[i, m:]), "frame %d: det rows at or beyond d_ndet written" % i
    assert det.guards_intact() and d_ndet.guards_intact()
    return kept


# frames of one batch: (k, passing).  d_k of the frame "dk>kcap" is set 500 above k_cap; it comes first, so an
# unclamped read would take rows 0..499 of the next frame ("k0"), which all hold STRAY_LOGIT
RESCORE_FRAMES = {"dk>kcap": (4400, 3000), "k0": (0, 0), "below": (300, 0), "one": (40, 1), "p63": (100, 63),
                  "p64": (100, 64), "p65": (90, 65), "k1024": (1024, 700), "k1025": (1025, 1025),
                  "p4096": (4400, 4096)}


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["full", "nms_cap", "det_cap"])
def test_rescore_nms(dev, what):
    """full: frames of k = 0, all below the threshold, 1 / 63 / 64 / 65 passing, k = 1024 / 1025 (either side of the
    1024-thread loop), exactly 4096 passing (64 mask words per row, a 4096-entry sort), d_k > k_cap; det_cap equal to
    the largest kept count: no flag.  nms_cap: 4097 passing: flag 8, the first 4096 passing candidates in candidate
    order go on.  det_cap: det_cap below one frame's kept count: flag 32, that frame keeps its first det_cap boxes in
    score order, the other is unchanged.  Everything against the model, rows beyond d_ndet untouched."""
    if what == "full":
        names = list(RESCORE_FRAMES)
        frames = [rescore_frame(k, n, seed=i) for i, (k, n) in enumerate(RESCORE_FRAMES.values())]
        k_cap = 4400
        kept = [rescore_model(dev, *f, det_cap=NMS_CAP)[2] for f in frames]
        det_cap = max(kept)
        det, d_ndet, status, _ = run_rescore(dev, frames, det_cap, k_cap=k_cap,
                                             dk_extra={names.index("dk>kcap"): k_cap + 500})
        assert status == 0, status
        check_rescore(dev, frames, det, d_ndet, det_cap)
        assert kept[names.index("below")] == 0 and kept[names.index("k0")] == 0
    elif what == "nms_cap":
        frames = [rescore_frame(4300, 4097, seed=40), rescore_frame(90, 65, seed=41)]
        # the 4097th passing candidate gets the best score: a kernel keeping the best 4096 instead would include it
        last = np.nonzero(sigmoid64(frames[0][1]) > SCORE_THR)[0][-1]
        frames[0][1][last] = F32(8.0)
        det, d_ndet, status, _ = run_rescore(dev, frames, NMS_CAP)
        assert status == FLAG_NMS_CAP, status
        check_rescore(dev, frames, det, d_ndet, NMS_CAP)
        assert not np.isin(det.t[0, :, 0].cpu().numpy(), frames[0][0][last, 0]).any()
    else:
        frames = [rescore_frame(1025, 1025, seed=50), rescore_frame(100, 63, seed=51)]
        kept = [rescore_model(dev, *f, det_cap=NMS_CAP)[2] for f in frames]
        det_cap = kept[0] - 7
        assert kept[1] <= det_cap
        det, d_ndet, status, _ = run_rescore(dev, frames, det_cap)
        assert status == FLAG_DET_CAP, status
        check_rescore(dev, frames, det, d_ndet, det_cap)


@pytest.mark.gpu
def test_rescore_nms_dirty_workspace(dev):
    """The rescoring path never clears its suppression bitmask: a large frame, then a small one on the same
    workspace, then the small one again on a workspace filled with 0xFF give the same bytes."""
    big = [rescore_frame(4400, 4096, seed=60)]
    small = [rescore_frame(300, 130, seed=61)]
    _, _, _, ws = run_rescore(dev, big, 512, k_cap=4400)
    det1, nd1, st1, ws = run_rescore(dev, small, 512, k_cap=4400, ws=ws)
    ws.fill_(SENTINEL)
    det2, nd2, st2, _ = run_rescore(dev, small, 512, k_cap=4400, ws=ws)
    assert st1 == st2 == 0
    assert torch.equal(det1.body(), det2.body()) and torch.equal(nd1.body(), nd2.body())
    assert det2.guards_intact() and nd2.guards_intact()
    check_rescore(dev, small, det1, nd1, 512)


# ------------------------------------------------------------------------------------------------------------------
# D. rotated IoU and NMS at degenerate geometry, bit for bit against the reference kernel (tests/golden/nms.npz)
# ------------------------------------------------------------------------------------------------------------------
ADV_SETS = ["adv_" + k for k in GROUPS] + ["adv_mix%d" % n for n in MIX_SIZES]


@pytest.fixture(scope="module")
def nms_golden(golden_dir):
    return np.load(os.path.join(golden_dir, "nms.npz"))


def test_adversarial_sets_match_golden(nms_golden):
    """The box sets are regenerated identically (CPU): the stored reference outputs belong to these boxes."""
    from tests.nms_box_sets import adversarial_sets
    for name, b in adversarial_sets().items():
        assert np.array_equal(b.view(np.int32), nms_golden[name + "_bev"].view(np.int32)), name


def thr_key(thr):
    return "t%g" % thr


@pytest.mark.gpu
@pytest.mark.parametrize("thr", THRESHOLDS, ids=thr_key)
@pytest.mark.parametrize("name", ADV_SETS + ["rand%d" % RANDOM_N])
def test_nms_mask_vs_reference(dev, nms_golden, name, thr):
    """sassd_nms_mask's upper triangle (column blocks >= the row's block) is bit-identical to the reference kernel's
    mask, including the pairs on both sides of the far-pair shortcut (reach^2 * 1.002 + 1e-6); nothing is written
    outside the [n, ceil(n / 64)] mask."""
    from sassd_b200 import lib
    boxes = nms_golden[name + "_bev"]
    ref = nms_golden["%s_mask_%s" % (name, thr_key(thr))]
    n = len(boxes)
    colb = (n + 63) // 64
    bg = Guarded(boxes.shape, torch.float32, dev)
    bg.t.copy_(torch.from_numpy(boxes))
    mask = Guarded((n, colb), torch.int64, dev)
    lib.check(lib.load().sassd_nms_mask(_p(bg.t), n, ctypes.c_float(thr), _p(mask.t), _stream()), "sassd_nms_mask")
    torch.cuda.synchronize()
    got = mask.t.cpu().numpy().view(np.uint64)
    upper = np.arange(colb)[None, :] >= (np.arange(n) // 64)[:, None]
    diff = np.nonzero((got != ref) & upper)
    assert len(diff[0]) == 0, "%d mask words differ, first (row, word) %s" % (len(diff[0]), list(zip(*diff))[:4])
    assert mask.guards_intact()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ADV_SETS)
def test_boxes_iou_bev_vs_reference(dev, nms_golden, name):
    """sassd_boxes_iou_bev over the full [n, n] matrix (diagonal and lower triangle included) is bit-identical to the
    reference kernel's boxesioubevLauncher."""
    from sassd_b200 import lib
    boxes = nms_golden[name + "_bev"]
    ref = nms_golden[name + "_iou"]
    n = len(boxes)
    bg = Guarded(boxes.shape, torch.float32, dev)
    bg.t.copy_(torch.from_numpy(boxes))
    iou = Guarded((n, n), torch.float32, dev)
    lib.check(lib.load().sassd_boxes_iou_bev(_p(bg.t), n, _p(bg.t), n, _p(iou.t), _stream()), "sassd_boxes_iou_bev")
    torch.cuda.synchronize()
    got = iou.t.cpu().numpy()
    diff = np.nonzero(got.view(np.int32) != ref.view(np.int32))
    assert len(diff[0]) == 0, "%d IoU values differ, first %s: got %s ref %s" % (
        len(diff[0]), list(zip(*diff))[:4], got[diff][:4], ref[diff][:4])
    assert iou.guards_intact()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 4097, RANDOM_N])
def test_nms_sorted_vs_reference_greedy(dev, nms_golden, n):
    """sassd_nms_sorted's keep list equals the reference's greedy loop on the reference kernel's mask: n = 0, 1,
    4097 (65 mask words, past the 64 of the rescoring path) and 5000 (shared memory sized at run time); keep entries
    beyond the count untouched.  n = 0 asks for a 0-byte workspace and passes none."""
    from sassd_b200 import lib
    L = lib.load()
    if n == 1:
        boxes, ref = nms_golden["n1_seed0_bev"], nms_golden["n1_seed0_mask"]
    else:
        boxes = nms_golden["rand%d_bev" % RANDOM_N][:max(n, 1)]
        ref = nms_golden["rand%d_mask_%s" % (RANDOM_N, thr_key(IOU_THR))]
    exp = greedy_keep(ref, n) if n else np.zeros(0, np.int64)
    bg = Guarded(boxes.shape, torch.float32, dev)
    bg.t.copy_(torch.from_numpy(np.ascontiguousarray(boxes)))
    keep = Guarded((max(n, 1),), torch.int64, dev)
    d_nkeep = Guarded((1,), torch.int32, dev)
    nb = L.sassd_nms_workspace_bytes(n)
    ws = torch.full((nb,), SENTINEL, dtype=torch.uint8, device=dev) if nb else None    # n = 0: no workspace
    lib.check(L.sassd_nms_sorted(_p(bg.t), n, ctypes.c_float(IOU_THR), _p(keep.t), _p(d_nkeep.t), _p(ws), nb,
                                 _stream()), "sassd_nms_sorted")
    torch.cuda.synchronize()
    m = int(d_nkeep.t.item())
    assert m == len(exp), (m, len(exp))
    assert np.array_equal(keep.t[:m].cpu().numpy(), exp)
    assert untouched(keep.t[m:])
    assert keep.guards_intact() and d_nkeep.guards_intact()


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
        print("\nlargest |err| / bound:")
        for k, r in sorted(MAX_RATIO.items()):
            print("  %-16s %.3e" % (k, r))
