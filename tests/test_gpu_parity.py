"""GPU parity tests (run on the B200 box): every CUDA stage, called through the C ABI
(ctypes), against the CPU oracle on the same seeded inputs and against the committed
golden fixtures produced by the reference's own Python.

Bar: bit-exact for voxel indices, rulebooks, anchors masks and NMS keep masks; fp32
feature / score / box tolerances are written next to each assertion.
"""
import os

import numpy as np
import pytest
import torch

from oracle import ref_pipeline as O
from sassd_b200.synth import synth_cloud

pytestmark = pytest.mark.gpu

VS = [0.05, 0.05, 0.1]
RG = [0, -40., -3., 70.4, 40., 1.]
CAR = dict(sizes=[1.6, 3.9, 1.56], anchor_strides=[0.4, 0.4, 1.0], anchor_offsets=[0.2, -39.8, -1.78],
           rotations=[0, 1.57])
PED = dict(CAR, sizes=[0.6, 0.8, 1.73])
CYC = dict(CAR, sizes=[0.6, 1.76, 1.73])
ORACLE_CFG = dict(voxel_size=VS, pc_range=RG, max_points=5, max_voxels=20000, sparse_shape=[40, 1600, 1408],
                  anchor_cfgs=[CAR], grid_offsets=(0., 40.), featmap_stride=.4, score_thr=0.3, iou_thr=0.1)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def vg(dev):
    from sassd_b200.voxel_generator import VoxelGenerator
    return VoxelGenerator(VS, RG, 5, 20000, device="cuda:0")


def _sd_from(z, prefix):
    return {k[len(prefix):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix)}


# ------------------------------------------------------------------ a1 voxelizer
def test_voxelize_golden_cases(vg, golden_dir):
    from sassd_b200.voxel_generator import VoxelGenerator
    z = np.load(os.path.join(golden_dir, "voxelize.npz"))
    for tag in ("small", "small_trunc", "edge"):
        maxv = int(z[tag + "_maxv"]) if tag + "_maxv" in z.files else 20000
        g = VoxelGenerator(VS, RG, 5, maxv, device="cuda:0")
        v, c, n = g.generate(z[tag + "_points"])
        assert np.array_equal(c, z[tag + "_coors"]), tag
        assert np.array_equal(n, z[tag + "_num"]), tag
        assert np.array_equal(v, z[tag + "_voxels"]), tag
    v, c, n = vg.generate(np.zeros((0, 4), np.float32))
    assert v.shape == (0, 5, 4) and c.shape == (0, 3) and n.shape == (0,)


@pytest.mark.parametrize("seed,fov", [(0, 28.0), (1, 45.0), (2, 180.0)])
def test_voxelize_full_clouds_bit_exact(vg, seed, fov):
    pts = synth_cloud(seed, fov_deg=fov)
    v, c, n = vg.generate(pts)
    vo, co, no = O.points_to_voxel(pts, VS, RG, 5, 20000)
    assert c.shape[0] == co.shape[0]
    assert np.array_equal(c, co) and np.array_equal(n, no) and np.array_equal(v, vo)
    if fov > 40:
        assert c.shape[0] == 20000  # the max_voxels cut is exercised


def test_voxelize_batch_and_mean(vg, dev):
    clouds = [synth_cloud(3), np.zeros((0, 4), np.float32), synth_cloud(4, fov_deg=45.0), synth_cloud(5)[:777]]
    counts = [p.shape[0] for p in clouds]
    pts = torch.from_numpy(np.concatenate(clouds, 0)).to(dev)
    off = torch.tensor(np.concatenate([[0], np.cumsum(counts)]), dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    voxels, coors, num, mean, frame_rows = vg.generate_device(pts, off, len(clouds), max(counts), status)
    fr = frame_rows.cpu().numpy()
    assert int(status.item()) == 0
    exp = [O.points_to_voxel(p, VS, RG, 5, 20000) for p in clouds]
    assert np.array_equal(np.diff(fr), [e[1].shape[0] for e in exp])
    for b, (vo, co, no) in enumerate(exp):
        s, e = fr[b], fr[b + 1]
        assert np.array_equal(coors[s:e, 1:].cpu().numpy(), co)
        assert np.all(coors[s:e, 0].cpu().numpy() == b)
        assert np.array_equal(num[s:e].cpu().numpy(), no)
        assert np.array_equal(voxels[s:e].cpu().numpy(), vo)
        if e > s:
            ref = O.simple_voxel(vo, no).numpy()
            np.testing.assert_allclose(mean[s:e].cpu().numpy(), ref, rtol=1e-6, atol=1e-6)
    # SimpleVoxel module alone (vxnet.py:110-116), golden from the reference class
    from sassd_b200.backbones import SimpleVoxel
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "voxelize.npz"))
    m = np.load(os.path.join(os.path.dirname(__file__), "golden", "modules.npz"))
    out = SimpleVoxel(4)(torch.from_numpy(z["small_voxels"]).to(dev), torch.from_numpy(z["small_num"]).to(dev))
    np.testing.assert_allclose(out.cpu().numpy(), m["sv_out"], rtol=1e-6, atol=1e-6)


# ------------------------------------------------------------------ a18 anchors + mask
def test_anchor_mask_bit_exact(vg, golden_dir):
    from sassd_b200.anchors import AnchorGeneratorStride, AnchorSet
    a = np.load(os.path.join(golden_dir, "anchors.npz"))
    z = np.load(os.path.join(golden_dir, "voxelize.npz"))
    for tag, cfgs in (("car", [CAR]), ("multi", [CAR, PED, CYC])):
        aset = AnchorSet([AnchorGeneratorStride(**c) for c in cfgs], vg, device="cuda:0")
        assert aset.anchors.shape[0] == int(a[tag + "_n"])
        np.testing.assert_array_equal(aset.anchors[:6], a[tag + "_anchors_head"])
        for ctag in ("small", "edge"):
            mask = aset.mask(z[ctag + "_coors"])
            assert np.array_equal(np.packbits(mask), a["%s_mask_%s" % (tag, ctag)]), (tag, ctag)
    aset = AnchorSet([AnchorGeneratorStride(**CAR)], vg, device="cuda:0")
    _, c, _ = O.points_to_voxel(synth_cloud(0), VS, RG, 5, 20000)
    mask = aset.mask(c)
    assert np.array_equal(np.packbits(mask), a["car_mask_full20k"])
    assert aset.mask(np.zeros((0, 3), np.int32)).sum() == 0


# ------------------------------------------------------------------ a5 rulebooks
def _random_sparse(B, shape, n, cin, seed):
    rs = np.random.RandomState(seed)
    cells = rs.choice(B * shape[0] * shape[1] * shape[2], size=n, replace=False)
    c = np.zeros((n, 4), np.int32)
    r = cells.copy()
    c[:, 3] = r % shape[2]; r //= shape[2]
    c[:, 2] = r % shape[1]; r //= shape[1]
    c[:, 1] = r % shape[0]; r //= shape[0]
    c[:, 0] = r
    return c, torch.from_numpy(rs.randn(n, cin).astype(np.float32))


def _frame_coords(seeds):
    cl = []
    for b, s in enumerate(seeds):
        _, c, _ = O.points_to_voxel(synth_cloud(s), VS, RG, 5, 20000)
        cl.append(np.pad(c, ((0, 0), (1, 0)), constant_values=b))
    return np.concatenate(cl, 0).astype(np.int32)


def _tile_masks(nbr):
    """per 128-row tile: bit k set when some row of the tile has a neighbour at offset k (SASSD_SPCONV_TILE_ROWS)."""
    n, taps = nbr.shape
    nt = (n + 127) // 128
    pad = np.full((nt * 128, taps), -1, np.int64)
    pad[:n] = nbr
    present = (pad.reshape(nt, 128, taps) >= 0).any(1)
    return (present * (1 << np.arange(taps))[None, :]).sum(1).astype(np.int32)


@pytest.mark.parametrize("case", ["random", "lidar"])
def test_rulebooks_bit_exact(dev, case):
    from sassd_b200 import ops, spconv
    if case == "random":
        B, shape = 3, [9, 21, 17]
        coords, _ = _random_sparse(B, shape, 700, 4, 0)
    else:
        B, shape = 2, [40, 1600, 1408]
        coords = _frame_coords([0, 1])
    x = spconv.SparseConvTensor(torch.zeros((coords.shape[0], 4), device=dev), torch.from_numpy(coords).to(dev),
                                shape, B)
    nbr, tmask = ops.rulebook_subm(x._indices, x.d_rows, shape, x.hash_index())
    onbr_s = O.subm_rulebook(coords, shape)
    assert np.array_equal(nbr.cpu().numpy(), onbr_s)
    assert np.array_equal(tmask.cpu().numpy(), _tile_masks(onbr_s))          # taps present per 128-row tile
    cap = min(8 * coords.shape[0], B * int(np.prod(ops.conv_out_shape(shape))))
    co, dn, nbr2, so, tmask2 = ops.rulebook_conv(x._indices, x.d_rows, B, shape, x.hash_index(), cap, x.status)
    oc, onbr, oshape = O.sparse_conv_rulebook(coords, shape)
    n = int(dn.item())
    assert so == oshape and n == oc.shape[0]
    assert np.array_equal(co[:n].cpu().numpy(), oc)          # sorted by flattened (b,z,y,x)
    assert np.array_equal(nbr2[:n].cpu().numpy(), onbr)
    assert np.array_equal(tmask2[: (n + 127) // 128].cpu().numpy(), _tile_masks(onbr))
    x.check_status()
    # spconv-v1 tables (canonical order)
    pairs, num = ops.rulebook_pairs(nbr2, dn)
    op, on = O.nbr_to_indice_pairs(onbr, n_cap=cap)
    assert np.array_equal(num.cpu().numpy(), on)
    assert np.array_equal(pairs.cpu().numpy(), op)
    # the fused form (the product path): the compaction pass hashes the output level as it writes the rows; the SubM
    # table of that level built on this hash must equal the oracle's (and the one built on a separate hash_build)
    idx_out = ops.HashIndex(cap, dev)
    co2, dn2, so2 = ops.rulebook_conv_outputs(x._indices, x.d_rows, B, shape, cap, x.status, ws_key="t_fused",
                                              index_out=idx_out)
    assert int(dn2.item()) == n and so2 == oshape and np.array_equal(co2[:n].cpu().numpy(), oc)
    nbr_next, _ = ops.rulebook_subm(co2, dn2, so2, idx_out)
    assert np.array_equal(nbr_next[:n].cpu().numpy(), O.subm_rulebook(oc, oshape))
    idx_sep = ops.hash_build(ops.HashIndex(cap, dev), co, dn, B, so, x.status)
    nbr_sep, _ = ops.rulebook_subm(co, dn, so, idx_sep)
    assert np.array_equal(nbr_next[:n].cpu().numpy(), nbr_sep[:n].cpu().numpy())
    x.check_status()


def test_rulebook_capacity_overflow_is_flagged(dev):
    from sassd_b200 import ops, spconv
    B, shape = 1, [8, 16, 16]
    coords, _ = _random_sparse(B, shape, 300, 4, 5)
    x = spconv.SparseConvTensor(torch.zeros((300, 4), device=dev), torch.from_numpy(coords).to(dev), shape, B)
    co, dn, nbr, so, _ = ops.rulebook_conv(x._indices, x.d_rows, B, shape, x.hash_index(), 10, x.status)
    assert int(dn.item()) == 10 and (int(x.status.item()) & 2)


# ------------------------------------------------------------------ a6/a7/a8 sparse conv + dense
PRECS = ["f16x3", "fp32"]


def _prec(name):
    from sassd_b200 import ops
    return {"fp32": ops.PREC_FP32, "tf32x3": ops.PREC_TF32X3, "f16x3": ops.PREC_F16X3}[name]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("cin,cout", [(4, 16), (16, 32), (64, 64), (32, 64)])
def test_sparse_conv_layers(dev, cin, cout, prec):
    from sassd_b200 import spconv
    B, shape = 2, [10, 24, 20]
    coords, feats = _random_sparse(B, shape, 1500, cin, cin + cout)
    w = torch.randn(3, 3, 3, cin, cout) * 0.1
    x = spconv.SparseConvTensor(feats.to(dev), torch.from_numpy(coords).to(dev), shape, B)
    sub = spconv.SubMConv3d(cin, cout, 3, bias=False, indice_key="s").to(dev)
    sub.precision = _prec(prec)
    sub.weight.data.copy_(w)
    y = sub(x)
    ref = O.indice_conv(feats, w.reshape(27, cin, cout), O.subm_rulebook(coords, shape))
    # fp32 FFMA / 3xFP16 tensor cores vs torch CPU mm + index_add: different summation order only
    np.testing.assert_allclose(y.features.cpu().numpy(), ref.numpy(), rtol=1e-4, atol=2e-5)
    dwn = spconv.SparseConv3d(cin, cout, 3, 2, padding=1, bias=False, indice_key="d").to(dev)
    dwn.precision = _prec(prec)
    dwn.weight.data.copy_(w)
    y2 = dwn(x)
    oc, onbr, oshape = O.sparse_conv_rulebook(coords, shape)
    ref2 = O.indice_conv(feats, w.reshape(27, cin, cout), onbr)
    assert np.array_equal(y2.indices.cpu().numpy(), oc) and y2.spatial_shape == oshape
    np.testing.assert_allclose(y2.features.cpu().numpy(), ref2.numpy(), rtol=1e-4, atol=2e-5)
    # dense(): [B, C, D, H, W] with zeros off the active set
    d = y2.dense()
    refd = O.dense_bev(ref2, oc, oshape, B).view(B, cout, *oshape)
    np.testing.assert_allclose(d.cpu().numpy(), refd.numpy(), rtol=1e-4, atol=2e-5)


def _make_model(dev, num_class=1, cfg_name="car_cfg.py", prec=None):
    """prec None = the product default (3xFP16 tcgen05 kernels); "fp32" / "tf32x3" select the other paths."""
    import sassd_b200 as S
    from sassd_b200 import checkpoint, ops
    cfg = S.Config.fromfile(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "configs", cfg_name))
    model, vgen, aset = S.build_from_config(cfg, device="cuda:0")
    sd = checkpoint.make_synthetic_state_dict(0, num_class)
    n, missing = checkpoint.load_state_dict_into(model, sd)
    assert all(("num_batches" in k) or k.startswith("neck.point_") for k in missing)
    assert model.neck.fcn.precision == ops.PREC_F16X3 and model.rpn_head.precision == ops.PREC_F16X3, \
        "the tensor-core path must be the default"
    if prec is not None and prec != "f16x3":
        model.set_precision(_prec(prec))
    return model, sd


@pytest.fixture(scope="module", params=PRECS)
def car_model(dev, request):
    return _make_model(dev, prec=request.param)


def test_vxnet_full_frames(dev, car_model):
    """The 13 ruled sparse convs + 1x1x1 on two real-size frames vs the oracle."""
    from sassd_b200 import spconv
    model, sd = car_model
    vl, cl, nl = [], [], []
    for s in (0, 1):
        v, c, n = O.points_to_voxel(synth_cloud(s), VS, RG, 5, 20000)
        vl.append(v); cl.append(c); nl.append(n)
    voxels, coors, num = O.merge_batch(vl, cl, nl)
    vx = O.simple_voxel(voxels, num)
    ref_f, ref_c, ref_shape = O.vxnet_forward(sd, vx, coors, [40, 1600, 1408])
    x = spconv.SparseConvTensor(vx.to(dev), torch.from_numpy(coors).to(dev), [40, 1600, 1408], 2)
    out, middle = model.neck.backbone(x)
    out.check_status()
    assert out.spatial_shape == ref_shape
    assert np.array_equal(out.indices.cpu().numpy(), ref_c)
    got = out.features.cpu().numpy()
    assert float(ref_f.abs().max()) < 10.0          # calibrated synthetic weights keep every frame O(1)
    # 14 layers of fp32 accumulation in a different order
    np.testing.assert_allclose(got, ref_f.numpy(), rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------ a9 BEVNet, a10 heads
def test_bevnet_golden(dev, golden_dir):
    from sassd_b200.necks import BEVNet
    m = np.load(os.path.join(golden_dir, "modules.npz"))
    net = BEVNet(in_features=20, num_filters=16).to(dev).eval()
    net.load_state_dict({k: v for k, v in _sd_from(m, "bev_sd/").items()}, strict=False)
    x, c6 = net(torch.from_numpy(m["bev_in"]).to(dev))
    np.testing.assert_allclose(x.cpu().numpy(), m["bev_x"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(c6.cpu().numpy(), m["bev_conv6"], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("ncls", [1, 3])
def test_rpn_head_decode_guided_golden(dev, golden_dir, ncls):
    from sassd_b200.single_stage_heads import SSDRotateHead
    m = np.load(os.path.join(golden_dir, "modules.npz"))
    p = "head%d_" % ncls
    head = SSDRotateHead(num_class=ncls, num_output_filters=16, num_anchor_per_loc=2).to(dev).eval()
    head.load_state_dict(_sd_from(m, p + "sd/"))
    box, cls, dirp = head(torch.from_numpy(m[p + "x"]).to(dev))
    np.testing.assert_allclose(box.cpu().numpy(), m[p + "box"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(dirp.cpu().numpy(), m[p + "dir"], rtol=1e-5, atol=1e-5)
    # guided anchors from the golden logits (the fixture rescales cls, so feed its tensors)
    ga, gl = head.get_guided_anchors(torch.from_numpy(m[p + "box"]).to(dev), torch.from_numpy(m[p + "cls"]).to(dev),
                                     torch.from_numpy(m[p + "dir"]).to(dev), torch.from_numpy(m[p + "anchors"]).to(dev),
                                     torch.from_numpy(m[p + "amask"]).to(dev), None, None, thr=.1)
    assert m[p + "anchors"].ndim == 3          # [B, Na, 7]: the reference decodes every frame with its own anchors
    for b in range(2):
        assert ga[b].shape == m[p + "ga%d" % b].shape
        np.testing.assert_allclose(ga[b].cpu().numpy(), m[p + "ga%d" % b], rtol=1e-5, atol=1e-5)
        assert np.array_equal(gl[b].cpu().numpy(), m[p + "gl%d" % b])


def test_pswarp_golden(dev, golden_dir):
    from sassd_b200.single_stage_heads import PSWarpHead
    from tests.golden_replay import pswarp_feature_and_boxes
    m = np.load(os.path.join(golden_dir, "modules.npz"))
    ps = PSWarpHead(grid_offsets=(0., 40.), featmap_stride=.4, in_channels=16, num_class=1, num_parts=28).to(dev).eval()
    ps.load_state_dict(_sd_from(m, "ps_sd/"), strict=False)
    feat, boxes = pswarp_feature_and_boxes()
    sc = ps(feat.to(dev), [b.to(dev) for b in boxes], is_test=True)
    for b in range(2):
        np.testing.assert_allclose(sc[b].cpu().numpy(), m["ps_scores%d" % b], rtol=1e-4, atol=2e-5)


# ------------------------------------------------------------------ a17 NMS
def _random_boxes(n, seed, spread=20.0):
    rs = np.random.RandomState(seed)
    x = rs.uniform(0, spread, n); y = rs.uniform(-spread / 2, spread / 2, n)
    w = rs.normal(1.6, 0.1, n); l = rs.normal(3.9, 0.3, n)
    r = rs.uniform(-4, 4, n)
    b7 = np.stack([x, y, np.full(n, -1.0), w, l, np.full(n, 1.5), r], 1).astype(np.float32)
    s = rs.uniform(0.3, 1.0, n).astype(np.float32)
    return b7, s


NMS_CASES = [(1, 0), (2, 1), (63, 2), (64, 3), (65, 4), (300, 5), (1500, 6)]
NMS_THR = 0.1


def nms_case(n, seed):
    """Scores and BEV boxes [n, 5] of one NMS case, and the boxes sorted by descending score (the kernels' input)."""
    from sassd_b200.single_stage_heads import boxes3d_to_bev_torch
    b7, s = _random_boxes(n, seed)
    bev = boxes3d_to_bev_torch(torch.from_numpy(b7))
    order = torch.sort(torch.from_numpy(s), descending=True, stable=True)[1]
    return s, bev, bev[order].contiguous()


@pytest.mark.parametrize("n,seed", NMS_CASES)
def test_nms_mask_and_keep(dev, golden_dir, n, seed):
    """Keep mask vs the CPU oracle; suppression bitmask bit for bit vs the one the UNMODIFIED reference CUDA kernel
    computed on the same boxes (tests/golden/nms.npz, made by tests/golden/make_golden_nms.py)."""
    from sassd_b200 import ops
    from sassd_b200.single_stage_heads import nms_gpu
    s, bev, sorted_bev = nms_case(n, seed)
    thr = NMS_THR
    mask = ops.nms_mask(sorted_bev.to(dev), thr).cpu().numpy().view(np.uint64)
    colb = (n + 63) // 64
    upper = np.zeros((n, colb), bool)
    for i in range(n):
        upper[i, i // 64:] = True
    g = np.load(os.path.join(golden_dir, "nms.npz"))
    key = "n%d_seed%d" % (n, seed)
    assert np.array_equal(sorted_bev.numpy(), g[key + "_bev"]), "the boxes differ from those the reference kernel saw"
    rm = g[key + "_mask"]
    assert rm.shape == mask.shape
    assert np.array_equal(mask[upper], rm[upper]), "suppression bitmask differs from the reference kernel"
    keep = nms_gpu(bev.to(dev), torch.from_numpy(s).to(dev), thr).cpu().numpy()
    okeep = O.nms_rotated(bev, torch.from_numpy(s), thr).numpy()
    iou = O.iou_matrix(sorted_bev.numpy())
    margin = np.abs(iou[np.triu_indices(n, 1)] - thr).min() if n > 1 else 1.0
    if margin > 1e-5:   # CPU libm / no-FMA oracle is only decisive away from the threshold
        assert np.array_equal(keep, okeep), "keep differs (min |IoU-thr| = %g)" % margin
    else:
        assert len(set(keep.tolist()) ^ set(okeep.tolist())) <= 2
    # IoU values agree with the oracle to fp32 round-off
    got = ops.boxes_iou_bev(sorted_bev.to(dev), sorted_bev.to(dev)).cpu().numpy()
    np.testing.assert_allclose(got, iou, rtol=0, atol=2e-5)


def test_rescore_nms_lists(dev):
    """get_rescore_bboxes (ssd_rotate_head.py:487-533) on lists, incl. empty / all-below-threshold frames."""
    import sassd_b200 as S
    from sassd_b200.single_stage_heads import PSWarpHead
    ps = PSWarpHead(grid_offsets=(0., 40.), featmap_stride=.4, in_channels=16, num_class=1, num_parts=28).to(dev)
    cfg = S.config.ConfigDict(score_thr=0.3, nms=dict(type="nms", iou_thr=0.1), max_per_img=100)
    frames = []
    for n, seed in ((200, 11), (0, 12), (50, 13), (700, 14)):
        b7, s = _random_boxes(max(n, 1), seed)
        logit = np.log(s / (1 - s)).astype(np.float32) - (2.0 if seed == 13 else 0.0)
        frames.append((torch.from_numpy(b7[:n]), torch.from_numpy(logit[:n]), torch.zeros(n, dtype=torch.int64)))
    got = ps.get_rescore_bboxes([f[0].to(dev) for f in frames], [f[1].to(dev) for f in frames],
                                [f[2].to(dev) for f in frames], [None] * len(frames), cfg)
    exp = O.get_rescore_bboxes([f[0] for f in frames], [f[1] for f in frames], [f[2] for f in frames], 0.3, 0.1)
    for b in range(len(frames)):
        if exp[0][b] is None:
            assert got[0][b] is None
            continue
        assert got[0][b].shape == exp[0][b].shape
        np.testing.assert_allclose(got[0][b], exp[0][b], rtol=0, atol=1e-6)
        np.testing.assert_allclose(got[1][b], exp[1][b], rtol=1e-6, atol=1e-6)
        assert np.array_equal(got[2][b], exp[2][b])


# ------------------------------------------------------------------ whole path
def _nhwc(t):
    """aux maps are fp32 NHWC tensors or ops.SplitMap (TMA tensor-core path)."""
    return t.float() if hasattr(t, "planes") else t


# Tolerances of the fp32 stages (north-star: "bbox regressions and class scores within 1e-4 fp32"):
#   * head outputs - box regressions (the 7 codes), class logits -> class scores, direction logits: 1e-4 absolute
#     (+ 1e-4 relative for the few codes above 1);
#   * activation maps (not a north-star quantity): |diff| <= 2e-4 + 1e-4 |x| - two fp32 evaluation orders of a
#     2304-term sum through 21 layers already differ by 1.2e-4 on the worst of nine million activations (measured: the
#     fp32 FFMA kernel vs the CPU oracle);
#   * decoded boxes = code * anchor diagonal (4.2 m) + anchor, exp(code) * size: 1e-3 absolute + 5e-4 relative (chain
#     tolerance: d exp(c) = exp(c) dc - a size code of 3 within 4e-4 is a 4e-4 relative change of a 78 m box; the decode
#     kernel itself is held to 1e-5 against the reference's decode on the golden logits);
#   * PSWarp on IDENTICAL inputs (our conv6 map and our guided boxes through the oracle's PSWarp head): class score
#     sigmoid(logit) 1e-4.  End to end the PSWarp logit also inherits the decoded boxes' ~1e-4 m differences: the
#     28-channel map of an untrained head is spatially rough (neighbouring pixels nearly independent), so a 1e-3 pixel
#     shift of the 28 sampling points moves the logit by ~1e-3 - the chain PSWarp score and the final detection score are
#     therefore held to 1e-3 end to end, the RPN class scores and box regressions to 1e-4.
# Discrete decisions (score > 0.1, score > 0.3, IoU > 0.1, sort order) can only be compared away from their thresholds:
# every stage is therefore ALSO checked bit-exactly on identical inputs (our guided boxes and scores through the
# oracle's rescoring + NMS must give our detections), and end to end the lists are matched as sets.
HEAD_ATOL, MAP_TOL, BOX_ATOL, PS_CHAIN_ATOL = 1e-4, 2e-4, 1e-3, 1e-3


def _match_detections(gb, gs, eb, es, tag):
    """Match two detection lists by box centre (NMS keeps centres apart); returns the number of matched pairs after
    checking their scores and boxes, and the numbers of unmatched detections on either side."""
    if eb is None or gb is None:
        return 0, 0 if gb is None else len(gb), 0 if eb is None else len(eb)
    d = np.abs(gb[:, None, :2] - eb[None, :, :2]).max(-1)          # [G, E]
    j = d.argmin(1)
    ok = d[np.arange(len(gb)), j] < 2e-3
    pairs = [(i, j[i]) for i in range(len(gb)) if ok[i]]
    assert len({e for _, e in pairs}) == len(pairs), tag
    for i, e in pairs:
        assert abs(gs[i] - es[e]) <= PS_CHAIN_ATOL, "%s: score %g vs %g" % (tag, gs[i], es[e])   # see the notes above
        np.testing.assert_allclose(gb[i], eb[e], rtol=5e-4, atol=BOX_ATOL, err_msg=tag)
    return len(pairs), len(gb) - len(pairs), len(eb) - len(pairs)


def _compare_frame(got, exp, tag):
    """End-to-end detection lists of one frame: matched as sets; a detection may be missing on one side only because
    a threshold decision upstream flipped within round-off, which is rare - at most 1 in 10 (at least 1)."""
    if exp[0] is None and got["boxes_lidar"] is None:
        return 0
    n, ug, ue = _match_detections(got["boxes_lidar"], got["scores"], exp[0], exp[1], tag)
    ne = 0 if exp[0] is None else len(exp[0])
    assert ug + ue <= max(1, ne // 10), "%s: %d matched, %d only ours, %d only oracle" % (tag, n, ug, ue)
    return n


def _expected_anchor_scores(st, b, num_class):
    """max_c sigmoid(cls) of every anchor of frame b in anchor order (class, y, x, rot) - fp32 like the reference."""
    cls = st["cls"][b]                                            # [ncls, H, W, 2*ncls]
    nc, H, W, _ = cls.shape
    s = torch.sigmoid(cls.reshape(nc, H, W, 2, num_class)).max(-1)[0]
    return s.reshape(-1).numpy()


def _check_against_oracle(model, sd, clouds, tag, cfg=ORACLE_CFG, num_class=1, min_total=1, map_tol=MAP_TOL):
    """raw points -> detections through forward_points vs the CPU oracle, stage by stage (see the tolerance notes
    above).  Integer stages bit-exact.  Returns the number of end-to-end detections compared."""
    B = len(clouds)
    out, aux = model.forward_points(clouds, return_aux=True)
    st = {}
    exp = O.forward_test(sd, clouds, cfg, num_class=num_class, stages=st)
    fr = aux["frame_rows"].cpu().numpy()
    for b in range(B):
        assert np.array_equal(aux["coors"][fr[b]:fr[b + 1], 1:].cpu().numpy(), st["coors"][b]), tag
        assert np.array_equal(aux["mask"][b].bool().cpu().numpy(), st["anchors_mask"][b]), tag
    assert np.array_equal(aux["sparse"].indices.cpu().numpy(), st["coors3"]), tag
    x = _nhwc(aux["x"]).permute(0, 3, 1, 2).cpu().numpy()
    head = aux["head"].cpu().numpy()                              # [B, H, W, box | cls | dir]
    na = 2 * num_class
    ks = aux["d_k"].cpu().numpy()
    total = 0
    for b in range(B):
        assert float(st["x"][b].abs().max()) < 10.0               # calibrated synthetic weights: all frames O(1)
        np.testing.assert_allclose(x[b], st["x"][b].numpy(), rtol=1e-4, atol=map_tol, err_msg="%s frame %d neck" % (tag, b))
        # --- the north-star's fp32 quantities: box regressions, class scores (logits too), direction logits
        hb = head[b]
        ebox = st["box"][b].permute(1, 2, 0, 3).reshape(hb.shape[0], hb.shape[1], -1).numpy()
        ecls = st["cls"][b].permute(1, 2, 0, 3).reshape(hb.shape[0], hb.shape[1], -1).numpy()
        edir = st["dir"][b].permute(1, 2, 0, 3).reshape(hb.shape[0], hb.shape[1], -1).numpy()
        o1, o2 = na * 7, na * 7 + na * num_class
        np.testing.assert_allclose(hb[..., :o1], ebox, rtol=1e-4, atol=HEAD_ATOL, err_msg="%s frame %d box codes" % (tag, b))
        np.testing.assert_allclose(hb[..., o2:o2 + na * 2], edir, rtol=1e-4, atol=HEAD_ATOL, err_msg="%s dir" % tag)
        sig = lambda v: 1.0 / (1.0 + np.exp(-v.astype(np.float64)))
        np.testing.assert_allclose(sig(hb[..., o1:o2]), sig(ecls), rtol=0, atol=HEAD_ATOL, err_msg="%s frame %d class scores" % (tag, b))
        # --- guided anchors: same selection except anchors whose score is within round-off of the 0.1 threshold
        gi = aux["guided_index"][b, :ks[b]].cpu().numpy()
        ei = st["guided_index"][b].numpy()
        escore = _expected_anchor_scores(st, b, num_class)
        flipped = np.setxor1d(gi, ei)
        assert np.all(np.abs(escore[flipped] - 0.1) <= 1e-4), "%s frame %d guided selection" % (tag, b)
        assert np.all(np.diff(gi) > 0)                             # order preserved
        common, ig, ie = np.intersect1d(gi, ei, return_indices=True)
        if num_class > 1:
            assert np.array_equal(aux["guided_labels"][b, :ks[b]].cpu().numpy()[ig], st["labels"][b].numpy()[ie])
        np.testing.assert_allclose(aux["guided"][b, :ks[b]].cpu().numpy()[ig], st["guided"][b].numpy()[ie], rtol=5e-4,
                                   atol=BOX_ATOL, err_msg="%s frame %d decoded boxes" % (tag, b))
        got_ps = aux["ps_scores"][b, :ks[b]].cpu().numpy().astype(np.float64)
        exp_ps = st["ps_scores"][b].numpy().astype(np.float64)[ie]
        np.testing.assert_allclose(sig(got_ps[ig]), sig(exp_ps), rtol=0, atol=PS_CHAIN_ATOL, err_msg="%s PSWarp scores (chain)" % tag)
        # the PSWarp head on identical inputs: our conv6 map and our guided boxes through the oracle's convs + sampling
        if ks[b]:
            c6 = _nhwc(aux["conv6"])[b:b + 1].permute(0, 3, 1, 2).cpu().float()
            same_ps = O.pswarp_forward(sd, c6, [aux["guided"][b, :ks[b]].cpu()], cfg["grid_offsets"], cfg["featmap_stride"])[0]
            np.testing.assert_allclose(sig(got_ps), sig(same_ps.numpy().astype(np.float64)), rtol=0, atol=1e-4,
                                       err_msg="%s frame %d PSWarp scores on identical inputs" % (tag, b))
        # --- rescoring + NMS on identical inputs: OUR guided boxes / logits / labels through the oracle = our detections
        same = O.get_rescore_bboxes([aux["guided"][b, :ks[b]].cpu()], [aux["ps_scores"][b, :ks[b]].cpu()],
                                    [aux["guided_labels"][b, :ks[b]].cpu().long()], cfg["score_thr"], cfg["iou_thr"])
        if same[0][0] is None:
            assert out[b]["boxes_lidar"] is None
        else:
            sg = sig(aux["ps_scores"][b, :ks[b]].cpu().numpy())
            tie = len(sg) > 1 and np.abs(sg - 0.3).min() > 1e-6
            if tie:      # decisive thresholds: the kept set, its order, scores and labels are bit-identical
                np.testing.assert_array_equal(out[b]["boxes_lidar"], same[0][0], err_msg="%s frame %d NMS on equal inputs" % (tag, b))
                np.testing.assert_array_equal(out[b]["label_preds"], same[2][0])
                np.testing.assert_allclose(out[b]["scores"], same[1][0], rtol=0, atol=1e-6)
        # --- end to end
        total += _compare_frame(out[b], (exp[0][b], exp[1][b], exp[2][b]), "%s frame %d" % (tag, b))
    assert total >= min_total, "%s: only %d detections compared" % (tag, total)
    return total


@pytest.mark.parametrize("seeds", [(0, 9), (1, 7)])
def test_end_to_end_points_to_detections(dev, car_model, seeds):
    """raw points -> detections through forward_points vs the CPU oracle, 2 frames, car_cfg, both precisions."""
    model, sd = car_model
    _check_against_oracle(model, sd, [synth_cloud(s) for s in seeds], "seeds %s" % (seeds,), min_total=10)


def test_end_to_end_batch16(dev):
    """BASELINE configs[2]: one batch of 16 frames (seeds 0..15) on the default tensor-core path vs the oracle."""
    model, sd = _make_model(dev)
    _check_against_oracle(model, sd, [synth_cloud(s) for s in range(16)], "batch16", min_total=100)


def test_reference_signature_forward_test(dev, car_model):
    """detector(return_loss=False, **data) with dataset-side inputs (tools/test.py:31, kitti.py:296-352)."""
    model, sd = car_model
    clouds = [synth_cloud(9)]
    vl, cl, nl, ml = [], [], [], []
    for p in clouds:
        v, c, n = model.voxel_generator.generate(p)
        vl.append(torch.from_numpy(v)); cl.append(torch.from_numpy(c)); nl.append(torch.from_numpy(n))
        ml.append(torch.from_numpy(model.anchor_set.mask(c)))
    anchors = [torch.from_numpy(model.anchor_set.anchors)] * len(clouds)
    res = model(img=None, img_meta=[dict(sample_idx=0)], return_loss=False, voxels=vl, coordinates=cl, num_points=nl,
                anchors=anchors, anchors_mask=ml, gt_labels=[None], gt_bboxes=[None], gt_types=[None])
    exp = O.forward_test(sd, clouds, ORACLE_CFG)
    _compare_frame(res[0], (exp[0][0], exp[1][0], exp[2][0]), "forward_test")
    fused = model.forward_points(clouds)
    # same detections from the fused raw-points path (its heads read TMA split maps, the reference-signature path
    # fp32 NHWC tensors: different kernels, a few ulp apart)
    assert fused[0]["boxes_lidar"].shape == res[0]["boxes_lidar"].shape
    np.testing.assert_allclose(fused[0]["boxes_lidar"], res[0]["boxes_lidar"], rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------ the other tensor-core split (3xTF32)
def test_end_to_end_tf32x3_path(dev):
    """The same raw-points -> detections comparison on the 3xTF32 tcgen05 kernels (selectable, not the default)."""
    model, sd = _make_model(dev, prec="tf32x3")
    # the TF32 split keeps 21 significand bits per operand (fp16 split: 22): activation maps at 4e-4
    _check_against_oracle(model, sd, [synth_cloud(0), synth_cloud(9)], "tf32x3", min_total=10, map_tol=4e-4)


@pytest.mark.parametrize("prec", PRECS)
def test_cuda_graph_replay_matches_eager(dev, prec):
    """The captured step must give the same detections as the eager launch sequence, also after the
    frame changes between replays (all sizes are device-side)."""
    model, sd = _make_model(dev, prec=prec)
    frames = [[synth_cloud(9)], [synth_cloud(0)], [synth_cloud(9)]]
    eager = [model.forward_points(f) for f in frames]
    model.enable_cuda_graph(1, 32768)
    for f, e in zip(frames, eager):
        g = model.forward_points(f)
        assert (g[0]["boxes_lidar"] is None) == (e[0]["boxes_lidar"] is None)
        if e[0]["boxes_lidar"] is not None:
            np.testing.assert_array_equal(g[0]["boxes_lidar"], e[0]["boxes_lidar"])
            np.testing.assert_array_equal(g[0]["scores"], e[0]["scores"])
    # a frame that does not fit the captured shape falls back to the eager path
    big = model.forward_points([synth_cloud(3, fov_deg=60.0)])
    assert isinstance(big, list) and len(big) == 1
    model.disable_cuda_graph()


def test_graph_is_recaptured_after_a_weight_reload(dev):
    """A captured step bakes in packed-weight addresses: loading new parameters must drop it (ADVICE r1)."""
    from sassd_b200 import checkpoint
    model, sd = _make_model(dev)
    frame = [synth_cloud(9)]
    model.enable_cuda_graph(1, 32768)
    a = model.forward_points(frame)
    sd2 = {k: (v * 1.25 if k.endswith("conv_cls.weight") else v) for k, v in sd.items()}
    checkpoint.load_state_dict_into(model, sd2)
    assert model._graph is None
    b = model.forward_points(frame)                     # re-captured with the new weights
    assert model._graph is not None
    model.disable_cuda_graph()
    c = model.forward_points(frame)                     # eager, new weights
    np.testing.assert_array_equal(b[0]["scores"], c[0]["scores"])
    assert a[0]["scores"].shape != b[0]["scores"].shape or not np.array_equal(a[0]["scores"], b[0]["scores"])
    # detect_stream slots are dropped the same way
    list(model.detect_stream([frame, frame], 1, 32768, depth=2))
    assert model._stream_slots is not None
    checkpoint.load_state_dict_into(model, sd)
    assert model._stream_slots is None
    d = list(model.detect_stream([frame], 1, 32768, depth=2))[0]
    np.testing.assert_array_equal(d[0]["scores"], a[0]["scores"])


@pytest.mark.parametrize("prec", PRECS)
def test_detect_stream_matches_forward_points(dev, prec):
    model, sd = _make_model(dev, prec=prec)
    frames = [[synth_cloud(s)] for s in (9, 0, 6, 9, 0)]
    ref = [model.forward_points(f) for f in frames]
    got = list(model.detect_stream(frames, 1, 32768))
    assert len(got) == len(ref)
    for g, e in zip(got, ref):
        assert (g[0]["boxes_lidar"] is None) == (e[0]["boxes_lidar"] is None)
        if e[0]["boxes_lidar"] is not None:
            np.testing.assert_array_equal(g[0]["boxes_lidar"], e[0]["boxes_lidar"])
            np.testing.assert_array_equal(g[0]["scores"], e[0]["scores"])
            np.testing.assert_array_equal(g[0]["label_preds"], e[0]["label_preds"])


@pytest.mark.parametrize("prec", PRECS)
def test_multi_class_config_end_to_end(dev, prec):
    """configs/multi_cfg.py (Car / Pedestrian / Cyclist, 211 200 anchors): labels, scores and boxes vs the oracle."""
    model, sd = _make_model(dev, num_class=3, cfg_name="multi_cfg.py", prec=prec)
    cfg3 = dict(ORACLE_CFG, anchor_cfgs=[CAR, PED, CYC])
    clouds = [synth_cloud(0), synth_cloud(9)]
    out, aux = model.forward_points(clouds, return_aux=True)
    assert aux["mask"].shape[1] == 211200
    _check_against_oracle(model, sd, clouds, "multi_cfg", cfg=cfg3, num_class=3, min_total=50)


def test_density_sweep_endpoints(dev, car_model):
    """BASELINE config 5 endpoints in one batch: a ~5 k-point and a ~120 k-point cloud (the latter hits the
    20 000-voxel cut) - integer stages bit-exact, same detections as the oracle, both precisions."""
    model, sd = car_model
    clouds = [synth_cloud(11, fov_deg=28.0, az_step_deg=0.6912), synth_cloud(12, fov_deg=180.0)]
    assert clouds[0].shape[0] < 6000 and clouds[1].shape[0] > 100000
    out, aux = model.forward_points(clouds, return_aux=True)
    fr = aux["frame_rows"].cpu().numpy()
    assert fr[2] - fr[1] == 20000
    _check_against_oracle(model, sd, clouds, "density sweep", min_total=10)


def _scattered_map(dev, B, H, W, C, D, seed):
    from sassd_b200 import ops
    torch.manual_seed(seed)
    n = 40
    coors = torch.zeros((n, 4), dtype=torch.int32, device=dev)
    coors[:, 0] = torch.randint(0, max(B - 1, 1), (n,), device=dev)      # the last frame stays empty
    coors[:, 1] = torch.randint(0, D, (n,), device=dev)
    coors[:, 2] = torch.randint(0, 12, (n,), device=dev)                 # active cells clustered in a corner ...
    coors[:, 3] = torch.randint(0, 20, (n,), device=dev)
    coors[n - 1, 2], coors[n - 1, 3] = H - 1, W - 1                      # ... plus one in the far corner
    key = ((coors[:, 0].long() * D + coors[:, 1].long()) * H + coors[:, 2].long()) * W + coors[:, 3].long()
    keep = torch.from_numpy(np.unique(key.cpu().numpy(), return_index=True)[1]).to(dev)
    rows = coors[keep].contiguous()
    cap = torch.zeros((64, 4), dtype=torch.int32, device=dev)
    cap[: rows.shape[0]] = rows
    feat = torch.randn(64, C, device=dev)
    d_rows = torch.tensor([rows.shape[0]], dtype=torch.int32, device=dev)
    return ops.sparse_to_bev_split(feat, cap, d_rows, C, D, H, W, B)


@pytest.mark.gpu
@pytest.mark.parametrize("out", ["split", "f32", "both"])
@pytest.mark.parametrize("B,H,W,taps,cout", [(3, 40, 52, 9, 256), (3, 40, 52, 9, 28), (3, 40, 52, 1, 256),
                                             (4, 200, 176, 9, 256)])
def test_constant_tiles_single_layer_bit_identical(dev, B, H, W, taps, cout, out):
    """A scattered (mostly zero) BEV map carries per-tile distances to its active cells; tiles out of the layer's
    reach skip loads and MMAs and store the layer's constant.  Must equal the all-tiles computation bit for bit,
    including a frame with no active cell, in each output mode (split-only constant tiles take their own store path),
    and on a map of more than 832 tiles (1100 at B = 4, 200x176), where the kernel decides per tile instead of from
    its verdict table."""
    from sassd_b200 import ops
    C, D = 64, 2
    x = _scattered_map(dev, B, H, W, C, D, taps * 100 + cout)
    far = (x.tile_dist > 9).sum().item()
    assert x.tile_dist is not None and 0 < far < x.tile_dist.numel()
    w = torch.randn(taps, D * C, cout, device=dev) * 0.1
    scale = torch.rand(cout, device=dev) + 0.5
    shift = torch.randn(cout, device=dev) * 0.3
    sp, fo = out != "f32", out != "split"
    sp_occ, f_occ = ops.conv2d_split(x, w, scale, shift, True, cout, out_split=sp, out_f32=fo)
    full = ops.SplitMap(x.planes, x.channels)                        # same map without the tile information
    sp_all, f_all = ops.conv2d_split(full, w, scale, shift, True, cout, out_split=sp, out_f32=fo)
    torch.cuda.synchronize()
    if fo:
        assert torch.equal(f_occ[..., :cout], f_all[..., :cout])
        assert torch.equal(f_occ[B - 1, H // 2, W // 2, :cout], torch.relu(shift))      # empty frame: act(shift)
    if sp:
        assert torch.equal(sp_occ.planes, sp_all.planes)
        exp = ops.SplitMap.from_float(torch.relu(shift).view(1, 1, 1, cout)).planes[:, 0, 0, 0, :cout]
        assert torch.equal(sp_occ.planes[:, B - 1, H // 2, W // 2, :cout], exp)


@pytest.mark.gpu
def test_constant_tiles_through_a_layer_chain_bit_identical(dev):
    """3x3 -> 3x3 -> 3x3 -> 1x1 -> 3x3 (small head): constants, reach and the border rule (zero padding differs from
    the constant) must reproduce the plain computation exactly at every layer."""
    from sassd_b200 import ops
    B, H, W, C, D = 2, 56, 80, 64, 1
    torch.manual_seed(5)
    layers = [(9, 64, 64), (9, 64, 64), (9, 64, 64), (1, 64, 64), (9, 64, 28)]
    params = [(torch.randn(t, ci, co, device=dev) * (0.3 / (t * ci) ** 0.5 * 4), torch.rand(co, device=dev) + 0.5,
               torch.randn(co, device=dev) * 0.3) for t, ci, co in layers]

    def run(use_tiles):
        ops.TILE_OCCUPANCY = use_tiles
        try:
            x = _scattered_map(dev, B, H, W, C, D, 77)
            outs = []
            for (t, ci, co), (w, sc, sh) in zip(layers, params):
                x, f = ops.conv2d_split(x, w, sc, sh, True, co, out_split=True, out_f32=True)
                outs.append((x.planes.clone(), f.clone(), x.reach))
            torch.cuda.synchronize()
            return outs
        finally:
            ops.TILE_OCCUPANCY = True
    with_tiles, plain = run(True), run(False)
    assert [o[2] for o in with_tiles] == [1, 2, 3, 3, 4]
    for i, (a, b) in enumerate(zip(with_tiles, plain)):
        assert torch.equal(a[0], b[0]), "split planes differ at layer %d" % i
        assert torch.equal(a[1], b[1]), "fp32 map differs at layer %d" % i


@pytest.mark.gpu
def test_constant_tile_skipping_leaves_detections_unchanged(dev):
    """Whole pipeline with and without the constant-region tile skipping: identical detections, bit for bit."""
    from sassd_b200 import ops
    model, sd = _make_model(dev)              # default precision: TMA dense convs on split maps
    frames = [[synth_cloud(s)] for s in (0, 9, 3)] + [[synth_cloud(1), synth_cloud(7)]]
    res = {}
    for flag in (True, False):
        ops.TILE_OCCUPANCY = flag
        try:
            res[flag] = [model.forward_points(f) for f in frames]
            _, aux = model.forward_points(frames[0], return_aux=True)
            # the path under test really is the one that skips: split maps, tile distances only with the flag on
            assert isinstance(aux["x"], ops.SplitMap) and (aux["x"].tile_dist is not None) == flag
            if flag:
                assert aux["x"].reach == 7 and int((aux["x"].tile_dist > 7).sum().item()) > 0
        finally:
            ops.TILE_OCCUPANCY = True
    ndet = 0
    for a, b in zip(res[True], res[False]):
        for fa, fb in zip(a, b):
            assert (fa["boxes_lidar"] is None) == (fb["boxes_lidar"] is None)
            if fa["boxes_lidar"] is not None:
                np.testing.assert_array_equal(fa["boxes_lidar"], fb["boxes_lidar"])
                np.testing.assert_array_equal(fa["scores"], fb["scores"])
                ndet += len(fa["scores"])
    assert ndet > 0
