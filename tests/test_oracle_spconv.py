"""Pin the oracle's spconv-v1 restatement BY DEFINITION (the reference vendors no
spconv source and holds no tests for it): SubMConv3d / SparseConv3d values must
equal torch.nn.functional.conv3d on the densified input, sampled at the active
output sites (SURVEY.md §A.2)."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import ref_pipeline as O


def _random_sparse(B, shape, n, cin, seed):
    rs = np.random.RandomState(seed)
    cells = rs.choice(B * shape[0] * shape[1] * shape[2], size=n, replace=False)
    c = np.zeros((n, 4), np.int32)
    r = cells.copy()
    c[:, 3] = r % shape[2]; r //= shape[2]
    c[:, 2] = r % shape[1]; r //= shape[1]
    c[:, 1] = r % shape[0]; r //= shape[0]
    c[:, 0] = r
    f = torch.from_numpy(rs.randn(n, cin).astype(np.float32))
    return c, f


def _densify(c, f, B, shape):
    d = torch.zeros(B, f.shape[1], *shape)
    ci = torch.from_numpy(c.astype(np.int64))
    d[ci[:, 0], :, ci[:, 1], ci[:, 2], ci[:, 3]] = f
    return d


def test_subm_equals_dense_conv3d():
    B, shape, cin, cout = 2, [6, 9, 8], 5, 7
    c, f = _random_sparse(B, shape, 150, cin, 0)
    w = torch.randn(3, 3, 3, cin, cout)
    nbr = O.subm_rulebook(c, shape)
    out = O.indice_conv(f, w.reshape(27, cin, cout), nbr)
    dense = F.conv3d(_densify(c, f, B, shape), w.permute(4, 3, 0, 1, 2).contiguous(), padding=1)
    ci = torch.from_numpy(c.astype(np.int64))
    ref = dense[ci[:, 0], :, ci[:, 1], ci[:, 2], ci[:, 3]]
    np.testing.assert_allclose(out.numpy(), ref.numpy(), rtol=1e-5, atol=1e-5)
    # centre offset always maps a site to itself
    assert np.array_equal(nbr[:, 13], np.arange(c.shape[0]))


def test_strided_equals_dense_conv3d_and_output_set():
    B, shape, cin, cout = 2, [6, 10, 8], 4, 6
    c, f = _random_sparse(B, shape, 120, cin, 1)
    w = torch.randn(3, 3, 3, cin, cout)
    oc, nbr, oshape = O.sparse_conv_rulebook(c, shape)
    assert oshape == [3, 5, 4]
    out = O.indice_conv(f, w.reshape(27, cin, cout), nbr)
    dense = F.conv3d(_densify(c, f, B, shape), w.permute(4, 3, 0, 1, 2).contiguous(), stride=2, padding=1)
    oi = torch.from_numpy(oc.astype(np.int64))
    ref = dense[oi[:, 0], :, oi[:, 1], oi[:, 2], oi[:, 3]]
    np.testing.assert_allclose(out.numpy(), ref.numpy(), rtol=1e-5, atol=1e-5)
    # active output set == cells whose receptive field touches an active input
    occ = F.conv3d(_densify(c, torch.ones(c.shape[0], 1), B, shape), torch.ones(1, 1, 3, 3, 3), stride=2, padding=1)
    want = torch.nonzero(occ[:, 0] > 0)
    assert np.array_equal(want.numpy(), oc.astype(np.int64))  # nonzero() is sorted == canonical order
    # everything outside the active set is exactly zero in the dense result only if no input touches it
    keys = O._flat(oc, oshape)
    assert np.all(np.diff(keys) > 0)


def test_dense_bev_channel_interleave():
    B, shape = 2, [5, 4, 3]
    c, f = _random_sparse(B, shape, 30, 6, 2)
    bev = O.dense_bev(f, c, shape, B)
    assert bev.shape == (2, 30, 4, 3)
    for i in range(c.shape[0]):
        b, z, y, x = c[i]
        for ch in range(6):
            assert bev[b, ch * 5 + z, y, x] == f[i, ch]
    assert int((bev != 0).sum()) == int((f != 0).sum())


def test_indice_pairs_canonical_form():
    B, shape = 1, [4, 6, 5]
    c, f = _random_sparse(B, shape, 40, 3, 3)
    nbr = O.subm_rulebook(c, shape)
    pairs, num = O.nbr_to_indice_pairs(nbr)
    assert pairs.shape == (2, 27, 40) and num.sum() == (nbr >= 0).sum()
    # symmetry of a submanifold rulebook: (i, o, k) <-> (o, i, 26-k)
    for k in range(27):
        fw = set(zip(pairs[0, k, :num[k]].tolist(), pairs[1, k, :num[k]].tolist()))
        bw = set(zip(pairs[1, 26 - k, :num[26 - k]].tolist(), pairs[0, 26 - k, :num[26 - k]].tolist()))
        assert fw == bw


def test_vxnet_tiny_end_to_end_vs_dense():
    """Whole VxNet on a tiny grid vs a dense conv3d network with active-site masking.  The dense emulation runs in
    float64: in fp32 its own summation order, which depends on the host's CPU kernels and thread count, uses up to
    1.2x of the tolerance on these 14 layers, so the tolerance is left to the fp32 oracle alone."""
    from sassd_b200.checkpoint import make_synthetic_state_dict
    sd = make_synthetic_state_dict(seed=3, num_class=1)
    B, shape = 1, [8, 16, 16]
    c, f = _random_sparse(B, shape, 200, 4, 4)
    feats, c3, shape3 = O.vxnet_forward(sd, f, c, shape)
    assert shape3 == [1, 2, 2] and feats.shape[1] == 64
    # dense emulation
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    x = _densify(c, f, B, shape).double()
    act = _densify(c, torch.ones(c.shape[0], 1), B, shape) > 0
    p = "neck.backbone."

    def bnrelu(x, name):
        return torch.relu(O.bn_eval(x, sd64, p + name))
    for block, idxs, kind, key in O.VXNET_PLAN:
        for i in idxs:
            w = sd64["%s%s.%d.weight" % (p, block, i)].permute(4, 3, 0, 1, 2).contiguous()
            if kind == "down":
                x = F.conv3d(x, w, stride=2, padding=1)
                act = F.conv3d(act.float(), torch.ones(1, 1, 3, 3, 3), stride=2, padding=1) > 0
            else:
                x = F.conv3d(x, w, padding=1)
            x = bnrelu(x, "%s.%d" % (block, i + 1)) * act
    w = sd64[p + "extra_conv.0.weight"].permute(4, 3, 0, 1, 2).contiguous()
    x = bnrelu(F.conv3d(x, w), "extra_conv.1") * act
    ci = torch.from_numpy(c3.astype(np.int64))
    ref = x[ci[:, 0], :, ci[:, 1], ci[:, 2], ci[:, 3]]
    np.testing.assert_allclose(feats.numpy(), ref.numpy(), rtol=1e-4, atol=1e-5)
    assert int(act.sum()) == c3.shape[0]
