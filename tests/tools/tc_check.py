"""GPU dev tool: timings and traces of the tensor-core conv kernels at pipeline shapes (each timed case also prints
its error against fp64).  The kernel-level correctness checks live in tests/test_conv_kernels.py."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np, torch
from sassd_b200 import ops

dev = torch.device("cuda:0")
torch.manual_seed(0)


def run(mode, M, cin, cout, taps, relu, H=0, W=0, B=0, nbr=None, d_rows=None, tag="", pattern=None, time_it=False):
    x = torch.randn(M, cin, device=dev)
    w = torch.randn(taps, cin, cout, device=dev) * 0.1
    if pattern == "ones":
        x.fill_(1.0); w.fill_(0.0); w[:, :, :] = 0.0
        for n in range(cout):
            w[0, n % cin, n] = 1.0 + n
    scale = torch.rand(cout, device=dev) + 0.5
    shift = torch.randn(cout, device=dev) * 0.1
    stride = (cout + 3) // 4 * 4
    outs = []
    for prec in (ops.PREC_FP32, ops.PREC_TF32X3, ops.PREC_F16X3):
        out = torch.zeros(M, stride, device=dev)
        ops.gconv(x, w, scale, shift, out, mode=mode, taps=taps, cin=cin, cout=cout, relu=relu, nbr=nbr, d_rows=d_rows,
                  rows_cap=M, batch=B, H=H, W=W, precision=prec)
        torch.cuda.synchronize()
        outs.append(out[:, :cout].clone())
    # fp64 reference
    xd, wd = x.double().cpu(), w.double().cpu()
    ref = torch.zeros(M, cout, dtype=torch.float64)
    if mode == ops.GCONV_ROWS or (mode == ops.GCONV_CONV2D and taps == 1):
        ref = xd @ wd[0]
    elif mode == ops.GCONV_CONV2D:
        img = xd.view(B, H, W, cin).permute(0, 3, 1, 2)
        wk = wd.view(3, 3, cin, cout).permute(3, 2, 0, 1)
        ref = torch.nn.functional.conv2d(img, wk, padding=1).permute(0, 2, 3, 1).reshape(M, cout)
    else:
        nb = nbr.cpu().long()
        for t in range(taps):
            o = torch.nonzero(nb[:, t] >= 0).view(-1)
            ref.index_add_(0, o, xd[nb[o, t]] @ wd[t])
    ref = ref * scale.double().cpu() + shift.double().cpu()
    if relu:
        ref = ref.clamp_min(0)
    e32 = (outs[0].double().cpu() - ref).abs().max().item()
    etc = (outs[1].double().cpu() - ref).abs().max().item()
    e16 = (outs[2].double().cpu() - ref).abs().max().item()
    sc = ref.abs().max().item()
    bad16 = e16 > 20 * max(e32, 1e-6 * sc)
    print("%-34s M=%-6d cin=%-3d cout=%-3d taps=%-2d  |ref|max %.3g  err ffma %.2e  tf32x3 %.2e  f16x3 %.2e  %s" %
          (tag, M, cin, cout, taps, sc, e32, etc, e16,
           "OK" if etc <= 20 * max(e32, 1e-6 * sc) and not bad16 else "MISMATCH"), flush=True)
    if bad16:
        d = (outs[2].double().cpu() - ref)
        bad = torch.nonzero(d.abs() > 1e-3 * max(sc, 1)).cpu()
        print("   f16 first bad (row, col):", bad[:8].tolist(), " n_bad", bad.shape[0])
        print("   f16 row0[:8]", outs[2][0, :8].tolist())
        print("   ref row0[:8]", ref[0, :8].tolist())
    if etc > 20 * max(e32, 1e-6 * sc):
        d = (outs[1].double().cpu() - ref)
        bad = torch.nonzero(d.abs() > 1e-3 * max(sc, 1)).cpu()
        print("   first bad (row, col):", bad[:8].tolist(), " n_bad", bad.shape[0])
        print("   tc  row0[:8]", outs[1][0, :8].tolist())
        print("   ref row0[:8]", ref[0, :8].tolist())
    if time_it:
        for prec, name in ((ops.PREC_FP32, "ffma"), (ops.PREC_TF32X3, "tf32x3"), (ops.PREC_F16X3, "f16x3")):
            out = torch.zeros(M, stride, device=dev)
            for _ in range(2):
                ops.gconv(x, w, scale, shift, out, mode=mode, taps=taps, cin=cin, cout=cout, relu=relu, nbr=nbr,
                          d_rows=d_rows, rows_cap=M, batch=B, H=H, W=W, precision=prec)
            torch.cuda.synchronize()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                ops.gconv(x, w, scale, shift, out, mode=mode, taps=taps, cin=cin, cout=cout, relu=relu, nbr=nbr,
                          d_rows=d_rows, rows_cap=M, batch=B, H=H, W=W, precision=prec)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 5
            fl = 2.0 * M * cin * cout * taps
            print("   %-6s %.3f ms  %.1f TFLOP/s (algorithmic fp32)" % (name, ms, fl / ms / 1e9), flush=True)


stage = sys.argv[1] if len(sys.argv) > 1 else "all"
if stage in ("perf", "all"):
    run(ops.GCONV_CONV2D, 200 * 176, 256, 256, 9, True, H=200, W=176, B=1, tag="BEV 3x3 256->256 B=1", time_it=True)
    run(ops.GCONV_CONV2D, 4 * 200 * 176, 256, 256, 9, True, H=200, W=176, B=4, tag="BEV 3x3 256->256 B=4", time_it=True)


def run_tma(B, H, W, cin, cout, taps, relu, tag, time_it=False):
    x = torch.randn(B, H, W, cin, device=dev)
    w = torch.randn(taps, cin, cout, device=dev) * 0.05
    scale = torch.rand(cout, device=dev) + 0.5
    shift = torch.randn(cout, device=dev) * 0.1
    xs = ops.SplitMap.from_float(x)
    sp, f32 = ops.conv2d_split(xs, w, scale, shift, relu, cout, out_split=True, out_f32=True)
    torch.cuda.synchronize()
    img = x.double().cpu().permute(0, 3, 1, 2)
    k = 3 if taps == 9 else 1
    wk = w.double().cpu().view(k, k, cin, cout).permute(3, 2, 0, 1)
    ref = torch.nn.functional.conv2d(img, wk, padding=k // 2).permute(0, 2, 3, 1)
    ref = ref * scale.double().cpu() + shift.double().cpu()
    if relu:
        ref = ref.clamp_min(0)
    sc = ref.abs().max().item()
    e1 = (f32[..., :cout].double().cpu() - ref).abs().max().item()
    e2 = (sp.float().double().cpu() - ref).abs().max().item()
    ok = e1 < 2e-5 * max(sc, 1) and e2 < 2e-5 * max(sc, 1)
    print("%-30s B=%d %dx%d cin=%-3d cout=%-3d taps=%d |ref|max %.3g  err f32-out %.2e  err split-out %.2e  %s" %
          (tag, B, H, W, cin, cout, taps, sc, e1, e2, "OK" if ok else "MISMATCH"), flush=True)
    if not ok:
        d = (f32[..., :cout].double().cpu() - ref).abs()
        bad = torch.nonzero(d > 1e-3 * max(sc, 1))
        print("   n_bad", bad.shape[0], "first", bad[:6].tolist())
        print("   got", f32[0, 0, 0, :6].tolist(), "ref", ref[0, 0, 0, :6].tolist())
    if time_it:
        for _ in range(2):
            ops.conv2d_split(xs, w, scale, shift, relu, cout, out_split=True, out_f32=False)
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1_ = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            ops.conv2d_split(xs, w, scale, shift, relu, cout, out_split=True, out_f32=False)
        e1_.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1_) / 5
        print("   tma f16x3 %.3f ms  %.1f TFLOP/s (algorithmic fp32)" % (ms, 2.0 * B * H * W * cin * cout * taps / ms / 1e9), flush=True)


if stage in ("tmaperf", "all"):
    run_tma(1, 200, 176, 256, 256, 9, True, "tma BEV 3x3 B=1", time_it=True)
    run_tma(4, 200, 176, 256, 256, 9, True, "tma BEV 3x3 B=4", time_it=True)
if stage in ("tmaperf1",):
    run_tma(1, 200, 176, 256, 256, 9, True, "tma BEV 3x3 B=1", time_it=True)
    run_tma(1, 200, 176, 256, 256, 1, True, "tma BEV 1x1 B=1", time_it=True)
    run_tma(4, 200, 176, 256, 256, 1, True, "tma BEV 1x1 B=4", time_it=True)
print("done")
if stage in ("tmafull",):
    run_tma(1, 200, 176, 256, 28, 9, True, "tma full 256->28")
    run_tma(1, 200, 176, 28, 28, 1, False, "tma full 28->28 1x1")
    run_tma(1, 200, 176, 256, 20, 1, False, "tma full 256->20 1x1")
    run_tma(2, 200, 176, 256, 20, 1, False, "tma full B=2 256->20 1x1")
    run_tma(1, 200, 176, 256, 64, 9, True, "tma full 256->64")
    run_tma(1, 200, 176, 256, 128, 9, True, "tma full 256->128")


def tile_masks(nb, n_rows):
    """What the rulebook kernels record: per 128-row tile, the taps that occur among its first n_rows rows."""
    M, taps = nb.shape
    nt = (M + 127) // 128
    pad = np.full((nt * 128, taps), -1, np.int64)
    pad[:n_rows] = nb[:n_rows]
    present = (pad.reshape(nt, 128, taps) >= 0).any(1)
    return (present * (1 << np.arange(taps))[None, :]).sum(1).astype(np.int32)


if stage in ("splitperf",):
    M, cin, cout, taps = 120000, 64, 64, 27
    rs = np.random.RandomState(1)
    x = torch.randn(M, cin, device=dev)
    w = torch.randn(taps, cin, cout, device=dev) * 0.1
    # spatially coherent-ish neighbours: mostly nearby rows
    nb = np.where(rs.rand(M, taps) < 0.35, np.clip(np.arange(M)[:, None] + rs.randint(-300, 300, (M, taps)), 0, M - 1), -1).astype(np.int32)
    nbr = torch.from_numpy(nb).to(dev)
    d_rows = torch.tensor([M], dtype=torch.int32, device=dev)
    planes = ops.features_to_split(x)
    P = int((nb >= 0).sum())

    def timed(tag, nbr_t, tm, n_chunks):
        for _ in range(2):
            ops.spconv_split(planes, w, None, None, True, cout, M, nbr=nbr_t, d_rows=d_rows, tile_mask=tm)
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            ops.spconv_split(planes, w, None, None, True, cout, M, nbr=nbr_t, d_rows=d_rows, tile_mask=tm)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        pairs = int((nbr_t.cpu().numpy() >= 0).sum())
        print("splitperf %s dbg=%s: %.3f ms  pair-model %.0f GB/s  (%.0f clk per executed chunk)" % (
            tag, os.environ.get("SASSD_SPS_DBG", "0"), ms, pairs * (4 * cin + 4 * cout + 8) / ms / 1e6,
            ms * 1e-3 * 1.9e9 / (n_chunks / 148)), flush=True)

    timed("all taps", nbr, None, 27 * (M / 128))
    # 30 % of the (tile, tap) combinations absent, like the level-2 SubM rulebook of a KITTI-shaped cloud
    nb2 = nb.copy()
    gone = rs.rand((M + 127) // 128, taps) < 0.3
    nb2[np.repeat(gone, 128, axis=0)[:M]] = -1
    tm = tile_masks(nb2, M)
    timed("30% tile-taps absent, masks", torch.from_numpy(nb2).to(dev), torch.from_numpy(tm).to(dev),
          float(sum(bin(int(v) & 0x7ffffff).count("1") for v in tm)))
    timed("30% tile-taps absent, no masks", torch.from_numpy(nb2).to(dev), None, 27 * (M / 128))
    # one-frame layer sizes: 7 500 rows (59 tiles, tap split) and 14 000 rows (110 tiles)
    for rows in (5300, 7500, 14000):
        sub = torch.from_numpy(np.where(nb[:rows] >= rows, -1, nb[:rows])).to(dev)
        d_rows = torch.tensor([rows], dtype=torch.int32, device=dev)
        M_full, M = M, rows
        timed("%d rows" % rows, sub, torch.from_numpy(tile_masks(sub.cpu().numpy(), rows)).to(dev), 27 * (rows / 128))
        M = M_full
        d_rows = torch.tensor([M], dtype=torch.int32, device=dev)

if stage in ("splittrace",):
    # SASSD_SPS_TRACE=2 python tests/tools/tc_check.py splittrace <rows>: per-CTA clock sums of the second launch
    rows = int(sys.argv[2]) if len(sys.argv) > 2 else 120000
    cin = cout = 64
    rs = np.random.RandomState(1)
    x = torch.randn(rows, cin, device=dev)
    w = torch.randn(27, cin, cout, device=dev) * 0.1
    nb = np.where(rs.rand(rows, 27) < 0.35, np.clip(np.arange(rows)[:, None] + rs.randint(-300, 300, (rows, 27)), 0, rows - 1), -1).astype(np.int32)
    gone = rs.rand((rows + 127) // 128, 27) < 0.3
    nb[np.repeat(gone, 128, axis=0)[:rows]] = -1
    nbr = torch.from_numpy(nb).to(dev)
    tm = torch.from_numpy(tile_masks(nb, rows)).to(dev)
    d_rows = torch.tensor([rows], dtype=torch.int32, device=dev)
    planes = ops.features_to_split(x)
    for _ in range(3):
        ops.spconv_split(planes, w, None, None, True, cout, rows, nbr=nbr, d_rows=d_rows, tile_mask=tm)
    torch.cuda.synchronize()
    print("splittrace done", rows)
