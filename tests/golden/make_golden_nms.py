"""Suppression bitmasks of the reference's rotated-NMS CUDA kernel (mmdet/ops/iou3d/src/iou3d_kernel.cu, unmodified,
compiled by oracle/build.py into oracle/_ref/libiou3d_ref.so) on the box sets of
tests/test_gpu_parity.py::test_nms_mask_and_keep, stored with those boxes as tests/golden/nms.npz.
Needs a CUDA device and the built reference library:

    python tests/golden/make_golden_nms.py [output .npz]
"""
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import build as OB  # noqa: E402
from tests.test_gpu_parity import NMS_CASES, NMS_THR, nms_case  # noqa: E402


def main(out):
    path = OB.build_ref()
    assert path, "oracle/_ref/libiou3d_ref.so (the reference NMS kernel) was not built"
    launch = getattr(ctypes.CDLL(path), "_Z11nmsLauncherPKfPyif")
    launch.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_float]
    launch.restype = None
    dev = torch.device("cuda:0")
    arrays = {}
    for n, seed in NMS_CASES:
        _, _, sorted_bev = nms_case(n, seed)
        boxes = sorted_bev.to(dev)
        mask = torch.zeros((n, (n + 63) // 64), dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        launch(ctypes.c_void_p(boxes.data_ptr()), ctypes.c_void_p(mask.data_ptr()), n, ctypes.c_float(NMS_THR))
        torch.cuda.synchronize()
        key = "n%d_seed%d" % (n, seed)
        arrays[key + "_bev"] = sorted_bev.numpy()
        arrays[key + "_mask"] = mask.cpu().numpy().view(np.uint64)
    np.savez_compressed(out, **arrays)
    print(out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "nms.npz"))
