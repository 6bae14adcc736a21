"""Outputs of the reference's rotated-NMS CUDA kernels (mmdet/ops/iou3d/src/iou3d_kernel.cu, unmodified, compiled by
oracle/build.py into oracle/_ref/libiou3d_ref.so), stored with their input boxes as tests/golden/nms.npz.

* n<N>_seed<S>_bev / _mask: nmsLauncher's suppression bitmask (IoU threshold 0.1) on the random box sets of
  tests/test_gpu_parity.py::test_nms_mask_and_keep.
* <set>_bev, <set>_mask_t<thr> (thr 0.1 and 0.0), and for the adversarial sets <set>_iou (boxesioubevLauncher's full
  [n, n] matrix of the set against itself): the sets of tests/nms_box_sets.py::adversarial_sets, checked by
  tests/test_detection_tail.py.

Needs a CUDA device and the built reference library:

    python tests/golden/make_golden_nms.py [output .npz]

When tests/golden/nms.npz exists, no key may disappear, and every output of a box set whose boxes come out unchanged
must come out with the same dtype, shape and bytes; the script fails otherwise, so regenerating cannot silently change
what the tests compare against.  A set whose boxes were changed on purpose in tests/nms_box_sets.py is listed.
"""
import ctypes
import os
import re
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import build as OB  # noqa: E402
from tests.nms_box_sets import THRESHOLDS, adversarial_sets  # noqa: E402
from tests.test_gpu_parity import NMS_CASES, NMS_THR, nms_case  # noqa: E402


def thr_key(thr):
    return "t%g" % thr


GOLDEN = os.path.join(ROOT, "tests", "golden", "nms.npz")


def main(out):
    path = OB.build_ref()
    assert path, "oracle/_ref/libiou3d_ref.so (the reference NMS kernel) was not built"
    lib = ctypes.CDLL(path)
    launch = getattr(lib, "_Z11nmsLauncherPKfPyif")
    launch.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_float]
    launch.restype = None
    iou_launch = getattr(lib, "_Z19boxesioubevLauncheriPKfiS0_Pf")
    iou_launch.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    iou_launch.restype = None
    dev = torch.device("cuda:0")

    def ref_mask(boxes, thr):
        n = boxes.shape[0]
        b = torch.from_numpy(np.ascontiguousarray(boxes)).to(dev)
        mask = torch.zeros((n, (n + 63) // 64), dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        launch(ctypes.c_void_p(b.data_ptr()), ctypes.c_void_p(mask.data_ptr()), n, ctypes.c_float(thr))
        torch.cuda.synchronize()
        return mask.cpu().numpy().view(np.uint64)

    def ref_iou(boxes):
        n = boxes.shape[0]
        b = torch.from_numpy(np.ascontiguousarray(boxes)).to(dev)
        iou = torch.full((n, n), float("nan"), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        iou_launch(n, ctypes.c_void_p(b.data_ptr()), n, ctypes.c_void_p(b.data_ptr()), ctypes.c_void_p(iou.data_ptr()))
        torch.cuda.synchronize()
        return iou.cpu().numpy()

    arrays = {}
    for n, seed in NMS_CASES:
        _, _, sorted_bev = nms_case(n, seed)
        key = "n%d_seed%d" % (n, seed)
        arrays[key + "_bev"] = sorted_bev.numpy()
        arrays[key + "_mask"] = ref_mask(sorted_bev.numpy(), NMS_THR)
    for name, boxes in adversarial_sets().items():
        arrays[name + "_bev"] = boxes
        for thr in THRESHOLDS:
            arrays["%s_mask_%s" % (name, thr_key(thr))] = ref_mask(boxes, thr)
        if name.startswith("adv_"):
            arrays[name + "_iou"] = ref_iou(boxes)
    if os.path.exists(GOLDEN):
        old = np.load(GOLDEN)
        same = changed = 0
        for k in old.files:
            assert k in arrays, "key %s would disappear" % k
            a, b = old[k], arrays[k]
            unchanged = a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()
            bev = re.sub(r"_(bev|mask(_t[0-9.]+)?|iou)$", "_bev", k)
            if old[bev].tobytes() == arrays[bev].tobytes() and old[bev].shape == arrays[bev].shape:
                assert unchanged, "key %s changed although its boxes did not" % k
            elif k == bev:
                print("boxes of %s changed in tests/nms_box_sets.py: its outputs are regenerated" % k[:-4])
            same += unchanged
            changed += not unchanged
        print("%d existing keys unchanged (dtype, shape, bytes), %d regenerated for changed boxes" % (same, changed))
    np.savez_compressed(out, **arrays)
    print(out, os.path.getsize(out), "bytes,", len(arrays), "keys")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else GOLDEN)
