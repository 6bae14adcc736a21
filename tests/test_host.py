"""CPU-side tests: host logic, the C-ABI library's exports, checkpoint format, config loader."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from sassd_b200 import lib as L
    hdr = open(os.path.join(ROOT, "include", "sassd_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(sassd_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 20
    lib = L.load()
    for name in declared:
        assert hasattr(lib, name), "libsassd_b200.so does not export %s" % name
    assert sorted(L.exported_symbols()) == declared
    assert lib.sassd_version() >= 100


def test_argument_validation_without_gpu():
    """Error paths that return before any CUDA call."""
    from sassd_b200 import lib as L
    lib = L.load()
    d = L.GConvDesc()
    assert lib.sassd_gconv(ctypes.byref(d), None, None, None, None, None, None, None, None) == -1
    assert lib.sassd_nms_sorted(None, 5, ctypes.c_float(0.1), None, None, None, 0, None) == -1
    assert lib.sassd_rulebook_conv_workspace_bytes(1, 20, 800, 704) > 20 * 800 * 704 // 8
    with pytest.raises(L.SassdError):
        L.check(-3, "x")
    assert L.decode_flags(2 | 8) == ["ROWS_CAP", "NMS_CAP"]
    # round-2 entry points
    assert lib.sassd_rulebook_conv_outputs_hash(None, None, 0, 1, 40, 1600, 1408, None, None, 0, None, None, 0, None,
                                                None, 0, None) == -1
    one = ctypes.c_void_p(8)            # never dereferenced on these paths: the argument checks come first
    assert lib.sassd_rulebook_conv_outputs_hash(one, one, 4, 1, 8, 16, 16, one, one, 10, one, one, 12, one, one, 1 << 20,
                                                None) == -1          # slots_out not a power of two >= 2 * rows_cap_out
    d = L.Conv2dDesc()
    d.batch, d.H, d.W, d.cin, d.cin_stored, d.cout, d.taps, d.relu = 1, 200, 176, 256, 256, 256, 9, 1
    # constant-region rule outside its validity range (ADVICE r1): reach beyond the recorded tile distances
    assert lib.sassd_conv2d_f16x3_occ(ctypes.byref(d), one, one, None, None, None, one, one, 10, one, None, None) == \
        -4
    d.H = 201                           # a 1-pixel partial edge tile cannot absorb a 3-pixel padding disturbance
    assert lib.sassd_conv2d_f16x3_occ(ctypes.byref(d), one, one, None, None, None, one, one, 4, one, None, None) == \
        -4
    # launch hint: returns the previous setting
    prev = lib.sassd_set_pdl(1)
    assert lib.sassd_set_pdl(prev) == 1


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "sa-ssd_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("oracle/", "").lower() or f == "checkpoint.py" or \
                    not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f


def test_config_loader_and_registry():
    import sassd_b200 as S
    cfg = S.Config.fromfile(os.path.join(ROOT, "configs", "car_cfg.py"))
    assert cfg.model.type == "SingleStageDetector" and cfg.test_cfg.extra.nms.iou_thr == 0.1
    model, vg, aset = S.build_from_config(cfg, device="cpu")
    assert type(model.neck).__name__ == "SpMiddleFHD" and type(model.extra_head).__name__ == "PSWarpHead"
    assert list(vg.grid_size) == [1408, 1600, 40]
    assert aset.anchors.shape == (70400, 7) and aset.feature_map_size == [1, 200, 176]
    assert sum(p.numel() for p in model.parameters()) == 5339548
    cfg3 = S.Config.fromfile(os.path.join(ROOT, "configs", "multi_cfg.py"))
    m3, _, a3 = S.build_from_config(cfg3, device="cpu")
    assert a3.anchors.shape == (211200, 7) and m3.rpn_head.head_channels == 72
    with pytest.raises(TypeError):
        S.obj_from_dict(dict(foo=1))
    with pytest.raises(FileNotFoundError):
        S.Config.fromfile("/nonexistent.py")


def test_reference_configs_load_unchanged(golden_dir):
    """The reference's two configs as Config.fromfile parsed them (tests/golden/reference_configs.json, made by
    tests/golden/make_golden_configs.py) build unchanged, and the project's configs hold the same values."""
    import sassd_b200 as S
    with open(os.path.join(golden_dir, "reference_configs.json")) as f:
        ref = json.load(f)
    for name, na in (("car_cfg.py", 70400), ("multi_cfg.py", 211200)):
        cfg = S.Config(ref[name])
        model, vg, aset = S.build_from_config(cfg, device="cpu")
        assert aset.anchors.shape[0] == na
        ours = json.loads(json.dumps(S.Config.fromfile(os.path.join(ROOT, "configs", name))._cfg_dict))
        assert ours["model"] == ref[name]["model"] and ours["test_cfg"] == ref[name]["test_cfg"], name
        for k, v in ref[name]["data"]["val"].items():
            assert ours["data"]["val"][k] == v, (name, k)


def test_checkpoint_roundtrip_reference_format(tmp_path):
    import sassd_b200 as S
    from sassd_b200 import checkpoint as C
    cfg = S.Config.fromfile(os.path.join(ROOT, "configs", "car_cfg.py"))
    model, _, _ = S.build_from_config(cfg, device="cpu")
    sd = C.make_synthetic_state_dict(0, 1)
    path = str(tmp_path / "checkpoint_epoch_1.pth")
    C.save_checkpoint(sd, path, epoch=1, module_prefix=True)   # saved through a DataParallel wrapper
    n, missing = C.load_params_from_file(model, path, to_cpu=True)
    assert n == len(sd)
    assert all("num_batches" in k or k.startswith("neck.point_") for k in missing)
    got = model.state_dict()
    for k, v in sd.items():
        assert torch.equal(got[k], v), k
    # spconv-v1 weight layout is kept: [kz, ky, kx, Cin, Cout]
    assert tuple(got["neck.backbone.conv0.0.weight"].shape) == (3, 3, 3, 4, 16)
    assert tuple(got["neck.backbone.extra_conv.0.weight"].shape) == (1, 1, 1, 64, 64)


def test_anchor_grid_matches_oracle_bitwise():
    from oracle import ref_pipeline as O
    from sassd_b200.anchors import AnchorGeneratorStride, rbbox2d_to_near_bbox
    car = dict(sizes=[1.6, 3.9, 1.56], anchor_strides=[0.4, 0.4, 1.0], anchor_offsets=[0.2, -39.8, -1.78],
               rotations=[0, 1.57])
    a = AnchorGeneratorStride(**car)([1, 200, 176]).reshape(-1, 7)
    oa, obv = O.make_anchors([car])
    assert np.array_equal(a, oa) and np.array_equal(rbbox2d_to_near_bbox(a[:, [0, 1, 3, 4, 6]]), obv)


def test_synthetic_cloud_shape_and_determinism():
    from sassd_b200.synth import synth_cloud
    a, b = synth_cloud(3), synth_cloud(3)
    assert a.dtype == np.float32 and a.shape[1] == 4 and np.array_equal(a, b)
    assert 18000 < a.shape[0] < 22000
    assert synth_cloud(3, fov_deg=180.0).shape[0] > 100000


def test_no_cpu_fallback():
    """The product path must fail loudly without a CUDA device."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from sassd_b200 import lib as L
    from sassd_b200.voxel_generator import VoxelGenerator
    vg = VoxelGenerator([0.05, 0.05, 0.1], [0, -40., -3., 70.4, 40., 1.], 5, 20000)
    with pytest.raises(L.SassdError):
        vg.generate(np.zeros((10, 4), np.float32))
