"""The reference's configs/car_cfg.py and configs/multi_cfg.py as sassd_b200.Config.fromfile parses them, reduced to
what build_from_config reads (model, test_cfg and the data-side keys of data.val), stored as
tests/golden/reference_configs.json.  Tuples are stored as JSON lists.  Run once with a checkout of the reference:

    python tests/golden/make_golden_configs.py <reference checkout>
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import sassd_b200 as S  # noqa: E402

NAMES = ("car_cfg.py", "multi_cfg.py")
DATA_KEYS = ("class_names", "generator", "anchor_generator", "anchor_area_threshold", "out_size_factor")


def main(ref_root):
    out = {}
    for name in NAMES:
        cfg = S.Config.fromfile(os.path.join(ref_root, "configs", name))
        val = {k: cfg.data["val"][k] for k in DATA_KEYS}
        out[name] = dict(model=cfg.model, test_cfg=cfg.test_cfg, data=dict(val=val))
    path = os.path.join(ROOT, "tests", "golden", "reference_configs.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(path)


if __name__ == "__main__":
    main(sys.argv[1])
