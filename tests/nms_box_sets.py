"""Adversarial BEV box sets [n, 5] (x1, y1, x2, y2, ry) for the rotated IoU / NMS kernels, built deterministically.

They sit where the rotated-overlap arithmetic is fragile and where a change of operation order or of FMA contraction
would flip a bit: identical boxes, the anchor rotations 0 and 1.57 and multiples of +-pi/2 on one centre, shared and
collinear edges (offset by one ulp), corners that touch, nested, tiny and long boxes, centres near x = 70 m, and pairs
whose circumscribed circles are just apart or just overlapping (the boundary of sassd_nms_mask's far-pair shortcut).
tests/golden/make_golden_nms.py stores the reference kernel's masks and IoU matrices of these sets in
tests/golden/nms.npz; tests/test_detection_tail.py checks the kernels against them.
"""
import numpy as np

F32 = np.float32
HALF_PI = float(F32(np.pi / 2))


def _bev(cx, cy, w, l, r):
    """boxes3d_to_bev_torch in fp32: (x - w/2, y - l/2, x + w/2, y + l/2, r)."""
    cx, cy, w, l, r = np.broadcast_arrays(*(np.asarray(v, F32) for v in (cx, cy, w, l, r)))
    hw, hl = w / F32(2), l / F32(2)
    return np.stack([cx - hw, cy - hl, cx + hw, cy + hl, r], -1).astype(F32).reshape(-1, 5)


def _dups():
    return np.repeat(_bev(12.3, -4.1, 1.6, 3.9, 0.3), 10, 0)


def _rotations():
    rots = [0.0, 1.57, HALF_PI, -HALF_PI, float(F32(np.pi)), -float(F32(np.pi)), float(F32(3 * np.pi / 2)),
            float(F32(2 * np.pi)), 3.0, -1.57]
    out = [_bev(20.0, 5.0, 1.6, 3.9, r) for r in rots]
    out += [_bev(20.0, 5.0, 2.0, 2.0, r) for r in rots[:4]]          # square: the rotations coincide geometrically
    return np.concatenate(out)


def _edges():
    a = np.array([[0, 0, 2, 4, 0]], F32)
    up, dn = np.nextafter(F32(2), F32(3)), np.nextafter(F32(2), F32(1))
    sets = [a,
            np.array([[2, 0, 4, 4, 0]], F32),                      # shares the edge x = 2
            np.array([[up, 0, 4, 4, 0]], F32),                     # one ulp apart
            np.array([[dn, 0, 4, 4, 0]], F32),                     # one ulp overlap
            np.array([[2, 1, 4, 3, 0]], F32),                      # part of the edge shared
            np.array([[0, 4, 2, 8, 0]], F32),                      # shares the edge y = 4
            np.array([[0, 0, 2, 4, HALF_PI]], F32),                # same box rotated by pi/2 about its centre
            np.array([[0, 2, 2, 6, 0]], F32),                      # collinear x edges, half overlap
            np.array([[0, 0, 2, 4, float(F32(np.pi))]], F32)]      # rotated by pi: same footprint
    return np.concatenate(sets)


def _corners():
    sets = [np.array([[0, 0, 2, 4, 0], [2, 4, 4, 8, 0], [-2, -4, 0, 0, 0], [2, -4, 4, 0, 0]], F32)]
    d = float(np.sqrt(2.0))                                        # unit squares at 45 deg touching corner to corner
    sets.append(_bev([30.0, 30.0 + d, 30.0], [0.0, 0.0, d], 1.0, 1.0, float(F32(np.pi / 4))))
    return np.concatenate(sets)


def _nested():
    return np.concatenate([_bev(40.0, -10.0, w, l, r) for w, l, r in
                           [(4.0, 8.0, 0.0), (1.6, 3.9, 0.0), (1.6, 3.9, 0.7), (0.5, 0.5, 1.2), (3.9, 3.9, 0.0),
                            (3.0, 6.0, 1.57)]])


def _tiny_long():
    return np.concatenate([_bev(50.0, 10.0, 0.01, 0.01, 0.0), _bev(50.0, 10.0, 0.01, 0.01, 0.5),
                           _bev(50.005, 10.005, 0.01, 0.01, 0.0), _bev(50.0, 10.0, 0.2, 20.0, 0.0),
                           _bev(50.0, 10.0, 0.2, 20.0, 1.57), _bev(50.0, 15.0, 20.0, 0.3, 0.2),
                           _bev(50.0, 10.0, 1.6, 3.9, 0.0)])


def _far_x():
    rs = np.random.RandomState(70)
    n = 24
    return _bev(70.0 + rs.uniform(-0.8, 0.8, n), 30.0 + rs.uniform(-1.5, 1.5, n), rs.normal(1.6, 0.05, n),
                rs.normal(3.9, 0.1, n), rs.choice([0.0, 1.57, 0.3], n))


REACH_FACTORS = (1 - 2e-3, 1 - 1e-3, 1 - 1e-4, 1 + 1e-4, 1 + 1e-3, 1 + 2e-3)


def _reach_pairs():
    """Pairs whose corners point at each other along the line of centres, at centre distance reach * f (reach = sum
    of the circumscribed radii): below 1 the corners overlap slightly, above 1 they are apart; around f = 1 + 1e-3 the
    squared distance crosses the shortcut's reach^2 * 1.002 + 1e-6.  The kernels turn a box's corners by -ry about its
    centre (x' = x cos + y sin, y' = -x sin + y cos), so the offset along the diagonal is turned the same way."""
    out = []
    for k, (w, l, theta, x0) in enumerate([(1.6, 3.9, 0.0, 5.0), (1.6, 3.9, 0.9, 15.0), (2.0, 2.0, 0.0, 25.0),
                                           (0.05, 0.08, 0.4, 35.0), (1.6, 3.9, 0.0, 69.5)]):
        reach = float(np.hypot(w, l))                                # 2 radii of equal boxes
        ux, uy = w / reach, l / reach                                # diagonal direction of the unrotated box
        c, s = np.cos(theta), np.sin(theta)
        dx, dy = c * ux + s * uy, -s * ux + c * uy                   # the diagonal, turned as the kernels turn corners
        for f in REACH_FACTORS:
            cy = -20.0 + 6.0 * k
            out.append(_bev(x0, cy, w, l, theta))
            out.append(_bev(x0 + f * reach * dx, cy + f * reach * dy, w, l, theta))
    return np.concatenate(out)


GROUPS = {"dups": _dups, "rotations": _rotations, "edges": _edges, "corners": _corners, "nested": _nested,
          "tiny_long": _tiny_long, "far_x": _far_x, "reach": _reach_pairs}
MIX_SIZES = (127, 129, 191, 193)      # 64k +- 1: partial last mask word, one column block more or less
RANDOM_N = 5000
THRESHOLDS = (0.1, 0.0)               # the product's IoU threshold, and "any overlap" (every positive IoU suppresses)


def adversarial_sets():
    """name -> float32 [n, 5] BEV boxes in the order the NMS kernels take them (already sorted by score)."""
    sets = {"adv_" + k: f() for k, f in GROUPS.items()}
    allb = np.concatenate(list(sets.values()))
    rs = np.random.RandomState(64)
    for n in MIX_SIZES:
        # the groups back to back, cut at n (127 and 129 hold only part of them: there are 137 group boxes); beyond
        # the groups, jittered copies of them (heavy overlap across column blocks); shuffled
        reps = int(np.ceil(n / len(allb)))
        b = np.concatenate([allb] * reps)[:n].copy()
        jit = rs.normal(0, 0.05, (n, 2)).astype(F32)
        b[len(allb):, 0:3:2] += jit[len(allb):, :1]
        b[len(allb):, 1:4:2] += jit[len(allb):, 1:]
        sets["adv_mix%d" % n] = b[rs.permutation(n)]
    rs = np.random.RandomState(5000)
    n = RANDOM_N
    sets["rand%d" % n] = _bev(rs.uniform(0, 70.4, n), rs.uniform(-40, 40, n), rs.normal(1.6, 0.1, n),
                              rs.normal(3.9, 0.3, n), rs.uniform(-4, 4, n))
    return sets
