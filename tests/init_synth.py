"""Synthetic monocular-initialisation pairs for SearchForInitialization (tests and tools only).

F2 is a frame as a 5 x nFeatures initialisation extractor leaves it (octaves spread over 8 levels, about 30 % at level 0); F1
holds F2's level-0 features moved by up to `max_move` pixels with up to `max_flip` flipped descriptor bits and a mostly
consistent rotation, shuffled among distractors.  vbPrevMatched starts as F1's own key points, as in
Tracking::MonocularInitialization."""
import numpy as np

from tests.oracle_lib import KP_DTYPE
from tests.proj_synth import flip_bits

W, H = 752.0, 480.0
BOUNDS = (0.0, 0.0, W, H)


def bounds_grid(bounds=BOUNDS):
    b = [np.float32(x) for x in bounds]
    return np.array(b + [np.float32(64) / (b[2] - b[0]), np.float32(48) / (b[3] - b[1])], np.float32)


def octaves(rng, n, p0=0.3):
    """Level 0 with probability p0, the rest over levels 1..7 with the 1/1.2 decay of mnFeaturesPerLevel."""
    w = np.array([1.2 ** -l for l in range(1, 8)])
    w = (1 - p0) * w / w.sum()
    return rng.choice(8, size=n, p=np.concatenate([[p0], w])).astype(np.int32)


def make_f2(rng, n, crowd=0, p0=0.3):
    kp = np.zeros(n, KP_DTYPE)
    if crowd:
        centres = rng.uniform([60, 60], [W - 60, H - 60], size=(crowd, 2))
        pts = centres[rng.integers(0, crowd, n)] + rng.normal(0, 12.0, size=(n, 2))
    else:
        pts = rng.uniform([0, 0], [W, H], size=(n, 2))
    kp["x"] = pts[:, 0].astype(np.float32); kp["y"] = pts[:, 1].astype(np.float32)
    kp["octave"] = octaves(rng, n, p0)
    kp["angle"] = rng.uniform(0, 360, n).astype(np.float32)
    kp["size"] = 31.0; kp["response"] = 50.0; kp["class_id"] = -1
    desc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    return kp, desc


def make_f1(rng, kp2, desc2, max_move=40.0, max_flip=60, n_distract=500, dup=1, rot_outliers=0.2):
    """F1 from F2's level-0 features (each one `dup` times), plus distractors; returns (kp1, desc1, prev_matched)."""
    src = np.repeat(np.nonzero(kp2["octave"] == 0)[0], dup)
    m = len(src)
    kp = np.zeros(m + n_distract, KP_DTYPE)
    ang = rng.uniform(0, 2 * np.pi, m); mag = rng.uniform(0, max_move, m)
    kp["x"][:m] = (kp2["x"][src] + mag * np.cos(ang)).astype(np.float32)
    kp["y"][:m] = (kp2["y"][src] + mag * np.sin(ang)).astype(np.float32)
    rot = np.where(rng.random(m) < rot_outliers, rng.uniform(0, 360, m), rng.normal(8.0, 6.0, m))
    kp["angle"][:m] = ((kp2["angle"][src] + rot) % 360).astype(np.float32)
    desc = np.zeros((m + n_distract, 32), np.uint8)
    desc[:m] = np.stack([flip_bits(rng, desc2[s], int(rng.integers(0, max_flip + 1))) for s in src]) if m else desc[:m]
    kp["x"][m:] = rng.uniform(0, W, n_distract).astype(np.float32); kp["y"][m:] = rng.uniform(0, H, n_distract).astype(np.float32)
    kp["octave"][m:] = octaves(rng, n_distract)
    kp["angle"][m:] = rng.uniform(0, 360, n_distract).astype(np.float32)
    desc[m:] = rng.integers(0, 256, size=(n_distract, 32), dtype=np.uint8)
    kp["size"] = 31.0; kp["response"] = 50.0; kp["class_id"] = -1
    perm = rng.permutation(m + n_distract)
    kp, desc = kp[perm], desc[perm]
    kp["angle"] = np.minimum(kp["angle"], np.float32(359.99))
    prev = np.stack([kp["x"], kp["y"]], 1).astype(np.float32)
    return kp, desc, prev


def init_pair(seed, n2=5000, crowd=0, max_move=40.0, max_flip=60, n_distract=None, dup=1):
    """The Tracking::MonocularInitialization shape: F2 with n2 features, F1 from its level-0 features plus distractors."""
    rng = np.random.default_rng(seed)
    kp2, desc2 = make_f2(rng, n2, crowd)
    kp1, desc1, prev = make_f1(rng, kp2, desc2, max_move, max_flip, n2 // 10 if n_distract is None else n_distract, dup)
    return kp1, desc1, prev, kp2, desc2


def next_frame(seed, kp2, desc2, max_move=8.0, max_flip=20):
    """A later frame of the same sequence: F2's features moved a little further, a few more bits flipped."""
    rng = np.random.default_rng(seed)
    kp = kp2.copy()
    kp["x"] = (kp["x"] + rng.uniform(-max_move, max_move, len(kp))).astype(np.float32)
    kp["y"] = (kp["y"] + rng.uniform(-max_move, max_move, len(kp))).astype(np.float32)
    desc = np.stack([flip_bits(rng, d, int(rng.integers(0, max_flip + 1))) for d in desc2]) if len(desc2) else desc2.copy()
    return kp, desc
