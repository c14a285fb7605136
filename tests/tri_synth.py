"""Seeded scenes for the batched SearchForTriangulation tests and tools/triangulation_latency.py: one key frame (KF1) and its
neighbours as LocalMapping::CreateNewMapPoints searches them.  numpy + the vocabulary transform of the package."""
import numpy as np

from tests import bow_synth


def level_tables(rng):
    """Per-neighbour pyramid: its own level count and scale factor (mvScaleFactors, mvLevelSigma2 as float32 chains)."""
    n_levels = int(rng.integers(4, 13))
    f = np.float32(rng.choice([1.2, 1.25, 1.3]))
    scale = np.cumprod(np.array([1.0] + [f] * (n_levels - 1), np.float32)).astype(np.float32)
    sigma2 = (scale * scale * np.float32(rng.uniform(20.0, 60.0))).astype(np.float32)      # wide gate: a good share passes
    return scale, sigma2


def make_scene(voc, seed, n_a, n_kf, n_b, levelsup=2):
    """KF1 and n_kf neighbours: each neighbour holds noisy copies of a random part of KF1 (rotated by its own angle) plus
    unrelated features, random keypoints, a random relative pose (F12, epipole) and its own level tables."""
    v, vdesc, parent = voc
    rng = np.random.default_rng(seed)
    desc_a = bow_synth.make_features(seed + 1, vdesc, parent, n_a)
    ang_a = rng.uniform(0, 360, n_a).astype(np.float32)
    kp_a = bow_synth.make_keypoints(seed + 2, n_a, ang_a)
    _, fv_a = v.transform(desc_a, levelsup)
    A = dict(kp=kp_a, desc=desc_a, free=(rng.random(n_a) < 0.7).astype(np.uint8), stereo=(rng.random(n_a) < 0.4).astype(np.uint8), fv=fv_a)
    nbs = []
    for k in range(n_kf):
        n_m = int(0.5 * min(n_a, n_b))
        src = rng.choice(n_a, n_m, replace=False)
        copies = bow_synth.flip_bits(rng, desc_a[src], rng.integers(0, 40, n_m))
        rest = bow_synth.make_features(seed + 100 + k, vdesc, parent, n_b - n_m)
        perm = rng.permutation(n_b)
        desc_b = np.concatenate([copies, rest])[perm]
        ang = rng.uniform(0, 360, n_b).astype(np.float32)
        rot = rng.uniform(0, 360)
        inv = np.empty(n_b, np.int64); inv[perm] = np.arange(n_b)
        good = rng.random(n_m) < 0.8
        ab = ((ang_a[src] - np.float32(rot) + rng.normal(0, 4, n_m).astype(np.float32)) % np.float32(360)).astype(np.float32)
        ang[inv[:n_m][good]] = np.where(ab >= 360, 0, ab)[good]
        scale, sigma2 = level_tables(rng)
        kp_b = bow_synth.make_keypoints(seed + 200 + k, n_b, ang, nlevels=len(scale))
        _, fv_b = v.transform(desc_b, levelsup)
        F, ep = bow_synth.fundamental(seed + 300 + k)
        nbs.append(dict(kp=kp_b, desc=desc_b, free=(rng.random(n_b) < 0.7).astype(np.uint8),
                        stereo=(rng.random(n_b) < 0.4).astype(np.uint8), fv=fv_b, F12=F, ep=ep, scale=scale, sigma2=sigma2))
    return A, nbs
