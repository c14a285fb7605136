"""Synthetic loop-closing scenes for the Sim3 SearchByProjection and the Sim3 Fuse (tests only).

The map, key frames and projections are those of tests/fuse_synth.py (pinhole 752 x 480, 8 levels).  The Sim3 searches read
neither mvuRight nor mvInvLevelSigma2, so the key frames are monocular.  A SearchByProjection scene is one key frame with a
share of its slots already holding a match (vpMatched != NULL on entry) and the covisible window's points projected into it."""
import numpy as np

from tests.fuse_synth import make_keyframe, make_map, make_pairs, scene


def sbp_scene(seed, n_points=8000, see=0.3, n_distract=500, occ_frac=0.3, crowd=0, pose_noise=0.6, max_flip=60):
    """Returns (K, occupied, P, pdesc): P holds valid / u / v / level per point (point i's descriptor = pdesc[i])."""
    rng = np.random.default_rng(seed)
    X, pdesc = make_map(rng, n_points, crowd)
    t = np.array([rng.uniform(-0.8, 0.8), rng.uniform(-0.3, 0.3), rng.uniform(-1, 1)])
    K = make_keyframe(rng, X, pdesc, t, stereo=False, see=see, n_distract=n_distract, max_flip=max_flip)
    P = make_pairs(rng, X, [K], [np.arange(n_points)], pose_noise=pose_noise)
    occupied = (rng.random(len(K["kp"])) < occ_frac).astype(np.uint8)
    return K, occupied, P, pdesc


def fuse_scene(seed, n_kf=6, n_points=1500, **kw):
    """The key frames of SearchAndFuse paired with every loop map point (tests/fuse_synth.scene, monocular key frames)."""
    X, pdesc, kfs, P = scene(seed, n_kf=n_kf, n_points=n_points, **kw)
    return [dict(k, ur=None) for k in kfs], P, pdesc
