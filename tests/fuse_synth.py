"""Synthetic local-mapping scenes for ORBmatcher::Fuse (tests only).

A shared map of 3-D points with descriptors, seen by several key frames (pinhole 752 x 480, fx = fy = 435): each key frame's
features are noisy projections of the points it sees (descriptor bit flips, all pyramid levels) plus distractors, and the key
frames mix stereo (mvuRight from the disparity, some features without a right match, a few at exactly 0.0) and monocular
(mvuRight = -1).  The pairs are the map points projected into each key frame with a small pose error, as Fuse would compute
them, with PredictScale near the observing feature's level."""
import numpy as np

from tests.oracle_lib import KP_DTYPE
from tests.proj_synth import SCALE, flip_bits

W, H = 752.0, 480.0
FX = FY = np.float32(435.0)
CX, CY = np.float32(376.0), np.float32(240.0)
BOUNDS = (0.0, 0.0, W, H)
INV_SIGMA2 = (np.float32(1.0) / (SCALE * SCALE)).astype(np.float32)        # mvInvLevelSigma2 = 1 / mvLevelSigma2, mvLevelSigma2 = s * s


def bounds_grid(bounds=BOUNDS):
    b = [np.float32(x) for x in bounds]
    return np.array(b + [np.float32(64) / (b[2] - b[0]), np.float32(48) / (b[3] - b[1])], np.float32)


def make_map(rng, n_points, crowd=0):
    """World points in front of the key frames, and their descriptors.  crowd > 0: the points sit in `crowd` tight clusters."""
    if crowd:
        c = np.stack([rng.uniform(-3, 3, crowd), rng.uniform(-2, 2, crowd), rng.uniform(4, 12, crowd)], 1)
        X = c[rng.integers(0, crowd, n_points)] + rng.normal(0, 0.03, (n_points, 3))
    else:
        X = np.stack([rng.uniform(-6, 6, n_points), rng.uniform(-4, 4, n_points), rng.uniform(2.5, 25, n_points)], 1)
    return X, rng.integers(0, 256, size=(n_points, 32), dtype=np.uint8)


def project(X, t):
    """Camera with identity rotation at t: (u, v, invz) in float32 (u = fx * x / z + cx)."""
    P = (X - t).astype(np.float32)
    invz = (np.float32(1.0) / P[:, 2]).astype(np.float32)
    u = (FX * P[:, 0] * invz + CX).astype(np.float32)
    v = (FY * P[:, 1] * invz + CY).astype(np.float32)
    return u, v, invz


def make_keyframe(rng, X, pdesc, t, stereo, bf=np.float32(47.9), see=0.7, n_distract=300, max_flip=60, jitter=0.8):
    """Features = projections of the points the key frame sees (noise, bit flips, all levels) plus distractors."""
    u, v, invz = project(X, t)
    seen = np.flatnonzero((rng.random(len(X)) < see) & (invz > 0) & (u > -5) & (u < W + 5) & (v > -5) & (v < H + 5))
    n = len(seen) + n_distract
    kp = np.zeros(n, KP_DTYPE)
    kp["x"][:len(seen)] = u[seen] + rng.normal(0, jitter, len(seen)); kp["y"][:len(seen)] = v[seen] + rng.normal(0, jitter, len(seen))
    kp["x"][len(seen):] = rng.uniform(0, W, n_distract); kp["y"][len(seen):] = rng.uniform(0, H, n_distract)
    kp["octave"] = rng.choice(8, n, p=[0.3, 0.2, 0.15, 0.1, 0.1, 0.06, 0.05, 0.04])
    kp["angle"] = rng.uniform(0, 360, n); kp["size"] = 31.0; kp["response"] = 50.0; kp["class_id"] = -1
    desc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    for j, p in enumerate(seen):
        desc[j] = flip_bits(rng, pdesc[p], int(rng.integers(0, max_flip + 1)))
    perm = rng.permutation(n)                                  # feature order unrelated to the point order
    kp, desc = kp[perm], desc[perm]
    obs = np.full(len(X), -1, np.int64)
    obs[seen] = np.argsort(perm)[:len(seen)]
    ur = None
    if stereo:
        iz = np.full(n, np.float32(1.0 / 8.0), np.float32)
        iz[obs[seen]] = invz[seen]
        ur = (kp["x"] - bf * iz + rng.normal(0, jitter, n)).astype(np.float32)
        ur[rng.random(n) < 0.25] = -1.0                            # no right match
        ur[rng.random(n) < 0.02] = 0.0                             # mvuRight == 0.0 takes the stereo gate
    return dict(kp=kp, desc=desc, ur=ur, bg=bounds_grid(), scale=SCALE, inv_sigma2=INV_SIGMA2, bf=np.float32(bf), t=t, obs=obs)


def make_pairs(rng, X, kfs, points_per_kf, pose_noise=0.6, valid_frac=0.9):
    """Pairs of each key frame with its map points (lists of point indices): projection with a pose error, PredictScale near
    the observing feature's level (random where the key frame does not observe the point)."""
    point, valid, u, v, invz, level, offs = [], [], [], [], [], [], [0]
    for k, K in enumerate(kfs):
        pts = np.asarray(points_per_kf[k], np.int64)
        uu, vv, iz = project(X[pts], K["t"])
        uu = (uu + rng.normal(0, pose_noise, len(pts))).astype(np.float32); vv = (vv + rng.normal(0, pose_noise, len(pts))).astype(np.float32)
        o = K["obs"][pts]
        lv = np.where(o >= 0, K["kp"]["octave"][np.maximum(o, 0)] + rng.choice([-1, 0, 0, 0, 1], len(pts)), rng.integers(0, 8, len(pts)))
        point.append(pts); u.append(uu); v.append(vv); invz.append(iz); level.append(np.clip(lv, 0, 7))
        valid.append((rng.random(len(pts)) < valid_frac) & (iz > 0))
        offs.append(offs[-1] + len(pts))
    cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt)  # noqa: E731
    return dict(kf_offsets=np.array(offs, np.int32), point=cat(point, np.int32), valid=cat(valid, np.uint8), u=cat(u, np.float32),
                v=cat(v, np.float32), invz=cat(invz, np.float32), level=cat(level, np.int32))


def scene(seed, n_kf=6, n_points=1500, crowd=0, n_distract=300, forward=True, pose_noise=0.6, max_flip=60, see=0.7):
    """forward=True: every key frame is paired with all map points (SearchInNeighbors' loop over the neighbours);
    forward=False: one key frame paired with all points (the final fuse into the current key frame)."""
    rng = np.random.default_rng(seed)
    X, pdesc = make_map(rng, n_points, crowd)
    kfs = [make_keyframe(rng, X, pdesc, np.array([rng.uniform(-0.8, 0.8), rng.uniform(-0.3, 0.3), rng.uniform(-1, 1)]), stereo=(k % 3 != 2),
                         see=see, n_distract=n_distract, max_flip=max_flip) for k in range(n_kf)]
    P = make_pairs(rng, X, kfs, [np.arange(n_points)] * n_kf, pose_noise=pose_noise)
    return X, pdesc, kfs, P
