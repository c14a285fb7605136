"""Seeded synthetic batches for orbx_search_by_bow_batch: one fixed feature set and a list of key frames, each holding
planted noisy copies of part of the fixed set (numpy only, built on bow_synth)."""
import numpy as np

from tests import bow_synth

# what a key frame of a batch is built to exercise
NORMAL, EMPTY, DISJOINT, INVALID = "normal", "empty", "disjoint", "invalid"


def make_batch(seed, voc_desc, parent, n, kf_sizes, kinds=None, match_frac=0.5, rot=37.0):
    """The fixed side (desc, angle, valid) and one dict per key frame (desc, angle, valid, kind).
    - the fixed set holds a few exact duplicate rows, and each key frame exact copies of fixed features and some of its planted
      copies twice, so that ties and failing ratio tests occur on both sides;
    - planted copies follow a dominant rotation with outliers, so the rotation filter has work;
    - kind EMPTY: n = 0; DISJOINT: attach_fvs moves its node ids off the vocabulary, so it shares no node with the fixed side;
      INVALID: no feature has a usable map point."""
    rng = np.random.default_rng(seed)
    desc = bow_synth.make_features(seed + 1, voc_desc, parent, n)
    n_dup = n // 20
    if n_dup:
        desc[rng.choice(n, n_dup, replace=False)] = desc[rng.choice(n, n_dup, replace=False)]
    angle = rng.uniform(0, 360, n).astype(np.float32)
    valid = (rng.random(n) < 0.85).astype(np.uint8)
    kinds = list(kinds) if kinds is not None else [NORMAL] * len(kf_sizes)
    kfs = []
    for k, (m, kind) in enumerate(zip(kf_sizes, kinds)):
        if kind == EMPTY:
            m = 0
        n_m = int(match_frac * min(n, m))
        src = rng.choice(n, n_m, replace=False)
        copies = bow_synth.flip_bits(rng, desc[src], rng.integers(0, 40, n_m))
        exact = rng.random(n_m) < 0.1
        copies[exact] = desc[src[exact]]
        n_twice = min(n_m // 20, m - n_m)
        planted = np.concatenate([copies, copies[:n_twice]])
        psrc = np.concatenate([src, src[:n_twice]])
        rest = bow_synth.make_features(seed + 100 + k, voc_desc, parent, m - len(planted))
        kdesc = np.concatenate([planted, rest]).astype(np.uint8)
        perm = rng.permutation(m)
        kdesc = kdesc[perm]
        kangle = rng.uniform(0, 360, m).astype(np.float32)
        inv = np.empty(m, np.int64)
        inv[perm] = np.arange(m)
        good = rng.random(len(planted)) < 0.8
        pa = (angle[psrc] - np.float32(rot) + rng.normal(0, 4, len(planted)).astype(np.float32)) % np.float32(360)
        pa = np.where(pa >= 360, 0, pa).astype(np.float32)
        kangle[inv[:len(planted)][good]] = pa[good]
        kvalid = (rng.random(m) < 0.85).astype(np.uint8)
        if kind == INVALID:
            kvalid[:] = 0
        kfs.append(dict(desc=kdesc, angle=kangle, valid=kvalid, kind=kind))
    return dict(desc=desc, angle=angle, valid=valid, kfs=kfs)


def attach_fvs(B, transform):
    """Set B["fv"] and every key frame's "fv" to transform(descriptors) (an object with node_ids / offsets / indices, built by
    calling its own type); a DISJOINT key frame's node ids are moved past every vocabulary node."""
    B["fv"] = transform(B["desc"])
    for kf in B["kfs"]:
        fv = transform(kf["desc"])
        if kf["kind"] == DISJOINT:
            fv = type(fv)(fv.node_ids + 10_000_000, fv.offsets, fv.indices)
        kf["fv"] = fv
    return B
