"""GPU tests of the round-2 entry points and robustness fixes: re-entrant matcher, device-resident stereo matching, the
one-call stereo frame, the sharded 2-NN behind the C ABI, handle state after a failed configuration, orbx_sync with a
caller's stream.  Everything goes through the C ABI (liborbx.so) and is compared with the CPU oracle, bit for bit."""
import ctypes as C
import threading

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from wut_cuda_orb_slam3_b200 import synth
from wut_cuda_orb_slam3_b200.capi import OrbxError, check, lib, ptr

pytestmark = pytest.mark.gpu


def test_knn2_device_is_reentrant_two_threads_two_streams(oracle):
    """ORBmatcher::DescriptorDistance users run on the Tracking, LocalMapping and LoopClosing threads at once (SURVEY.md §3.3):
    two host threads, two streams, different databases (both chunked, so both need scratch), 200 calls each."""
    import torch
    dev = torch.device("cuda:0")
    cases = []
    for t, (nq, ndb, seed) in enumerate([(700, 300_000, 21), (1100, 260_000, 22)]):
        db = synth.descriptors(seed, ndb); q = synth.descriptors(seed, nq, is_query=True, ndb=ndb, plant_every=3)
        db[ndb // 2] = db[5]; q[0] = db[5]                         # a tie
        ridx, rdist = oracle.knn2(q, db)
        cases.append((torch.from_numpy(q).to(dev), torch.from_numpy(db).to(dev), nq, ndb, ridx, rdist))
    errors = []

    def worker(t):
        try:
            d_q, d_db, nq, ndb, ridx, rdist = cases[t]
            st = torch.cuda.Stream(device=dev)
            d_idx = torch.empty((nq, 2), dtype=torch.int32, device=dev); d_dist = torch.empty_like(d_idx)
            for it in range(200):
                d_idx.fill_(-7); d_dist.fill_(-7)
                st.wait_stream(torch.cuda.current_stream(dev))
                orbx.knn2_device(d_q, nq, d_db, ndb, d_idx, d_dist, stream=st.cuda_stream)
                st.synchronize()
                if not (np.array_equal(d_idx.cpu().numpy(), ridx) and np.array_equal(d_dist.cpu().numpy(), rdist)):
                    errors.append((t, it))
                    return
        except Exception as e:          # noqa: BLE001
            errors.append((t, repr(e)))

    ths = [threading.Thread(target=worker, args=(t,)) for t in range(2)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    assert not errors, errors


def _pair(seed=31, cols=752, rows=480):
    return synth.image(seed, cols, rows, view=0, max_disp=40), synth.image(seed, cols, rows, view=1, max_disp=40)


def test_stereo_match_extractors_with_different_capacity(oracle):
    """exL sized for 4 frames, exR for 1: the level slabs of the two pyramids lie at different offsets (ADVICE r1)."""
    L, R = _pair()
    exL = orbx.ORBextractor(1200, 1.2, 8, 20, 7, max_cols=752, max_rows=480, max_batch=4)
    exR = orbx.ORBextractor(1200, 1.2, 8, 20, 7, max_cols=752, max_rows=480, max_batch=1)
    nm, n, kps, desc = exL.extract_batch(np.stack([L, L, L, L]))          # grows exL's slot to 4 frames
    _, kL, dL = exL(L, None, (0, 0)); _, kR, dR = exR(R, None, (0, 0))
    u, d = orbx.compute_stereo_matches(exL, exR, kL, dL, kR, dR, 47.9, 435.2)
    oL = oracle.extractor(1200, 1.2, 8, 20, 7); oR = oracle.extractor(1200, 1.2, 8, 20, 7)
    okL, odL, _ = oL.extract(L, (0, 0)); okR, odR, _ = oR.extract(R, (0, 0))
    ou, od, kept = oracle.stereo_match(oL, oR, okL, odL, okR, odR, 47.9, 435.2)
    assert kept > 50 and np.array_equal(u, ou) and np.array_equal(d, od)
    # the other way round
    u2, d2 = orbx.compute_stereo_matches(exR, exL, kR, dR, kL, dL, 47.9, 435.2)
    ou2, od2, _ = oracle.stereo_match(oR, oL, okR, odR, okL, odL, 47.9, 435.2)
    assert np.array_equal(u2, ou2) and np.array_equal(d2, od2)


@pytest.mark.parametrize("cols,rows,nf", [(752, 480, 1200), (1241, 376, 2000)])
def test_extract_stereo_one_call_equals_separate_calls(oracle, cols, rows, nf):
    """orbx_extract_stereo (Frame.cc:124-143 in one call, matcher on device-resident features) against the three-call path
    and against the oracle; repeated so that the captured graphs and the second-call state are exercised."""
    exL = orbx.ORBextractor(nf, 1.2, 8, 20, 7); exR = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    sL = orbx.ORBextractor(nf, 1.2, 8, 20, 7); sR = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    oL = oracle.extractor(nf, 1.2, 8, 20, 7); oR = oracle.extractor(nf, 1.2, 8, 20, 7)
    for rep, seed in enumerate([31, 32, 31, 33]):
        L, R = _pair(seed, cols, rows)
        kL, dL, kR, dR, u, d = orbx.extract_stereo(exL, exR, L, R, 47.9, 435.2)
        _, k1, d1 = sL(L, None, (0, 0)); _, k2, d2 = sR(R, None, (0, 0))
        assert kL.tobytes() == k1.tobytes() and kR.tobytes() == k2.tobytes()
        assert np.array_equal(dL, d1) and np.array_equal(dR, d2)
        u1, dd1 = orbx.compute_stereo_matches(sL, sR, k1, d1, k2, d2, 47.9, 435.2)
        assert np.array_equal(u, u1) and np.array_equal(d, dd1), rep
        if rep < 2:
            okL, odL, _ = oL.extract(L, (0, 0)); okR, odR, _ = oR.extract(R, (0, 0))
            ou, od, kept = oracle.stereo_match(oL, oR, okL, odL, okR, odR, 47.9, 435.2)
            assert kept > 50 and np.array_equal(u, ou) and np.array_equal(d, od)


def test_stereo_match_device_on_batch_outputs(oracle):
    """orbx_stereo_match_device queued behind orbx_extract_batch_device on one stream: counts are read on the device."""
    import torch
    dev = torch.device("cuda:0")
    L, R = _pair(35)
    ex = orbx.ORBextractor(1200, 1.2, 8, 20, 7, max_cols=752, max_rows=480, max_batch=2)
    cap = ex.max_keypoints(480, 752)
    d_img = torch.from_numpy(np.stack([L, R])).to(dev)
    d_kps = torch.zeros((2, cap, 7), dtype=torch.float32, device=dev); d_desc = torch.zeros((2, cap, 32), dtype=torch.uint8, device=dev)
    d_n = torch.zeros(2, dtype=torch.int32, device=dev); d_nm = torch.zeros(2, dtype=torch.int32, device=dev)
    d_u = torch.full((cap,), -5.0, dtype=torch.float32, device=dev); d_d = torch.full((cap,), -5.0, dtype=torch.float32, device=dev)
    st = torch.cuda.Stream(device=dev)
    st.wait_stream(torch.cuda.current_stream(dev))
    ex.extract_batch_device(d_img, 2, 480, 752, 752, 480 * 752, d_kps, d_desc, cap, d_n, d_nm, (0, 0), stream=st.cuda_stream)
    check(lib().orbx_stereo_match_device(ex._h, 0, ex._h, 1, ptr(d_kps[0]), ptr(d_desc[0]), ptr(d_n[0:]), cap, ptr(d_kps[1]), ptr(d_desc[1]),
                                         ptr(d_n[1:]), cap, 47.9, 435.2, ptr(d_u), ptr(d_d), C.c_void_p(st.cuda_stream)))
    check(lib().orbx_sync(ex._h))          # must cover the caller's stream too
    n = d_n.cpu().numpy()
    oL = oracle.extractor(1200, 1.2, 8, 20, 7); oR = oracle.extractor(1200, 1.2, 8, 20, 7)
    okL, odL, _ = oL.extract(L, (0, 0)); okR, odR, _ = oR.extract(R, (0, 0))
    ou, od, kept = oracle.stereo_match(oL, oR, okL, odL, okR, odR, 47.9, 435.2)
    assert n[0] == len(okL) and n[1] == len(okR)
    assert np.array_equal(d_u.cpu().numpy()[:n[0]], ou) and np.array_equal(d_d.cpu().numpy()[:n[0]], od)
    assert (d_u.cpu().numpy()[n[0]:] == -5.0).all()
    # the probes wait for the caller's stream as well and refuse frames the last call did not produce
    assert np.array_equal(ex.pyramid_level(0, frame=1), R)
    with pytest.raises(OrbxError):
        ex.pyramid_level(0, frame=2)


def test_sharded_knn2_world1_through_nccl(oracle):
    """orbx_comm_* + orbx_knn2_sharded with a one-rank NCCL communicator (the 2..8-rank run is tools/sharded_check.py)."""
    import torch
    dev = torch.device("cuda:0")
    ndb, nq = 120_001, 999
    db = synth.descriptors(9, ndb); q = synth.descriptors(9, nq, is_query=True, ndb=ndb, plant_every=2)
    sm = orbx.ShardedMatcher(0, 1, 0, lambda b: b)
    assert sm.nccl_version() > 20000
    first, cnt = sm.shard_rows(ndb, 1, 0)
    assert (first, cnt) == (0, ndb)
    d_db = torch.from_numpy(db).to(dev); d_q = torch.from_numpy(q).to(dev)
    d_idx = torch.empty((nq, 2), dtype=torch.int32, device=dev); d_dist = torch.empty_like(d_idx)
    for _ in range(3):
        sm.knn2(d_q, nq, d_db, ndb, 0, d_idx, d_dist)
    torch.cuda.synchronize()
    ridx, rdist = oracle.knn2(q, db)
    assert np.array_equal(d_idx.cpu().numpy(), ridx) and np.array_equal(d_dist.cpu().numpy(), rdist)
    sm.close()


def test_failed_configuration_leaves_handle_usable(oracle):
    """A shape the extractor cannot take (aspect ratio > 64:1) must fail every time it is offered — not only the first — and
    the handle must keep working for supported shapes afterwards (ADVICE r1: half-built geometry with geom_valid set)."""
    ex = orbx.ORBextractor(500, 1.2, 4, 20, 7)
    good = synth.image(3, 320, 240)
    nm0, k0, d0 = ex(good)
    bad = synth.image(4, 4000, 70)
    for _ in range(3):
        with pytest.raises(OrbxError):
            ex(bad)
        with pytest.raises(OrbxError):
            ex.pyramid_level(0)                    # nothing is probe-able after a failed call
    nm1, k1, d1 = ex(good)
    assert nm1 == nm0 and k1.tobytes() == k0.tobytes() and np.array_equal(d1, d0)


def test_distribute_octree_rejects_duplicate_pixels():
    xs = np.array([10, 50, 10, 70], np.int32); ys = np.array([20, 30, 20, 90], np.int32); sc = np.array([30, 40, 50, 60], np.int32)
    with pytest.raises(OrbxError):
        orbx.distribute_octree(xs, ys, sc, 0, 200, 0, 100, 10)


def test_single_frame_forked_graph_equals_serial(oracle, monkeypatch):
    """The per-level fork/join graph of orbx_extract against the serial launch order (profiling forces the serial path) on the
    same handle, several frames and shapes (graph re-capture on a shape change)."""
    ex = orbx.ORBextractor(1000, 1.2, 8, 20, 7)
    for (cols, rows, seed) in [(752, 480, 1), (752, 480, 2), (640, 480, 3), (752, 480, 4), (752, 480, 5)]:
        img = synth.image(seed, cols, rows)
        r1 = ex(img)
        ex.profile_begin()
        r2 = ex(img)
        ex.profile_end()
        r3 = ex(img)
        for r in (r2, r3):
            assert r[0] == r1[0] and r[1].tobytes() == r1[1].tobytes() and np.array_equal(r[2], r1[2])
        oex = oracle.extractor(1000, 1.2, 8, 20, 7)
        ok, od, onm = oex.extract(img, (0, 0))
        assert r1[0] == onm and np.array_equal(r1[1]["x"], ok["x"]) and np.array_equal(r1[1]["y"], ok["y"]) and np.array_equal(r1[2], od)


def test_pyramid_host_mirror_equals_probe(oracle):
    """mvImagePyramid without blocking copies: the pinned host mirror filled during orbx_extract equals the probe copies and
    the oracle pyramid, level by level with borders, across calls (graph replay) and a shape change."""
    ex = orbx.ORBextractor(1000, 1.2, 8, 20, 7)
    ex.set_pyramid_mirror(True)
    plain = orbx.ORBextractor(1000, 1.2, 8, 20, 7)
    for (cols, rows, seed) in [(752, 480, 11), (752, 480, 12), (640, 360, 13), (752, 480, 14)]:
        img = synth.image(seed, cols, rows)
        r1 = ex(img); r0 = plain(img)
        assert r1[0] == r0[0] and r1[1].tobytes() == r0[1].tobytes() and np.array_equal(r1[2], r0[2])
        oex = oracle.extractor(1000, 1.2, 8, 20, 7)
        oex.extract(img, (0, 0))
        for level in range(8):
            m = ex.pyramid_mirror(level, with_border=True)
            assert np.array_equal(m, ex.pyramid_level(level, with_border=True)), level
            assert np.array_equal(m, oex.pyramid_level(level, with_border=True)), level
            assert np.array_equal(ex.pyramid_mirror(level), plain.pyramid_level(level))
    ex.set_pyramid_mirror(False)
    ex(synth.image(15, 752, 480))


def test_reference_frame_call_site_against_the_adapter():
    """The reference's own call site — src/Frame.cc:111-127 (stereo Frame constructor: accessor block + the two ExtractORB
    threads) and 420-455 (extractorParenthesis, Frame::ExtractORB) — compiled UNCHANGED against csrc/adapter/ORBextractor.h
    (oracle/build_ref.sh slices it at build time from the checkout named by ORB_REFERENCE_ROOT) must fill mvKeys / mDescriptors /
    mvKeysRight / mDescriptorsRight / monoLeft / monoRight and the scale tables exactly as the C ABI does."""
    import math
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "oracle", "_ref", "frame_callsite_test")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/frame_callsite_test not built (needs ORB_REFERENCE_ROOT at build time)")
    out = subprocess.check_output([exe, "31", "1200"], text=True)
    lines = [ln for ln in out.splitlines() if ln.startswith("rep=")]
    assert len(lines) == 2, out

    def fnv(h, data):
        for b in bytes(data):
            h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
        return h
    L, R = synth.image(31, 752, 480, view=0, max_disp=40), synth.image(31, 752, 480, view=1, max_disp=40)
    exL = orbx.ORBextractor(1200, 1.2, 8, 20, 7); exR = orbx.ORBextractor(1200, 1.2, 8, 20, 7)
    nmL, kL, dL = exL(L, None, (0, 0)); nmR, kR, dR = exR(R, None, (0, 0))
    hl = fnv(fnv(1469598103934665603, kL.tobytes()), dL.tobytes())
    hr = fnv(fnv(1469598103934665603, kR.tobytes()), dR.tobytes())
    ht = 1469598103934665603
    for t in (exL.GetScaleFactors(), exL.GetInverseScaleFactors(), exL.GetScaleSigmaSquares(), exL.GetInverseScaleSigmaSquares()):
        ht = fnv(ht, np.asarray(t, np.float32).tobytes())
    for ln in lines:
        m = re.search(r"N=(\d+) Nright=(\d+) monoLeft=(-?\d+) monoRight=(-?\d+) levels=(\d+) scale=([\d.]+) logscale=([\d.]+) left=([0-9a-f]+) "
                      r"right=([0-9a-f]+) tables=([0-9a-f]+)", ln)
        assert m, ln
        assert int(m.group(1)) == len(kL) and int(m.group(2)) == len(kR) and int(m.group(3)) == nmL and int(m.group(4)) == nmR
        assert int(m.group(5)) == 8 and abs(float(m.group(6)) - 1.2000000477) < 1e-7
        assert abs(float(m.group(7)) - math.log(np.float32(1.2))) < 1e-6
        assert m.group(8) == "%016x" % hl and m.group(9) == "%016x" % hr and m.group(10) == "%016x" % ht


def test_batched_distinctive_descriptors_vs_oracle_and_reference(oracle, request):
    """orbx_distinctive_descriptors (one warp per map point) against the oracle's restatement and the reference's own compiled
    core of MapPoint::ComputeDistinctiveDescriptors (src/MapPoint.cc:368-397) — live where libref.so is built, else its stored
    answers: ties between medians (first row wins), N = 1, N = 2, empty points, N up to 64 on the GPU and beyond (host path)."""
    rng = np.random.default_rng(5)
    counts = [0, 1, 2, 3, 5, 8, 13, 33, 64, 65, 100, 0, 7] + [int(x) for x in rng.integers(1, 40, 300)]
    descs, offsets = [], [0]
    for n in counts:
        base = synth.descriptors(1000 + len(offsets), max(n, 1))[:n].copy()
        if n >= 4:                                     # near-duplicates and exact duplicates: equal medians
            base[1] = base[0]
            base[3] = base[2]; base[3, 0] ^= 1
        descs.append(base)
        offsets.append(offsets[-1] + n)
    allD = np.concatenate(descs) if offsets[-1] else np.zeros((0, 32), np.uint8)
    best = orbx.distinctive_descriptors(allD, np.array(offsets, np.int32))
    from tests import ref_lib
    ref = ref_lib.load() if ref_lib.available() else None
    got, want = [], []
    for p, n in enumerate(counts):
        if n == 0:
            assert best[p] == -1
            continue
        exp = oracle.distinctive_descriptor(descs[p])
        assert best[p] == exp, (p, n, best[p], exp)
        assert orbx.distinctive_descriptor(descs[p]) == exp
        if p < 40:
            got.append(exp)
            if ref:
                want.append(ref.distinctive_descriptor(descs[p]))
    ref_lib.Pin(request.node.name)("reference", [np.array(got, np.int32)], ref and [np.array(want, np.int32)])


def test_left_right_extractors_on_two_host_threads(oracle):
    """The reference runs the left and the right extractor on two std::threads (src/Frame.cc:124-127): two handles, two host
    threads, 150 frames each through the captured forked graph, different shapes per side, every result equal to the
    single-threaded answer of a third handle (and a sample to the oracle)."""
    shapes = [(752, 480, 1200), (640, 400, 900)]
    frames = [[synth.image(100 * t + i, c, r) for i in range(6)] for t, (c, r, _) in enumerate(shapes)]
    want = []
    for t, (c, r, nf) in enumerate(shapes):
        ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
        want.append([ex(im, None, (0, 1000) if t else (0, 0)) for im in frames[t]])
    errors = []

    def worker(t):
        try:
            c, r, nf = shapes[t]
            ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
            for it in range(150):
                k = it % 6
                nm, kp, d = ex(frames[t][k], None, (0, 1000) if t else (0, 0))
                w = want[t][k]
                if nm != w[0] or kp.tobytes() != w[1].tobytes() or not np.array_equal(d, w[2]):
                    errors.append((t, it))
                    return
        except Exception as e:          # noqa: BLE001
            errors.append((t, repr(e)))

    ths = [threading.Thread(target=worker, args=(t,)) for t in range(2)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    assert not errors, errors
    oex = oracle.extractor(1200, 1.2, 8, 20, 7)
    ok, od, onm = oex.extract(frames[0][0], (0, 0))
    assert want[0][0][0] == onm and np.array_equal(want[0][0][1]["x"], ok["x"]) and np.array_equal(want[0][0][2], od)


@pytest.mark.parametrize("lapping", [(0, 1000), (300, 500), (0, 0)])
def test_lapping_area_in_batches_and_single_frames_agree(oracle, lapping):
    """The packing is fused into the descriptor kernel for a few frames when the lapping area decides the row (all / none) and
    is a separate kernel otherwise and for batches: the three paths must agree with each other and with the oracle."""
    imgs = np.stack([synth.image(300 + f, 752, 480) for f in range(9)])
    single = orbx.ORBextractor(1000, 1.2, 8, 20, 7)
    batch = orbx.ORBextractor(1000, 1.2, 8, 20, 7)
    nm, n, kps, desc = batch.extract_batch(imgs, lapping)
    oex = oracle.extractor(1000, 1.2, 8, 20, 7)
    for f in range(9):
        m1, k1, d1 = single(imgs[f], None, lapping)
        assert int(nm[f]) == m1 and int(n[f]) == len(k1)
        assert kps[f, :n[f]].tobytes() == k1.tobytes() and np.array_equal(desc[f, :n[f]], d1)
        if f < 2:
            ok, od, onm = oex.extract(imgs[f], lapping)
            assert m1 == onm and np.array_equal(k1["x"], ok["x"]) and np.array_equal(k1["y"], ok["y"]) and np.array_equal(d1, od)


@pytest.mark.parametrize("cols,rows,nlevels,scale", [(752, 480, 8, 1.2), (1241, 376, 8, 1.2), (640, 480, 5, 1.44), (333, 211, 6, 1.3),
                                                     (1300, 100, 4, 1.2), (97, 83, 3, 1.15), (520, 390, 4, 1.5)])
def test_batch_pyramid_streaming_kernel_is_bit_exact(oracle, cols, rows, nlevels, scale):
    """ComputePyramid on batches (src/ORBextractor.cc:1309-1329) takes the warp-streaming resize kernel (bordered items, IDP.2A
    horizontal pass): every byte of every bordered level of every frame equals the oracle's, and a single frame (tiled kernel)
    gives the same bytes."""
    F = 9
    imgs = np.stack([synth.image(500 + f, cols, rows) for f in range(F)])
    ex = orbx.ORBextractor(300, scale, nlevels, 20, 7, max_batch=F)
    ex.extract_batch(imgs)
    got = [[ex.pyramid_level(l, frame=f, with_border=True) for l in range(nlevels)] for f in (0, 4, F - 1)]
    for k, f in enumerate((0, 4, F - 1)):
        oex = oracle.extractor(300, scale, nlevels, 20, 7)
        oex.extract(imgs[f], (0, 0))
        for l in range(nlevels):
            want = oex.pyramid_level(l, with_border=True)
            assert got[k][l].shape == want.shape
            assert np.array_equal(got[k][l], want), (f, l, np.argwhere(got[k][l] != want)[:4])
    ex(imgs[4])
    for l in range(nlevels):
        assert np.array_equal(ex.pyramid_level(l, with_border=True), got[1][l]), l


def test_tiled_pyramid_kernel_matches_streaming_kernel():
    """ORBX_PYR_PIPE=0 selects the tiled resize kernel (the fallback of the streaming one, e.g. without tensor maps): a child
    process with the switch set must produce the same bordered pyramid bytes as this process (streaming kernel, compared with
    the oracle in the tests above)."""
    import hashlib, os, subprocess, sys
    code = ("import hashlib, numpy as np, wut_cuda_orb_slam3_b200 as orbx\n"
            "from wut_cuda_orb_slam3_b200 import synth\n"
            "h = hashlib.sha1()\n"
            "for cols, rows, scale in ((752, 480, 1.2), (333, 211, 1.3)):\n"
            "    ex = orbx.ORBextractor(500, scale, 6, 20, 7)\n"
            "    ex(synth.image(77, cols, rows))\n"
            "    for l in range(6): h.update(ex.pyramid_level(l, with_border=True).tobytes())\n"
            "print(h.hexdigest())\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    digests = []
    for v in ("0", "1"):
        env = dict(os.environ, ORBX_PYR_PIPE=v, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
        digests.append(subprocess.check_output([sys.executable, "-c", code], env=env, text=True, cwd=root).strip().splitlines()[-1])
    assert digests[0] == digests[1]
