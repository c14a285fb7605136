"""Python mirror of ORB_SLAM3::ORBextractor (reference include/ORBextractor.h:52-120) over the C ABI.

Names and argument meaning follow the reference class: ORBextractor(nfeatures, scaleFactor, nlevels, iniThFAST,
minThFAST); operator() -> __call__(image, mask, vLappingArea) returning (monoIndex, keypoints, descriptors);
GetLevels / GetScaleFactor / GetScaleFactors / GetInverseScaleFactors / GetScaleSigmaSquares /
GetInverseScaleSigmaSquares; mvImagePyramid (lazy device->host copies).
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import KP_DTYPE, check, lib, ptr


class ORBextractor:
    HARRIS_SCORE = 0
    FAST_SCORE = 1

    def __init__(self, nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST, device=0, max_cols=0, max_rows=0, max_batch=0):
        self._h = C.c_void_p()
        check(lib().orbx_create(int(nfeatures), float(scaleFactor), int(nlevels), int(iniThFAST), int(minThFAST), int(device),
                                int(max_cols), int(max_rows), int(max_batch), C.byref(self._h)))
        self.nfeatures, self.nlevels, self.device = int(nfeatures), int(nlevels), int(device)
        self._shape = None

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().orbx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- accessors (include/ORBextractor.h:70-90) -------------------------------------------------------------
    def GetLevels(self):
        return lib().orbx_get_levels(self._h)

    def GetScaleFactor(self):
        return lib().orbx_get_scale_factor(self._h)

    def _tables(self):
        n = self.nlevels
        out = [np.zeros(n, np.float32) for _ in range(4)] + [np.zeros(n, np.int32)]
        check(lib().orbx_get_tables(self._h, *[ptr(a) for a in out]))
        return out

    def GetScaleFactors(self):
        return self._tables()[0]

    def GetInverseScaleFactors(self):
        return self._tables()[1]

    def GetScaleSigmaSquares(self):
        return self._tables()[2]

    def GetInverseScaleSigmaSquares(self):
        return self._tables()[3]

    def GetFeaturesPerLevel(self):
        return self._tables()[4]

    def max_keypoints(self, rows=None, cols=None):
        """Upper bound on keypoints per frame; pass the image shape (the bound depends on nIni = round(width / height) of
        DistributeOctTree, src/ORBextractor.cc:589, which a handle that has not seen an image yet cannot know)."""
        if rows is not None and cols is not None:
            return lib().orbx_max_keypoints_for(self._h, int(rows), int(cols))
        return lib().orbx_max_keypoints(self._h)

    def level_size(self, cols, rows, level):
        w, h = C.c_int(0), C.c_int(0)
        check(lib().orbx_level_size(self._h, cols, rows, level, C.byref(w), C.byref(h)))
        return w.value, h.value

    # ---- operator() (src/ORBextractor.cc:1227-1307) -----------------------------------------------------------
    def __call__(self, image, mask=None, vLappingArea=(0, 0)):
        """image: HxW uint8 numpy array (host).  Returns (monoIndex, keypoints[KP_DTYPE], descriptors[N,32]);
        monoIndex is -1 for an empty image, exactly like the reference."""
        if image is None or image.size == 0:
            return -1, np.zeros(0, KP_DTYPE), np.zeros((0, 32), np.uint8)
        if image.ndim == 3:
            return self.extract_color(image, True, vLappingArea)
        assert image.dtype == np.uint8 and image.ndim == 2, "CV_8UC1 expected (src/ORBextractor.cc:1235)"
        if image.strides[1] != 1:
            image = np.ascontiguousarray(image)
        rows, cols = image.shape
        cap = self.max_keypoints(rows, cols)
        kps = np.zeros(cap, KP_DTYPE)
        desc = np.zeros((cap, 32), np.uint8)
        n, nm = C.c_int(0), C.c_int(0)
        check(lib().orbx_extract(self._h, ptr(image), rows, cols, image.strides[0], int(vLappingArea[0]), int(vLappingArea[1]),
                                 ptr(kps), ptr(desc), cap, C.byref(n), C.byref(nm)))
        self._shape = (rows, cols)
        return nm.value, kps[:n.value].copy(), desc[:n.value].copy()

    def extract_color(self, image, rgb=True, vLappingArea=(0, 0)):
        """Tracking::GrabImage* + operator(): HxWx3 / HxWx4 uint8 image, rgb = mbRGB (channel 0 is red); the cvtColor to grey
        (src/Tracking2.cc:289-316) runs on the device in front of the pyramid."""
        assert image.dtype == np.uint8 and image.ndim == 3 and image.shape[2] in (3, 4)
        if image.strides[2] != 1 or image.strides[1] != image.shape[2]:
            image = np.ascontiguousarray(image)
        rows, cols, ch = image.shape
        cap = self.max_keypoints(rows, cols)
        kps = np.zeros(cap, KP_DTYPE)
        desc = np.zeros((cap, 32), np.uint8)
        n, nm = C.c_int(0), C.c_int(0)
        check(lib().orbx_extract_color(self._h, ptr(image), rows, cols, image.strides[0], ch, int(bool(rgb)), int(vLappingArea[0]),
                                       int(vLappingArea[1]), ptr(kps), ptr(desc), cap, C.byref(n), C.byref(nm)))
        self._shape = (rows, cols)
        return nm.value, kps[:n.value].copy(), desc[:n.value].copy()

    def extract_batch(self, images, vLappingArea=(0, 0)):
        """images: [F,H,W] uint8 numpy array (host, ideally page-locked).  Returns (n_mono[F], n[F], kps[F,cap], desc[F,cap,32])."""
        assert images.dtype == np.uint8 and images.ndim == 3 and images.strides[2] == 1
        F, rows, cols = images.shape
        cap = self.max_keypoints(rows, cols)
        kps = np.zeros((F, cap), KP_DTYPE)
        desc = np.zeros((F, cap, 32), np.uint8)
        n = np.zeros(F, np.int32)
        nm = np.zeros(F, np.int32)
        ptrs = (C.c_void_p * F)(*[images.ctypes.data + f * images.strides[0] for f in range(F)])
        check(lib().orbx_extract_batch(self._h, ptrs, F, rows, cols, images.strides[1], int(vLappingArea[0]), int(vLappingArea[1]),
                                       ptr(kps), ptr(desc), cap, ptr(n), ptr(nm)))
        self._shape = (rows, cols)
        return nm, n, kps, desc

    def extract_batch_device(self, d_images, n_frames, rows, cols, pitch, frame_stride, d_kps, d_desc, capacity, d_n, d_nm,
                             vLappingArea=(0, 0), stream=None):
        """Device-resident batch: every argument named d_* is a device pointer (int) or a torch CUDA tensor."""
        check(lib().orbx_extract_batch_device(self._h, ptr(d_images), frame_stride, n_frames, rows, cols, pitch, int(vLappingArea[0]),
                                              int(vLappingArea[1]), ptr(d_kps), ptr(d_desc), capacity, ptr(d_n), ptr(d_nm),
                                              ptr(stream) if stream else None))
        self._shape = (rows, cols)

    def extract_stereo_batch(self, left, right, bf, maxD):
        """The stereo Frame constructor (src/Frame.cc:124-143) over N rectified pairs on this one handle: left / right are [N,H,W]
        uint8 numpy arrays (host, ideally page-locked).  Returns (nL[N], nR[N], kpL[N,cap], descL[N,cap,32], kpR[N,cap],
        descR[N,cap,32], uRight[N,cap], depth[N,cap]); rows of pair i past nL[i] / nR[i] are undefined."""
        assert left.dtype == np.uint8 and right.dtype == np.uint8 and left.ndim == 3 and left.shape == right.shape
        assert left.strides == right.strides and left.strides[2] == 1
        N, rows, cols = left.shape
        cap = self.max_keypoints(rows, cols)
        kL = np.zeros((N, cap), KP_DTYPE); kR = np.zeros((N, cap), KP_DTYPE)
        dL = np.zeros((N, cap, 32), np.uint8); dR = np.zeros((N, cap, 32), np.uint8)
        u = np.full((N, cap), -1.0, np.float32); d = np.full((N, cap), -1.0, np.float32)
        nL = np.zeros(N, np.int32); nR = np.zeros(N, np.int32)
        pl = (C.c_void_p * max(N, 1))(*[left.ctypes.data + i * left.strides[0] for i in range(N)])
        pr = (C.c_void_p * max(N, 1))(*[right.ctypes.data + i * right.strides[0] for i in range(N)])
        check(lib().orbx_extract_stereo_batch(self._h, pl, pr, N, rows, cols, left.strides[1], float(bf), float(maxD), ptr(kL), ptr(dL),
                                              ptr(nL), ptr(kR), ptr(dR), ptr(nR), cap, ptr(u), ptr(d)))
        self._shape = (rows, cols)
        return nL, nR, kL, dL, kR, dR, u, d

    def extract_stereo_batch_device(self, d_left, d_right, n_pairs, rows, cols, pitch, frame_stride, bf, maxD, d_kpL, d_descL, d_nL,
                                    d_kpR, d_descR, d_nR, capacity, d_uRight, d_depth, stream=None):
        """Device-resident stereo batch: every argument named d_* is a device pointer (int) or a torch CUDA tensor; the outputs are
        [n_pairs][capacity] slabs (counts [n_pairs])."""
        check(lib().orbx_extract_stereo_batch_device(self._h, ptr(d_left), ptr(d_right), frame_stride, n_pairs, rows, cols, pitch,
                                                     float(bf), float(maxD), ptr(d_kpL), ptr(d_descL), ptr(d_nL), ptr(d_kpR), ptr(d_descR),
                                                     ptr(d_nR), capacity, ptr(d_uRight), ptr(d_depth), ptr(stream) if stream else None))
        self._shape = (rows, cols)

    def extract_rgbd_batch(self, images, depths, K, dist, bf, depth_factor):
        """The RGB-D Frame constructor (src/Frame.cc:202-260) over N frames on this handle: images [N,H,W] uint8 grey, depths the
        RAW [N,H,W] uint16 or float32 maps (host, ideally page-locked), depth_factor = mDepthMapFactor.  Returns (n[N], kp[N,cap],
        kp_un[N,cap], desc[N,cap,32], uRight[N,cap], depth[N,cap]); rows of frame i past n[i] are undefined."""
        from .prep import _depth_type, rgbd_calib
        assert images.dtype == np.uint8 and images.ndim == 3 and images.strides[2] == 1
        assert depths.ndim == 3 and depths.shape == images.shape and depths.strides[2] == depths.itemsize
        N, rows, cols = images.shape
        calib, _keep = rgbd_calib(K, dist, bf, depth_factor)
        cap = self.max_keypoints(rows, cols)
        kp = np.zeros((N, cap), KP_DTYPE); kp_un = np.zeros((N, cap), KP_DTYPE); desc = np.zeros((N, cap, 32), np.uint8)
        u = np.full((N, cap), -1.0, np.float32); z = np.full((N, cap), -1.0, np.float32)
        n = np.zeros(N, np.int32)
        pi = (C.c_void_p * max(N, 1))(*[images.ctypes.data + i * images.strides[0] for i in range(N)])
        pd = (C.c_void_p * max(N, 1))(*[depths.ctypes.data + i * depths.strides[0] for i in range(N)])
        check(lib().orbx_extract_rgbd_batch(self._h, pi, pd, N, rows, cols, images.strides[1], _depth_type(depths), depths.strides[1],
                                            C.byref(calib), ptr(kp), ptr(kp_un), ptr(desc), cap, ptr(n), ptr(u), ptr(z)))
        self._shape = (rows, cols)
        return n, kp, kp_un, desc, u, z

    def extract_rgbd_batch_device(self, d_images, d_depths, n_frames, rows, cols, pitch, frame_stride, depth_type, depth_pitch,
                                  depth_frame_stride, K, dist, bf, depth_factor, d_kp, d_kp_un, d_desc, capacity, d_n, d_uRight, d_depth,
                                  stream=None):
        """Device-resident RGB-D batch: every argument named d_* is a device pointer (int) or a torch CUDA tensor; depth_type 0 =
        uint16, 1 = float32; the outputs are [n_frames][capacity] slabs (counts [n_frames])."""
        from .prep import rgbd_calib
        calib, _keep = rgbd_calib(K, dist, bf, depth_factor)
        check(lib().orbx_extract_rgbd_batch_device(self._h, ptr(d_images), frame_stride, pitch, ptr(d_depths), depth_frame_stride,
                                                   depth_pitch, int(depth_type), n_frames, rows, cols, C.byref(calib), ptr(d_kp),
                                                   ptr(d_kp_un), ptr(d_desc), capacity, ptr(d_n), ptr(d_uRight), ptr(d_depth),
                                                   ptr(stream) if stream else None))
        self._shape = (rows, cols)

    def sync(self):
        check(lib().orbx_sync(self._h))

    STAGES = ("pyramid", "fast", "blur", "octree", "orient_describe", "pack")

    def profile_begin(self):
        check(lib().orbx_profile_begin(self._h))

    def profile_end(self):
        """Returns ({stage: summed milliseconds}, n_chunks) measured with CUDA events on the launching stream."""
        ms = np.zeros(len(self.STAGES), np.float32)
        n = C.c_int(0)
        check(lib().orbx_profile_end(self._h, ptr(ms), C.byref(n)))
        return dict(zip(self.STAGES, ms.tolist())), n.value

    # ---- mvImagePyramid (include/ORBextractor.h:92) and stage probes -----------------------------------------
    @property
    def mvImagePyramid(self):
        return [self.pyramid_level(l) for l in range(self.nlevels)]

    def pyramid_level(self, level, frame=0, with_border=False):
        rows, cols = self._shape
        w, h = self.level_size(cols, rows, level)
        b = 38 if with_border else 0
        out = np.zeros((h + b, w + b), np.uint8)
        check(lib().orbx_get_pyramid_level(self._h, frame, level, ptr(out), out.strides[0], int(with_border)))
        return out

    def set_pyramid_mirror(self, enable=True):
        """Keep a pinned host mirror of the bordered pyramid current (filled on a copy branch during every __call__)."""
        check(lib().orbx_set_pyramid_mirror(self._h, int(enable)))

    def pyramid_mirror(self, level, with_border=False):
        """mvImagePyramid[level] from the host mirror (a copy of the library's pinned storage)."""
        base = C.c_void_p(); step = C.c_size_t(); w = C.c_int(); h = C.c_int()
        check(lib().orbx_get_pyramid_mirror(self._h, level, C.byref(base), C.byref(step), C.byref(w), C.byref(h)))
        bw, bh = w.value + 38, h.value + 38
        buf = np.ctypeslib.as_array(C.cast(base, C.POINTER(C.c_uint8)), shape=(bh * step.value,)).reshape(bh, step.value)[:, :bw]
        return buf.copy() if with_border else buf[19:19 + h.value, 19:19 + w.value].copy()

    def blurred_level(self, level, frame=0):
        rows, cols = self._shape
        w, h = self.level_size(cols, rows, level)
        out = np.zeros((h, w), np.uint8)
        check(lib().orbx_get_blurred_level(self._h, frame, level, ptr(out), out.strides[0]))
        return out

    def candidates(self, level, frame=0):
        rows, cols = self._shape
        w, h = self.level_size(cols, rows, level)
        cap = max((w * h) // 4 + 64, 64)
        xs = np.zeros(cap, np.int32); ys = np.zeros(cap, np.int32); sc = np.zeros(cap, np.int32)
        n = lib().orbx_get_candidates(self._h, frame, level, ptr(xs), ptr(ys), ptr(sc), cap)
        if n < 0:
            check(n)
        return xs[:n].copy(), ys[:n].copy(), sc[:n].copy()

    def level_keypoints(self, level, frame=0):
        cap = self.max_keypoints()
        kps = np.zeros(cap, KP_DTYPE); desc = np.zeros((cap, 32), np.uint8)
        n = lib().orbx_get_level_keypoints(self._h, frame, level, ptr(kps), ptr(desc), cap)
        if n < 0:
            check(n)
        return kps[:n].copy(), desc[:n].copy()


def distribute_octree(xs, ys, scores, minX, maxX, minY, maxY, nFeatures, device=0):
    """ORBextractor::DistributeOctTree (src/ORBextractor.cc:584-774) on the GPU kernel; returns retained input indices."""
    xs = np.ascontiguousarray(xs, np.int32); ys = np.ascontiguousarray(ys, np.int32); scores = np.ascontiguousarray(scores, np.int32)
    cap = max(nFeatures + 8, 4 * 64 + 1)               # max(N + 4, 4 * nIni + 1), nIni <= 64
    out = np.zeros(cap, np.int32)
    n = C.c_int(0)
    check(lib().orbx_distribute_octree(device, ptr(xs), ptr(ys), ptr(scores), len(xs), minX, maxX, minY, maxY, nFeatures, ptr(out), cap,
                                       C.byref(n)))
    return out[:n.value].copy()


def compute_tables(nfeatures, scaleFactor, nlevels):
    out = [np.zeros(nlevels, np.float32) for _ in range(4)] + [np.zeros(nlevels, np.int32)]
    check(lib().orbx_compute_tables(nfeatures, float(scaleFactor), nlevels, *[ptr(a) for a in out]))
    return dict(scale=out[0], inv=out[1], sigma2=out[2], invsigma2=out[3], nfeat=out[4])
