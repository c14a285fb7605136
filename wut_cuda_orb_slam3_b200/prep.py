"""Host mirror of the preparation steps either side of the extractor (SURVEY.md §8(f)3) over the C ABI:
Frame::UndistortKeyPoints (src/Frame.cc:777-810), the stereo rectification of System::TrackStereo (src/System.cc:253-260) and
the RGB-D Frame constructor (src/Frame.cc:202-260, with Tracking::GrabImageRGBD's conversions).  GPU only; no CPU fallback."""
import ctypes as C

import numpy as np

from .capi import KP_DTYPE, RgbdCalibC, check, lib, ptr

DEPTH_TYPES = {np.dtype(np.uint16): 0, np.dtype(np.float32): 1}      # CV_16U, CV_32F


def undistort_keypoints(keypoints, K, dist, new_K=None, device=0):
    """K / new_K = (fx, fy, cx, cy); dist = mDistCoef (4, 5, 8 or 12 floats).  Returns mvKeysUn."""
    kps = np.ascontiguousarray(keypoints, KP_DTYPE)
    K = np.ascontiguousarray(K, np.float32)
    P = K if new_K is None else np.ascontiguousarray(new_K, np.float32)
    d = np.ascontiguousarray(dist, np.float32)
    out = np.zeros_like(kps)
    check(lib().orbx_undistort_keypoints(device, ptr(kps), len(kps), ptr(K), ptr(d), len(d), ptr(P), ptr(out)))
    return out


def rgbd_calib(K, dist, bf, depth_factor):
    """orbx_rgbd_calib from K = (fx, fy, cx, cy), dist = mDistCoef (0, 4, 5, 8 or 12 floats), mbf and mDepthMapFactor.  Returns
    (struct, coefficient array); keep the array alive while the struct is in use."""
    d = np.ascontiguousarray(dist if dist is not None else [], np.float32)
    c = RgbdCalibC()
    c.K[:] = [float(v) for v in np.asarray(K, np.float32)]
    c.dist = d.ctypes.data if len(d) else None
    c.n_dist = len(d)
    c.bf = float(bf)
    c.depth_factor = float(depth_factor)
    return c, d


def _depth_type(depth):
    if depth.dtype not in DEPTH_TYPES:
        raise TypeError("depth map must be uint16 (CV_16U) or float32 (CV_32F), got %s" % depth.dtype)
    return DEPTH_TYPES[depth.dtype]


def extract_rgbd(ex, image, depth, K, dist, bf, depth_factor, rgb=True):
    """The RGB-D Frame constructor in one call (src/Frame.cc:202-260): image HxW grey or HxWx3 / HxWx4 colour (rgb = mbRGB),
    depth the RAW HxW map (uint16 or float32) and depth_factor = mDepthMapFactor, applied as Tracking::GrabImageRGBD does.
    Returns (mvKeys, mvKeysUn, descriptors, mvuRight, mvDepth)."""
    image = np.asarray(image, np.uint8)
    if image.ndim == 3 and (image.strides[2] != 1 or image.strides[1] != image.shape[2]):
        image = np.ascontiguousarray(image)
    if image.ndim == 2 and image.strides[1] != 1:
        image = np.ascontiguousarray(image)
    rows, cols = image.shape[:2]
    ch = image.shape[2] if image.ndim == 3 else 1
    depth = np.asarray(depth)
    if depth.strides[1] != depth.itemsize:
        depth = np.ascontiguousarray(depth)
    assert depth.shape == (rows, cols), (depth.shape, image.shape)
    calib, _keep = rgbd_calib(K, dist, bf, depth_factor)
    cap = ex.max_keypoints(rows, cols)
    kp = np.zeros(cap, KP_DTYPE); kp_un = np.zeros(cap, KP_DTYPE); desc = np.zeros((cap, 32), np.uint8)
    u = np.full(cap, -1.0, np.float32); z = np.full(cap, -1.0, np.float32)
    n = C.c_int(0)
    check(lib().orbx_extract_rgbd(ex._h, ptr(image), rows, cols, image.strides[0], ch, int(bool(rgb)), ptr(depth), _depth_type(depth),
                                  depth.strides[0], C.byref(calib), ptr(kp), ptr(kp_un), ptr(desc), cap, C.byref(n), ptr(u), ptr(z)))
    ex._shape = (rows, cols)
    k = n.value
    return kp[:k].copy(), kp_un[:k].copy(), desc[:k].copy(), u[:k].copy(), z[:k].copy()


class Rectifier:
    """cv::remap(im, out, M1, M2, INTER_LINEAR) with fixed CV_32FC1 maps (cv::initUndistortRectifyMap), maps kept on the device."""

    def __init__(self, map_x=None, map_y=None, device=0, resize=None):
        """resize=(src_rows, src_cols, dst_rows, dst_cols) builds the cv::resize(im, out, newImSize) variant instead."""
        self.device = device
        if resize is not None:
            sr, sc, dr, dc = resize
            self.shape = (dr, dc)
            h = C.c_void_p()
            check(lib().orbx_resizer_create(device, sr, sc, dr, dc, C.byref(h)))
            self._h = h
            return
        mx = np.ascontiguousarray(map_x, np.float32); my = np.ascontiguousarray(map_y, np.float32)
        assert mx.shape == my.shape and mx.ndim == 2
        self.shape = mx.shape
        self.device = device
        h = C.c_void_p()
        check(lib().orbx_rectifier_create(device, ptr(mx), ptr(my), mx.strides[0], mx.shape[0], mx.shape[1], C.byref(h)))
        self._h = h

    def remap(self, image):
        img = np.ascontiguousarray(image, np.uint8)
        out = np.zeros(self.shape, np.uint8)
        check(lib().orbx_remap(self._h, ptr(img), img.shape[0], img.shape[1], img.strides[0], ptr(out), out.strides[0]))
        return out

    def remap_device(self, d_src, src_rows, src_cols, src_pitch, src_frame_stride, n_frames, d_dst, dst_pitch, dst_frame_stride, stream=None):
        check(lib().orbx_remap_device(self._h, ptr(d_src), src_rows, src_cols, src_pitch, src_frame_stride, n_frames, ptr(d_dst), dst_pitch,
                                      dst_frame_stride, ptr(stream) if stream is not None else None))

    def close(self):
        if self._h:
            lib().orbx_rectifier_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
