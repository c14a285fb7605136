"""The blur of batched extraction (>= 8 frames per call with tensor maps: blur_mma_kernel, int8 MMAs on the tensor cores) against
the oracle's 7x7 Gaussian, byte for byte, on every frame and level.  The other blur comparisons extract single frames, which take
blur_kernel.  Contents that stress the integer ranges and the tile edges: synthetic scenes, all-255 frames (largest sums), noise
and checkerboards, at the configs' shapes (1241 px rows are not 16-byte aligned) and at one small shape whose level sizes are not
multiples of 16."""
import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from wut_cuda_orb_slam3_b200 import synth

pytestmark = pytest.mark.gpu

SHAPES = [(752, 480), (1241, 376), (1280, 720), (234, 170)]


def frames(cols, rows, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:rows, 0:cols]
    out = [synth.image(seed + f, cols, rows) for f in range(4)]
    out += [np.full((rows, cols), 255, np.uint8)] * 2
    out += [rng.integers(0, 256, (rows, cols), dtype=np.uint8) for _ in range(2)]
    out += [(((xx + yy) & 1) * 255).astype(np.uint8), ((((xx // 3) + (yy // 5)) & 1) * 255).astype(np.uint8)]
    return np.stack(out)


@pytest.mark.parametrize("cols,rows", SHAPES)
def test_batch_blur_matches_oracle(oracle, cols, rows):
    imgs = frames(cols, rows, 300 + cols)
    ex = orbx.ORBextractor(1000, 1.2, 8, 20, 7)
    ex.extract_batch(imgs, (0, 0))
    if cols == 234:
        sizes = [ex.level_size(cols, rows, level) for level in range(8)]
        assert all(w % 16 and h % 16 for w, h in sizes), sizes
    # the oracle's blur of the GPU's own pyramid level is the reference's blurred level (the pyramid is checked elsewhere) ...
    oex = oracle.extractor(1000, 1.2, 8, 20, 7)
    oex.extract(imgs[0], (0, 0))
    for level in range(8):
        assert np.array_equal(oracle.blur(ex.pyramid_level(level, frame=0)), oex.blurred_level(level)), level
    # ... and the batch kernel's output must equal it everywhere
    for f in range(len(imgs)):
        for level in range(8):
            ref = oracle.blur(ex.pyramid_level(level, frame=f))
            got = ex.blurred_level(level, frame=f)
            assert np.array_equal(got, ref), (f, level, int((got != ref).sum()))
