"""CPU checks of sliding-window inference's host side: the window placement predict_mask(window=, stride=) builds and
its validation."""
import math

import numpy as np
import pytest

from iswm_b200.predict import _windows


def _coverage(L, w, offs):
    c = np.zeros(L, np.int64)
    for o in offs:
        c[o:o + w] += 1
    return c


@pytest.mark.parametrize("H,W,window,stride", [
    (300, 452, 128, 96), (257, 450, (128, 160), (100, 120)), (512, 512, 128, 128), (500, 500, 128, 32),
    (6144, 6144, 512, 384), (100, 452, 128, 96), (100, 90, 128, 96), (64, 64, 64, 1), (17, 300, (16, 48), (5, 48))])
def test_placement_counts_offsets_and_coverage(H, W, window, stride):
    g = _windows(H, W, window, stride)
    wins = (window, window) if isinstance(window, int) else window
    strides = (stride, stride) if isinstance(stride, int) else stride
    assert g.stride == strides
    for L, win, s, w, offs in ((H, wins[0], strides[0], g.size[0], g.ys), (W, wins[1], strides[1], g.size[1], g.xs)):
        assert w == min(win, L)
        assert len(offs) == math.ceil((L - w) / s) + 1
        assert offs == [min(i * s, L - w) for i in range(len(offs))]
        assert offs[0] == 0 and offs[-1] == L - w                # the last window snapped to the border
        assert all(b > a for a, b in zip(offs, offs[1:]))
        assert all(b - a == s for a, b in zip(offs[:-1], offs[1:-1]))
        c = _coverage(L, w, offs)
        assert c.min() >= 1                                       # every pixel covered
        assert c.max() <= math.ceil(w / s) + 1


def test_examples():
    g = _windows(300, 452, 128, 96)
    assert g.size == (128, 128) and g.ys == [0, 96, 172] and g.xs == [0, 96, 192, 288, 324]
    # s = w / 4: up to 5 windows per axis over a pixel
    g = _windows(512, 512, 128, 32)
    assert len(g.ys) == 13 and _coverage(512, 128, g.ys).max() == 4
    g = _windows(500, 500, 128, 32)
    assert g.ys[-2:] == [352, 372] and _coverage(500, 128, g.ys).max() == 5
    # stride == window tiles the scene; the remainder is a snapped last window
    assert _windows(512, 500, 128, 128).ys == [0, 128, 256, 384] and _windows(512, 500, 128, 128).xs == [0, 128, 256, 372]


def test_scenes_smaller_than_the_window():
    g = _windows(100, 90, 128, 96)                                # both axes: one window, the whole scene
    assert g.size == (100, 90) and g.ys == [0] and g.xs == [0]
    g = _windows(100, 452, 128, 96)                               # one axis
    assert g.size == (100, 128) and g.ys == [0] and g.xs == [0, 96, 192, 288, 324]
    g = _windows(100, 452, (128, 160), (100, 120))                # non-square windows
    assert g.size == (100, 160) and g.xs == [0, 120, 240, 292]


def test_default_stride_is_two_thirds_of_the_window():
    assert _windows(1024, 1024, 256).stride == (170, 170)
    assert _windows(1024, 1024, (512, 96)).stride == (341, 64)
    assert _windows(1024, 1024, 16).stride == (10, 10)


@pytest.mark.parametrize("window,stride", [(15, None), ((16, 15), None), (8, 4), (128, 0), (128, -3), (128, 129),
                                           ((128, 160), (100, 161)), ((128, 160), (0, 10)), ((128, 160, 3), None),
                                           (128, (1, 2, 3)), (128.0, None), (128, 64.0)])
def test_bad_requests_raise(window, stride):
    with pytest.raises(ValueError):
        _windows(300, 300, window, stride)
