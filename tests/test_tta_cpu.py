"""CPU checks of test-time augmentation's host side: the view list predict_mask builds from (scales, flip), its
validation, and the ctypes mirror of IswmTtaView."""
import ctypes

import pytest

from iswm_b200 import _lib
from iswm_b200.predict import _tta_views


def test_views_in_order_with_rounded_sizes():
    assert _tta_views((0.75, 1.0, 1.25), True, 200, 232) == [
        (0.75, (150, 174), False), (0.75, (150, 174), True), (1.0, (200, 232), False), (1.0, (200, 232), True),
        (1.25, (250, 290), False), (1.25, (250, 290), True)]
    assert _tta_views([0.5, 2], False, 37, 53) == [(0.5, (19, 27), False), (2.0, (74, 106), False)]
    assert len(_tta_views((0.5, 0.75, 1.0, 1.25), True, 64, 64)) == 8


@pytest.mark.parametrize("scales,flip", [((), False), ((0.0,), False), ((-0.5,), True), ((float("nan"),), False),
                                         ((float("inf"),), False), ((0.24,), False), ((0.5, 0.75, 1.0, 1.25, 1.5), True),
                                         ((1.0,) * 9, False)])
def test_bad_requests_raise(scales, flip):
    with pytest.raises(ValueError):
        _tta_views(scales, flip, 64, 64)


def test_view_record_matches_the_header_layout():
    assert ctypes.sizeof(_lib.TtaView) == 32 and _lib.TtaView.Hi.offset == 8 and _lib.TtaView.flip.offset == 24
