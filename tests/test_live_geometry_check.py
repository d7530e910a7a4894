"""The window / hop validation of live sessions and the lockstep online driver (no GPU needed)."""
import numpy as np
import pytest

from septfa_b200.live import check_geometry


@pytest.mark.parametrize("window,hop", [(48000, 16000), (48000, 8000), (48000, 4000), (32000, 8000), (40000, 12000),
                                        (49152, 4096), (48000, 4800), (512, 256), (160000, 16000),
                                        (np.int64(48000), np.int32(4000))])
def test_check_geometry_accepts(window, hop):
    assert check_geometry(window, hop) == (int(window), int(hop))


@pytest.mark.parametrize("window,hop", [
    (48000, 24016),    # window < 2 hops
    (48000, 240),      # hop < 256
    (48000, 4008),     # hop not a multiple of 16
    (48008, 4000),     # window not a multiple of 16
    (160016, 16000),   # window > 10 s
    (48000.0, 4000),   # not an integer sample count
    (48000, True),
])
def test_check_geometry_refuses(window, hop):
    with pytest.raises(ValueError):
        check_geometry(window, hop)
