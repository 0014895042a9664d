"""CPU: rcc_ba_covariance_blocks rejects a missing handle before it touches a device."""
import numpy as np

from robot_camera_calibration_b200 import _lib


def test_null_handle_is_rejected():
    lib = _lib.load()
    pairs = np.array([_lib.BLOCK_VIEW, 0, _lib.BLOCK_MARKER, 1], np.int32)
    out = np.zeros(36)
    assert lib.rcc_ba_covariance_blocks(None, 1, pairs.ctypes.data_as(_lib.c_int32_p),
                                        out.ctypes.data_as(_lib.c_double_p)) == _lib.RCC_BAD_ARG
    assert lib.rcc_ba_covariance_blocks(None, 0, None, None) == _lib.RCC_BAD_ARG
