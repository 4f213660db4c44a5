"""CPU checks of odg_policy_create_hidden (include/odg_policy.h): widths and dims are validated before the device is looked
at, so these calls fail with ODG_ERR_INVALID on a machine without a GPU as on one with a B200."""
import ctypes as C

import pytest

INVALID = -1


@pytest.mark.parametrize("S,A,h1,h2", [(12, 8, 768, 384), (12, 8, 1024, 256), (12, 8, 256, 256), (12, 8, 512, 512),
                                       (65, 8, 1024, 512), (12, 17, 1024, 512), (0, 8, 1024, 512), (12, 0, 512, 256)])
def test_create_hidden_refuses_unsupported_widths_and_dims(S, A, h1, h2):
    from opendog_b200 import lib
    L = lib.load()
    h = C.c_void_p()
    assert L.odg_policy_create_hidden(S, A, h1, h2, 0, C.byref(h)) == INVALID
    assert b"odg_policy_create" in L.odg_last_error()
    assert h.value is None


def test_create_hidden_refuses_a_null_handle_pointer():
    from opendog_b200 import lib
    L = lib.load()
    assert L.odg_policy_create_hidden(12, 8, 1024, 512, 0, None) == INVALID
