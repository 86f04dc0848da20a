"""CPU: the MVRC loss entry points of the C ABI reject bad arguments with an error code and a message (no device needed:
the checks run before any launch)."""
import ctypes
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "vl-bert_b200", "libvlbert_b200.so")


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        import importlib.util
        spec = importlib.util.spec_from_file_location("vlb_build", os.path.join(ROOT, "vl-bert_b200", "build.py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        m.build()
    handle = ctypes.CDLL(LIB)
    P, I = ctypes.c_void_p, ctypes.c_int
    for name, args in (("vlb_soft_target_rows", [P, I, I, I, P, P]),
                       ("vlb_soft_ce_forward", [P, I, I, P, I, P, P, P, I, P, P, P, P]),
                       ("vlb_soft_ce_backward", [P, I, I, P, I, P, P, I, P, P, P])):
        getattr(handle, name).restype = I
        getattr(handle, name).argtypes = args
    handle.vlb_last_error_string.restype = ctypes.c_char_p
    return handle


def test_bad_arguments_return_error_codes(lib):
    x = 16      # a non-null address that is never dereferenced: every call below fails its argument check first
    assert lib.vlb_soft_target_rows(None, 8, 17, 17, x, None) != 0
    assert lib.vlb_soft_target_rows(x, 8, 17, 16, x, None) != 0                       # row stride below C
    assert b"soft_target_rows" in lib.vlb_last_error_string()
    assert lib.vlb_soft_ce_forward(x, 20, 17, x, 17, x, x, x, 8, x, x, x, None) != 0    # ld not a multiple of 8
    assert lib.vlb_soft_ce_forward(x, 24, 17, x, 17, x, x, x, 8, None, x, x, None) != 0
    assert b"soft_ce_forward" in lib.vlb_last_error_string()
    assert lib.vlb_soft_ce_backward(x, 24, 17, x, 17, x, x, 0, x, x, None) != 0        # no rows
    assert lib.vlb_soft_ce_backward(x, 24, 17, x, 17, x, x, 8, x, None, None) != 0     # no per-row weights
    assert b"soft_ce_backward" in lib.vlb_last_error_string()
