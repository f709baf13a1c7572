"""povar_bundle_adjust_async without a GPU: the entry point and its ctypes signature, the argument checks of the C
entry point that come before any device work, and the Python wrapper's checks before the library is called."""
import ctypes

import pytest

from povar_b200 import capi


def test_entry_point_and_signature_exist():
    lib = capi.load()
    fn = lib.povar_bundle_adjust_async
    assert fn.restype is ctypes.c_int
    assert len(fn.argtypes) == 7
    assert capi.SIGNATURES["povar_bundle_adjust_async"][1][1] is ctypes.POINTER(capi.Options)


def _call(h, opt, cap):
    return capi.load().povar_bundle_adjust_async(h, ctypes.byref(opt) if opt is not None else None, None, cap, None,
                                                 None, None)


def test_null_handle_or_negative_capacity_is_invalid():
    opt = capi.default_options()
    assert _call(None, opt, 10) == capi.ERR_INVALID
    assert _call(None, opt, -1) == capi.ERR_INVALID
    assert _call(None, None, 10) == capi.ERR_INVALID


class _NoLib:
    def __getattr__(self, name):
        raise AssertionError(f"the library was called ({name})")


def _solver():
    s = object.__new__(capi.Solver)
    s.lib = _NoLib()
    s.h = capi._H(1)
    s.device_index = 0
    s.options = capi.default_options()
    return s


@pytest.mark.parametrize("change,match", [
    (lambda s: {"options": object()}, "Options"),
    (lambda s: {"options": capi.default_options(max_num_iterations_step_1=-1)}, "negative"),
    (lambda s: {"options": capi.default_options(max_num_iterations_step_2=-3)}, "negative"),
    (lambda s: setattr(s, "h", None) or {}, "closed"),
])
def test_wrapper_checks_come_before_the_library(change, match):
    s = _solver()
    kw = change(s)
    with pytest.raises(ValueError, match=match):
        s.bundle_adjust_async(**kw)
    s.h = None   # nothing to destroy
