"""Device-resident input without a GPU: the ctypes mirror of povar_device_problem_desc, the descriptor checks of
povar_create_device that come before any device work, and DeviceProblem's checks of its tensors."""
import ctypes

import pytest
import torch

from povar_b200 import capi


def _desc(**kw):
    d = capi.DeviceProblemDesc(num_cams=2, num_lms=3, num_obs=4, lm_begin=0, lm_end=3, obs_cam=0x1000,
                               obs_lm=0x2000, obs_uv=0x3000, cam_P=0x4000, stream=None)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def _create(desc):
    lib = capi.load()
    h = capi._H()
    opt = capi.default_options()
    return lib.povar_create_device(ctypes.byref(desc) if desc is not None else None, ctypes.byref(opt), None,
                                   ctypes.byref(h))


def test_mirror_matches_the_library_struct():
    assert capi.load().povar_abi_sizeof(9) == ctypes.sizeof(capi.DeviceProblemDesc)


def test_null_or_malformed_descriptor_is_invalid():
    assert _create(None) == capi.ERR_INVALID
    assert _create(_desc(obs_lm=None)) == capi.ERR_INVALID
    assert _create(_desc(cam_P=None)) == capi.ERR_INVALID
    assert _create(_desc(num_cams=0)) == capi.ERR_INVALID
    for lb, le in ((2, 1), (-1, 3), (0, 4)):
        assert _create(_desc(lm_begin=lb, lm_end=le)) == capi.ERR_INVALID, (lb, le)
    assert b"landmark range" in capi.load().povar_last_error(None)


def test_too_many_observations_is_unsupported():
    assert _create(_desc(num_obs=1 << 31)) == capi.ERR_UNSUPPORTED


def test_well_formed_descriptor_without_gpu_is_no_device():
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    assert _create(_desc()) == capi.ERR_NO_DEVICE


def _tensors(n=5, C=2):
    return dict(cam_P=torch.zeros(C, 3, 4, dtype=torch.float64), obs_cam=torch.zeros(n, dtype=torch.int32),
                obs_lm=torch.arange(n, dtype=torch.int32), obs_uv=torch.zeros(n, 2, dtype=torch.float64))


@pytest.mark.parametrize("change,match", [
    (lambda t: t.update(obs_cam=t["obs_cam"].long()), "dtype"),
    (lambda t: t.update(obs_lm=t["obs_lm"].float()), "dtype"),
    (lambda t: t.update(obs_uv=t["obs_uv"].float()), "dtype"),
    (lambda t: t.update(cam_P=t["cam_P"].float()), "dtype"),
    (lambda t: t.update(obs_uv=t["obs_uv"].t().contiguous().t()), "contiguous"),
    (lambda t: t.update(cam_P=torch.zeros(3, 4, 2, dtype=torch.float64).transpose(1, 2)), "contiguous"),
    (lambda t: t.update(obs_lm=t["obs_lm"][:4].clone()), r"\[N\]"),
    (lambda t: t.update(obs_uv=torch.zeros(5, 3, dtype=torch.float64)), r"\[N, 2\]"),
    (lambda t: t.update(cam_P=torch.zeros(2, 11, dtype=torch.float64)), "cam_P must be"),
    (lambda t: t.update(cam_P=torch.zeros(0, 12, dtype=torch.float64)), "cam_P must be"),
    (lambda t: t.update(obs_cam=t["obs_cam"].numpy()), "torch tensor"),
    (lambda t: None, "CUDA tensor"),
])
def test_device_problem_rejects_bad_tensors(change, match):
    t = _tensors()
    change(t)
    with pytest.raises(ValueError, match=match):
        capi.DeviceProblem(**t, num_lms=5)


@pytest.mark.parametrize("num_lms,lm_range", [(5, (3, 2)), (5, (-1, 2)), (5, (0, 6)), (-1, None)])
def test_device_problem_rejects_bad_ranges(num_lms, lm_range):
    with pytest.raises(ValueError, match="range|num_lms"):
        capi.DeviceProblem(**_tensors(), num_lms=num_lms, lm_range=lm_range)
