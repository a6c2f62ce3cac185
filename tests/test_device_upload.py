"""CPU-side checks of the device-buffer upload (psulvsb_batch_upload_device, capi.DeviceProblem): the tensor checks of
DeviceProblem and the error without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi


def pts(n, dtype=torch.float64):
    return torch.zeros((n, 3), dtype=dtype)


def test_device_problem_refuses_cpu_tensors():
    with pytest.raises(ValueError, match="src must be a CUDA tensor"):
        capi.DeviceProblem(pts(8), pts(8))
    with pytest.raises(ValueError, match="must be a torch tensor"):
        capi.DeviceProblem(np.zeros((8, 3)), np.zeros((8, 3)))


@pytest.mark.parametrize("bad, match", [
    (dict(src=pts(8, torch.float32)), "src must be torch.float64"),
    (dict(dst=pts(8, torch.float32)), "dst must be torch.float64"),
    (dict(src=torch.zeros((3, 8), dtype=torch.float64)), r"src must have shape \['\*', 3\]"),
    (dict(src=torch.zeros(24, dtype=torch.float64)), "src must have shape"),
    (dict(dst=pts(9)), r"dst must have shape \[8, 3\]"),
    (dict(src=torch.zeros((3, 8), dtype=torch.float64).T), "src must be contiguous"),
    (dict(ori_src=pts(8)), "ori_src and ori_dst go together"),
    (dict(keep_mask=torch.ones(8, dtype=torch.int32)), "keep_mask and reduce_map go together"),
    (dict(), "src must be a CUDA tensor"),
])
def test_device_problem_refuses_wrong_dtypes_and_shapes(bad, match):
    kw = dict(src=pts(8), dst=pts(8))
    kw.update(bad)
    with pytest.raises(ValueError, match=match):
        capi.DeviceProblem(**kw)


def test_device_problem_refuses_wrong_pre_filter_arrays():
    kw = dict(src=pts(4), dst=pts(4), ori_src=pts(8), ori_dst=pts(8))
    with pytest.raises(ValueError, match=r"ori_dst must have shape \[8, 3\]"):
        capi.DeviceProblem(pts(4), pts(4), pts(8), pts(7), torch.ones(8, dtype=torch.int32),
                           torch.zeros(8, dtype=torch.int32))
    with pytest.raises(ValueError, match="keep_mask must be torch.int32"):
        capi.DeviceProblem(**kw, keep_mask=torch.ones(8, dtype=torch.int64), reduce_map=torch.zeros(8, dtype=torch.int32))
    with pytest.raises(ValueError, match=r"reduce_map must have shape \[8\]"):
        capi.DeviceProblem(**kw, keep_mask=torch.ones(8, dtype=torch.int32), reduce_map=torch.zeros(4, dtype=torch.int32))
    with pytest.raises(ValueError, match="pairs must be"):
        capi.DeviceProblem.from_matches(pts(8), pts(8), torch.zeros((4, 2), dtype=torch.int64))
    with pytest.raises(ValueError, match="d_src_cloud must be a CUDA tensor"):
        capi.DeviceProblem.from_matches(pts(8), pts(8), torch.zeros((4, 2), dtype=torch.int32))


def test_upload_device_without_a_device():
    L = capi.lib()
    if L.psulvsb_device_count() > 0:
        pytest.skip("a CUDA device is present")
    arr = (capi.Problem * 1)()
    assert L.psulvsb_batch_upload_device(None, None, arr, 1) == capi.ERR_NO_DEVICE
    assert b"no CUDA device" in L.psulvsb_last_error()
    with pytest.raises(capi.PsulvsbError) as e:
        capi.Handle(0)
    assert e.value.code == capi.ERR_NO_DEVICE
    h = capi.Handle.__new__(capi.Handle)  # a handle that was never created: the entry point still answers first
    h._h = C.c_void_p()
    with pytest.raises(capi.PsulvsbError) as e:
        h.upload_device([])
    assert e.value.code == capi.ERR_NO_DEVICE

