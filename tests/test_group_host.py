"""CPU: the device-group entry points (fm_group_*) load through capi, and without a GPU fm_group_create fails with
FM_ERR_CUDA and says why instead of falling back."""
import ctypes as C

import pytest

from conftest import have_gpu
from frog_b200 import capi

GROUP_SYMBOLS = ["fm_group_create", "fm_group_destroy", "fm_group_last_error", "fm_group_synchronize",
                 "fm_group_clear_images", "fm_group_upload_image", "fm_group_match"]


def test_group_symbols_load(built):
    L = capi.load()
    for name in GROUP_SYMBOLS:
        assert name in capi.PUBLIC_SYMBOLS
        assert getattr(L, name).argtypes is not None, f"{name} has no ctypes signature in capi"


@pytest.mark.skipif(have_gpu(), reason="checks the no-GPU failure mode")
def test_group_create_without_device(built):
    L = capi.load()
    h = C.c_void_p(1234)
    devs = (C.c_int * 2)(0, 1)
    assert L.fm_group_create(devs, 2, C.byref(h)) == capi.ERR_CUDA
    assert not h.value
    text = L.fm_group_last_error(None).decode()
    assert "no CUDA device" in text
    with pytest.raises(capi.FrogMatchError, match="no CUDA device"):
        capi.Group([0])
