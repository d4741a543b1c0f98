"""CPU-only checks of the 16 x 16-window attention backward entry point: it rejects every other geometry before it
touches a pointer or the device."""
import pytest

from diffusesg_b200 import native

DSG_ERR_INVALID = 1


@pytest.mark.parametrize("window,shift,res", [(8, 0, 64), (10, 5, 40), (16, 4, 64), (16, 8, 40), (16, 0, 24)])
def test_w16_attention_backward_rejects_other_geometries(window, shift, res):
    lib = native.lib()
    fake = 4096    # never dereferenced: the arguments are checked first
    rc = lib.dsg_tr_window_attention_bwd_w16(fake, fake, fake, fake, fake, 2, res, window, shift, 3, None)
    assert rc == DSG_ERR_INVALID
    msg = lib.dsg_last_error().decode()
    assert "16 x 16" in msg and f"window {window}, shift {shift}, res {res}" in msg, msg


def test_w16_attention_backward_rejects_missing_tensors():
    rc = native.lib().dsg_tr_window_attention_bwd_w16(None, 4096, 4096, 4096, 4096, 2, 64, 16, 8, 3, None)
    assert rc == DSG_ERR_INVALID
