"""sdrgpu_chan_update_selection: exported with a prototype, and its NULL / count checks run before the handle is touched,
also without a GPU.  The refusals that need a live channelizer are in test_selection_update_gpu.py."""
import ctypes as C

import pytest


def _args(n=1):
    from sdrtrunk_b200 import native
    chans = (native.OutputChannel * max(n, 1))(*[native.OutputChannel(i, -1, 0, 96.0) for i in range(max(n, 1))])
    prev = (C.c_int * max(n, 1))(*([-1] * max(n, 1)))
    return chans, prev


def test_symbol_is_exported_with_a_prototype():
    from sdrtrunk_b200 import native
    lib = C.CDLL(native.LIB_PATH)
    assert hasattr(lib, "sdrgpu_chan_update_selection")
    assert "sdrgpu_chan_update_selection" in native.PROTOTYPES


@pytest.mark.parametrize("n", [0, -2])
def test_null_and_empty_arguments_are_refused(n):
    from sdrtrunk_b200 import native
    L = native.lib()
    chans, prev = _args()
    assert L.sdrgpu_chan_update_selection(None, chans, prev, 1, None, 0) == native.ERR_INVALID_ARG
    assert b"NULL" in L.sdrgpu_last_error()
    fake = C.c_void_p(16)   # never dereferenced: the NULL / count checks come first
    assert L.sdrgpu_chan_update_selection(fake, None, prev, 1, None, 0) == native.ERR_INVALID_ARG
    assert L.sdrgpu_chan_update_selection(fake, chans, None, 1, None, 0) == native.ERR_INVALID_ARG
    assert L.sdrgpu_chan_update_selection(fake, chans, prev, n, None, 0) == native.ERR_INVALID_ARG


def test_python_wrapper_refuses_a_previous_list_of_another_length():
    """updateOutputChannels checks the list lengths before it calls the library"""
    from sdrtrunk_b200 import native
    from sdrtrunk_b200.dsp import ComplexPolyphaseChannelizerM2
    ch = ComplexPolyphaseChannelizerM2.__new__(ComplexPolyphaseChannelizerM2)
    ch.mChannelCount = 96
    with pytest.raises(native.IllegalArgumentException):
        ch.updateOutputChannels([([3], 0), ([4], 0)], [0])
