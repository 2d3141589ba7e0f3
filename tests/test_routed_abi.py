"""The routed pipeline's entry points refuse NULL handles and arguments before anything touches the device, also
without a GPU."""
import ctypes


def test_routed_pipeline_refuses_null_arguments():
    from sdrtrunk_b200 import native
    L = native.lib()
    invalid = 1   # SDRGPU_ERR_INVALID_ARG
    h = ctypes.c_void_p()
    route = (ctypes.c_int * 1)(0)
    none = (ctypes.c_void_p * 1)(None)
    assert L.sdrgpu_pipeline_create_routed(None, None, 0, None, 0, None) == invalid
    assert L.sdrgpu_pipeline_create_routed(ctypes.byref(h), None, 1, none, 1, route) == invalid
    assert L.sdrgpu_pipeline_create_routed(ctypes.byref(h), none, 1, None, 1, route) == invalid
    assert L.sdrgpu_pipeline_create_routed(ctypes.byref(h), none, 1, none, 1, None) == invalid
    assert L.sdrgpu_pipeline_create_routed(ctypes.byref(h), none, 0, none, 1, route) == invalid
    assert L.sdrgpu_pipeline_create_routed(ctypes.byref(h), none, 1, none, 0, route) == invalid
    assert L.sdrgpu_pipeline_create_routed(ctypes.byref(h), none, 1, none, 1, route) == invalid   # NULL channelizer
    assert not h.value
    outputs = (native.BankOutput * 1)()
    assert L.sdrgpu_pipeline_process_routed(None, None, 0, native.HOST, outputs, native.HOST) == invalid
    assert L.sdrgpu_pipeline_process_routed(None, None, 0, native.HOST, None, native.HOST) == invalid
    assert b"NULL" in L.sdrgpu_last_error()
