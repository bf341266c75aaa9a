"""CPU: argument validation of the CUDA-graph building blocks of the C ABI (no device needed: every check runs before
the first CUDA call)."""
import ctypes as C

import mscs_b200
import torch
from mscs_b200 import _ops


def test_philox_stream_dev_rejects_bad_pointers():
    lib = mscs_b200.load()
    ok_call, ok_draws = C.c_void_p(0x10000), C.c_void_p(0x20000)     # never dereferenced: validation fails first
    for call, draws, what in [(None, ok_draws, b"call_dev"), (C.c_void_p(0x10004), ok_draws, b"call_dev"),
                              (ok_call, None, b"draws_dev"), (ok_call, C.c_void_p(0x20008), b"draws_dev")]:
        rc = lib.mscs_philox_stream_dev(1, call, 64, draws, None)
        assert rc < 0, (call, draws)
        assert what in lib.mscs_last_error()


def test_forward_chain_without_plan_host_still_validates():
    lib = mscs_b200.load()
    from mscs_b200 import _lib
    args = _lib.ForwardChainArgs()          # every pointer null: rejected before anything is enqueued
    assert lib.mscs_forward_chain(C.byref(args), None, None, None) < 0
    assert b"null pointer" in lib.mscs_last_error()


def test_graph_mode_is_off_outside_a_capture():
    spec = _ops.LossSpec(num_classes=20, temperature=0.1, cs_temperature=0.1, sampler="philox")
    assert _ops.graph_mode(spec, 1, False, torch.zeros(1, 8, 8), [torch.zeros(1, 4, 2, 2)], None) is False
    assert _ops.GRAPH_CALL_BASE == 2 ** 62
