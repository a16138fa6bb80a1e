"""Fused sketch-program runs without a device: what gcs_b200_program_run_fused[_host] and
SketchProgram::runFused refuse before any device call, with their return codes and exact messages."""
import ctypes as C

import numpy as np
import pytest

import host_lib as H
import program_tangents_lib as P
import sketch_gen as S


def test_the_fused_entry_points_check_their_arguments_first(gcs, built):
    capi = gcs.capi
    lib = capi.load()
    buf = (C.c_double * 8)()
    ms = (C.c_float * 3)()
    for fn, last in ((lib.gcs_b200_program_run_fused, None), (lib.gcs_b200_program_run_fused_host, ms)):
        cases = [
            ((None, 1, buf, buf, None, -1, buf, buf, last), b"n_tangents must be >= 0 (got -1)"),
            ((None, 1, buf, buf, None, -7, None, None, last), b"n_tangents must be >= 0 (got -7)"),
            ((None, 1, buf, buf, None, 2, None, buf, last), b"null tangent table (dvalues or dpositions)"),
            ((None, 1, buf, buf, None, 2, buf, None, last), b"null tangent table (dvalues or dpositions)"),
            ((None, 1, buf, buf, None, 0, None, None, last), b"null program"),
            ((None, 0, buf, buf, None, 0, None, None, last), b"null program"),
            ((None, 1, buf, buf, None, 2, buf, buf, last), b"null program"),
        ]
        for args, message in cases:
            before = lib.gcs_b200_launch_count()
            assert fn(*args) == capi.GCS_E_INVALID, message
            assert lib.gcs_b200_last_error() == message
            assert lib.gcs_b200_launch_count() == before


@pytest.fixture(scope="module")
def host(built):
    built.build_host()
    lib = H.load()
    vp, dp = C.c_void_p, C.POINTER(C.c_double)
    lib.gcs_host_program_run_fused.argtypes = [vp, C.c_int64, dp, C.c_int, dp, dp, dp, C.POINTER(C.c_uint32), C.c_int,
                                               C.POINTER(C.c_int64)]
    return lib


@pytest.mark.parametrize("K,T,message", [(1, -1, "SketchProgram::runFused: T must be >= 0 (got -1)"),
                                         (0, 0, "SketchProgram::run: K must be >= 1"),
                                         (-3, 2, "SketchProgram::run: K must be >= 1")])
def test_run_fused_refuses_before_any_device_call(host, K, T, message):
    el, lv = S.make_sketch(300, seed=31, first_shape=1)
    prog = P.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    d = prog.describe()
    vals = np.ones((1, d["values"]))
    dvals = np.zeros((1, d["values"], max(T, 1)))
    pos, dpos = np.zeros((1, d["slots"], 4)), np.zeros((1, d["slots"], 4, max(T, 1)))
    rc = host.gcs_host_program_run_fused(prog.handle, K, H._dp(vals), T, H._dp(dvals), H._dp(pos), H._dp(dpos), None, 1, None)
    assert rc == -1
    assert H.last_error() == message
