"""Fixed 2:4-sparse FP8 operators (libxsmm_b200_sp24_create_fp8 / _execute_fp8): the host-side rejections.  Every -95 case
of create and the -97 rejections that need no handle are decided before any CUDA call, so they run without a GPU: nothing
is launched, the sticky error carries the code and a message naming the bad argument."""
import numpy as np
import pytest


def rejected(xs, code, fragment, call):
    xs.clear_error()
    n0 = xs.launch_count()
    out = call()
    assert xs.launch_count() == n0
    got, msg = xs.last_error()
    xs.clear_error()
    assert got == code, msg
    assert fragment in msg, msg
    return out


A = np.zeros((4, 16), np.uint8)


@pytest.mark.parametrize("M,K,lda,a,fmt,fragment", [
    (0, 16, 16, A, 0, "M=0"),
    (-3, 16, 16, A, 0, "M=-3"),
    (4, 0, 16, A, 1, "K=0"),
    (4, -1, 16, A, 0, "K=-1"),
    (4, 16, 15, A, 0, "lda=15"),
    (4, 16, 16, None, 0, "a=(nil)"),
    (4, 16, 16, A, 2, "format=2"),
    (4, 16, 16, A, -1, "format=-1"),
])
def test_create_fp8_rejects_bad_shape_before_any_cuda_call(xs, M, K, lda, a, fmt, fragment):
    h = rejected(xs, -95, fragment, lambda: xs.sp24_create_fp8(M, K, lda, a, fmt))
    assert not h


def test_sp24_class_raises_on_fp8_rejection(xs):
    xs.clear_error()
    n0 = xs.launch_count()
    with pytest.raises(ValueError, match=r"sp24_create_fp8 failed \(-95\)"):
        xs.Sp24(np.zeros((4, 16), np.uint8), lda=8, fmt="e4m3")
    assert xs.launch_count() == n0
    assert xs.last_error()[0] == 0      # the class took the error over


@pytest.mark.parametrize("fmt", [None, "e4m3fn", "fp8"])
def test_sp24_class_needs_the_format_of_raw_bytes(xs, fmt):
    n0 = xs.launch_count()
    with pytest.raises(ValueError, match="fmt"):
        xs.Sp24(np.zeros((4, 16), np.uint8), fmt=fmt)
    assert xs.launch_count() == n0


@pytest.mark.parametrize("transb,transc,N,b_fmt,ldb,ldc", [
    ("N", "N", 16, 0, 16, 16),     # only the handle is wrong
    ("X", "N", 16, 0, 16, 16),     # every other argument wrong as well: the handle is checked first
    ("N", "N", 16, 7, 16, 16),
    ("N", "N", -1, 0, 16, 16),
])
def test_execute_fp8_rejects_null_handle(xs, transb, transc, N, b_fmt, ldb, ldc):
    rejected(xs, -97, "NULL handle",
             lambda: xs.sp24_execute_fp8(None, transb, transc, N, 0x1000, b_fmt, ldb, 1.0, 0.0, 0x2000, ldc))
