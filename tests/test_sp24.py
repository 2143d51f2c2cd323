"""Fixed 2:4-sparse bf16 operators (libxsmm_b200_sp24_*): the host-side rejections.  Every -95 case of create and the
-97 rejections that need no handle are decided before any CUDA call, so they run without a GPU: nothing is launched, the
sticky error carries the code and a message naming the bad argument."""
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


A = np.zeros((4, 8), np.uint16)


@pytest.mark.parametrize("M,K,lda,a,fragment", [
    (0, 8, 8, A, "M=0"),
    (-3, 8, 8, A, "M=-3"),
    (4, 0, 8, A, "K=0"),
    (4, -1, 8, A, "K=-1"),
    (4, 8, 7, A, "lda=7"),
    (4, 8, 8, None, "a=(nil)"),
])
def test_create_rejects_bad_shape_before_any_cuda_call(xs, M, K, lda, a, fragment):
    h = rejected(xs, -95, fragment, lambda: xs.sp24_create_bfloat16(M, K, lda, a))
    assert not h


def test_sp24_class_raises_on_rejection(xs):
    xs.clear_error()
    n0 = xs.launch_count()
    with pytest.raises(ValueError, match=r"\(-95\)"):
        xs.Sp24(np.zeros((4, 8), np.uint16), lda=4)
    assert xs.launch_count() == n0
    assert xs.last_error()[0] == 0      # the class took the error over


@pytest.mark.parametrize("transb,transc,N,ldb,ldc", [
    ("N", "N", 16, 16, 16),     # only the handle is wrong
    ("X", "N", 16, 16, 16),     # every other argument wrong as well: the handle is checked first
    ("N", "N", -1, 16, 16),
])
def test_execute_rejects_null_handle(xs, transb, transc, N, ldb, ldc):
    rejected(xs, -97, "NULL handle", lambda: xs.sp24_execute(None, transb, transc, N, 0x1000, ldb, 0.0, 0x2000, ldc))


def test_destroy_null_is_a_no_op(xs):
    xs.clear_error()
    xs.sp24_destroy(None)
    assert xs.last_error()[0] == 0
