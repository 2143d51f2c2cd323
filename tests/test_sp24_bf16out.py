"""bf16 output with a per-row bias for the 2:4-sparse operators (libxsmm_b200_sp24_execute_bf16out / _execute_fp8_bf16out,
Sp24.execute(bias=, c_dtype=), Sp24.linear): the refusals decided before the library is called, and the library's NULL-handle
check of both new entries.  None needs a GPU: the operators below carry no handle, so a refusal that slipped through would
reach the library as a NULL-handle error, which every test rules out."""
import numpy as np
import pytest


def refused(xs, match, call):
    """call raises ValueError(match) and neither launches nor reaches the library"""
    xs.clear_error()
    n0 = xs.launch_count()
    with pytest.raises(ValueError, match=match):
        call()
    assert xs.launch_count() == n0
    assert xs.last_error()[0] == 0, xs.last_error()


def op_without_handle(xs, M, K, fp8=False, fmt=None):
    op = xs.Sp24.__new__(xs.Sp24)
    op.M, op.K, op.lda, op.fp8, op.format, op.handle = M, K, K, fp8, (xs.FP8_FORMATS[fmt] if fp8 else None), None
    return op


def test_bias_needs_bf16_c(xs):
    import torch
    op = op_without_handle(xs, 64, 32)
    bias = torch.zeros(64, dtype=torch.bfloat16)
    c32 = torch.zeros((64, 16), dtype=torch.float32)
    refused(xs, "bias needs bf16 C", lambda: op.execute(0x1000, c32, 16, bias=bias))
    refused(xs, "bias needs bf16 C", lambda: op.execute(0x1000, 0x2000, 16, bias=0x3000))                 # raw C is fp32 by default
    refused(xs, "bias needs bf16 C", lambda: op.execute(0x1000, 0x2000, 16, bias=0x3000, c_dtype="fp32"))
    op8 = op_without_handle(xs, 64, 32, True, "e4m3")
    refused(xs, "bias needs bf16 C", lambda: op8.execute(0x1000, 0x2000, 16, bias=0x3000, b_fmt="e4m3"))


@pytest.mark.parametrize("c_dtype,tensor_dtype,match", [
    ("bf16", "float32", "does not match"),
    ("fp32", "bfloat16", "does not match"),
    ("fp16", None, "c_dtype must be"),
    ("bfloat16", None, "c_dtype must be"),
])
def test_c_dtype_must_agree_with_the_tensor(xs, c_dtype, tensor_dtype, match):
    import torch
    op = op_without_handle(xs, 64, 32)
    c = 0x2000 if tensor_dtype is None else torch.zeros((64, 16), dtype=getattr(torch, tensor_dtype))
    refused(xs, match, lambda: op.execute(0x1000, c, 16, c_dtype=c_dtype))


@pytest.mark.parametrize("dtype,n", [("float32", 64), ("float16", 64), ("bfloat16", 63), ("bfloat16", 65)])
def test_torch_bias_must_hold_m_bf16_values(xs, dtype, n):
    import torch
    op = op_without_handle(xs, 64, 32)
    c = torch.zeros((64, 16), dtype=torch.bfloat16)
    refused(xs, "bias must be", lambda: op.execute(0x1000, c, 16, bias=torch.zeros(n, dtype=getattr(torch, dtype))))


def test_fp8_format_mismatch_with_bf16_c(xs):
    import torch
    op8 = op_without_handle(xs, 64, 32, True, "e4m3")
    b = torch.zeros((32, 16), dtype=torch.float8_e4m3fn)
    c = torch.zeros((64, 16), dtype=torch.bfloat16)
    refused(xs, "does not match", lambda: op8.execute(b, c, 16, b_fmt="e5m2"))
    refused(xs, "fmt", lambda: op8.execute(0x1000, c, 16))                          # raw bytes need b_fmt


def test_linear_refuses_wrong_x(xs):
    import torch
    M, K = 64, 32
    op = op_without_handle(xs, M, K)
    x = torch.zeros((3, 5, K), dtype=torch.bfloat16)
    refused(xs, "torch tensor", lambda: op.linear(np.zeros((5, K), np.uint16)))
    refused(xs, "bfloat16", lambda: op.linear(x.float()))
    refused(xs, "bfloat16", lambda: op.linear(x.to(torch.float8_e4m3fn)))
    refused(xs, "last dimension", lambda: op.linear(torch.zeros((5, K + 8), dtype=torch.bfloat16)))
    refused(xs, "last dimension", lambda: op.linear(x.transpose(1, 2)))
    refused(xs, "contiguous", lambda: op.linear(torch.zeros((K, 10), dtype=torch.bfloat16).t()[::2]))
    refused(xs, "alpha", lambda: op.linear(x, alpha=0.5))
    refused(xs, "16-byte boundary", lambda: op.linear(torch.zeros(K + 1, dtype=torch.bfloat16)[1:]))
    refused(xs, "CUDA tensor", lambda: op.linear(x))                                # a host x is never copied


@pytest.mark.parametrize("fp8,K,unit", [(False, 36, 8), (False, 100, 8), (True, 40, 16), (True, 72, 16)])
def test_linear_refuses_k_the_tma_rule_refuses(xs, fp8, K, unit):
    import torch
    op = op_without_handle(xs, 64, K, fp8, "e4m3" if fp8 else None)
    x = torch.zeros((4, K), dtype=torch.float8_e4m3fn if fp8 else torch.bfloat16)
    refused(xs, "K=%d must be a multiple of %d" % (K, unit), lambda: op.linear(x))


def test_linear_fp8_operator_takes_float8_x(xs):
    import torch
    op8 = op_without_handle(xs, 64, 32, True, "e5m2")
    refused(xs, "float8", lambda: op8.linear(torch.zeros((4, 32), dtype=torch.bfloat16)))
    refused(xs, "float8", lambda: op8.linear(torch.zeros((4, 32), dtype=torch.uint8)))
    for dt in (torch.float8_e4m3fn, torch.float8_e5m2):      # both formats reach the device check (x is on the host here)
        refused(xs, "CUDA tensor", lambda: op8.linear(torch.zeros((4, 32), dtype=dt), alpha=0.25))


@pytest.mark.parametrize("bias,match", [
    ("array", "torch tensor"),
    ("float32", "bias must be"),
    ("short", "bias must be"),
    ("strided", "bias must be"),
])
def test_linear_refuses_wrong_bias(xs, bias, match):
    import torch
    M, K = 64, 32
    op = op_without_handle(xs, M, K)
    b = {"array": lambda: np.zeros(M, np.uint16), "float32": lambda: torch.zeros(M),
         "short": lambda: torch.zeros(M - 1, dtype=torch.bfloat16),
         "strided": lambda: torch.zeros(2 * M, dtype=torch.bfloat16)[::2]}[bias]()
    refused(xs, match, lambda: op.linear(torch.zeros((4, K), dtype=torch.bfloat16), bias=b))


def test_raw_entries_reject_a_null_handle_before_any_cuda_call(xs):
    for call in (lambda: xs.sp24_execute_bf16out(None, "T", "T", 16, 0x1000, 32, 0x3000, 0.0, 0x2000, 64),
                 lambda: xs.sp24_execute_fp8_bf16out(None, "N", "N", 16, 0x1000, 0, 16, 1.0, None, 0.0, 0x2001, 16)):
        xs.clear_error()
        n0 = xs.launch_count()
        call()
        code, msg = xs.last_error()
        xs.clear_error()
        assert xs.launch_count() == n0
        assert code == -97 and "NULL handle" in msg, msg
