"""CPU: argument checks of the masked categorical (graphenvs_b200.policy, ge_masked_log_prob*) that need no device."""
import ctypes as C

import pytest
import torch

from graphenvs_b200 import _native, policy


def _args(R=4, A=40, dt=torch.float32):
    return torch.zeros((R, A), dtype=dt), torch.zeros((R, (A + 31) // 32), dtype=torch.int32), torch.zeros(R, dtype=torch.int32)


def test_package_exports_masked_log_prob():
    import graphenvs_b200
    assert graphenvs_b200.masked_log_prob is policy.masked_log_prob


@pytest.mark.parametrize("bad, err, match", [
    (lambda x, m, a: (x.double(), m, a), TypeError, "float32 or bfloat16"),
    (lambda x, m, a: (x, m.long(), a), TypeError, "mask_bits must be int32"),
    (lambda x, m, a: (x, m, a.float()), TypeError, "actions must be int32 or int64"),
    (lambda x, m, a: (x, m[:, :1], a), ValueError, "mask_bits shape"),
    (lambda x, m, a: (x, m[:3], a), ValueError, "mask_bits shape"),
    (lambda x, m, a: (x, m, a[:3]), ValueError, "actions shape"),
    (lambda x, m, a: (x[:, :0], m[:, :0], a), ValueError, "A = 0"),
    (lambda x, m, a: (x.numpy(), m, a), TypeError, "must be a torch.Tensor"),
    (lambda x, m, a: (x, m, a), ValueError, "runs on CUDA only"),            # CPU tensors
])
def test_masked_log_prob_rejects_bad_arguments_before_any_native_call(bad, err, match, monkeypatch):
    def no_native():
        raise AssertionError("native library reached")
    monkeypatch.setattr(_native, "lib", no_native)
    with pytest.raises(err, match=match):
        policy.masked_log_prob(*bad(*_args()))


def test_native_entry_points_reject_bad_arguments():
    L = _native.lib()
    x = C.c_void_p(16)   # never dereferenced: the checks come first
    assert L.ge_masked_log_prob(x, 7, 4, 40, x, x, x, x, x, None) == -1
    assert b"dtype" in L.ge_last_error()
    assert L.ge_masked_log_prob(x, 0, 0, 40, x, x, x, x, x, None) == -1
    assert L.ge_masked_log_prob(x, 1, 4, 0, x, x, x, x, x, None) == -1
    assert L.ge_masked_log_prob(None, 0, 4, 40, x, x, x, x, x, None) == -1
    assert L.ge_masked_log_prob(x, 0, 4, 40, x, x, None, x, x, None) == -1
    assert L.ge_masked_log_prob_backward(x, 0, 4, 40, x, x, x, x, None, None, None, None) == -1
    assert L.ge_masked_log_prob_backward(x, 2, 4, 40, x, x, x, x, None, None, x, None) == -1
    d = _native.GeBatch()
    d.kind, d.B, d.N, d.M = 0, 8, 40, 80
    assert L.ge_fill_layout(C.byref(d)) == 0
    assert L.ge_sample_logits(C.byref(d), x, 3, 0, 1, 0, x, None, None, None) == -1
    assert L.ge_sample_logits(C.byref(d), None, 0, 0, 1, 0, x, None, None, None) == -1
    assert b"null" in L.ge_last_error()
    assert L.ge_sample_logits(None, x, 0, 0, 1, 0, x, None, None, None) == -1
