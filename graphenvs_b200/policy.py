"""Masked categorical over policy logits for the update step of a training loop (csrc/ge_policy.cu).

    log_prob, entropy = masked_log_prob(logits, mask_bits, actions)

`logits` [..., A] float32 / bfloat16 on a CUDA device, `mask_bits` [..., ceil(A/32)] int32 (the packed masks of
info['mask_bits'], e.g. stored per step in a [T, B, AW] rollout buffer), `actions` [...] int32 / int64.  Returns float32
[...] tensors; differentiable with respect to `logits`.  Only the logits of valid actions are read; the edge semantics
(empty rows, actions outside the mask) are those of ge_masked_log_prob in include/graphenvs_b200.h.
"""
import ctypes as C

import torch

from . import _native

_DTYPES = {torch.float32: _native.LOGITS_F32, torch.bfloat16: _native.LOGITS_BF16}


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def check_logits(logits, mask_bits, actions):
    """Validates the three tensors (no native call); returns (rows, A)."""
    for name, t in (("logits", logits), ("mask_bits", mask_bits), ("actions", actions)):
        if not isinstance(t, torch.Tensor):
            raise TypeError("masked_log_prob: %s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if logits.dtype not in _DTYPES:
        raise TypeError("masked_log_prob: logits must be float32 or bfloat16, got %s" % logits.dtype)
    if mask_bits.dtype != torch.int32:
        raise TypeError("masked_log_prob: mask_bits must be int32 (the packed words of info['mask_bits']), got %s" % mask_bits.dtype)
    if actions.dtype not in (torch.int32, torch.int64):
        raise TypeError("masked_log_prob: actions must be int32 or int64, got %s" % actions.dtype)
    if logits.dim() < 1:
        raise ValueError("masked_log_prob: logits must be [..., A]")
    A = int(logits.shape[-1])
    if A < 1:
        raise ValueError("masked_log_prob: A = 0 actions")
    lead = tuple(logits.shape[:-1])
    if mask_bits.dim() != logits.dim() or tuple(mask_bits.shape) != lead + ((A + 31) // 32,):
        raise ValueError("masked_log_prob: mask_bits shape %s does not match logits %s (expected %s)"
                         % (tuple(mask_bits.shape), tuple(logits.shape), lead + ((A + 31) // 32,)))
    if tuple(actions.shape) != lead:
        raise ValueError("masked_log_prob: actions shape %s does not match logits %s (expected %s)"
                         % (tuple(actions.shape), tuple(logits.shape), lead))
    for name, t in (("logits", logits), ("mask_bits", mask_bits), ("actions", actions)):
        if not t.is_cuda:
            raise ValueError("masked_log_prob: %s is on %s; the masked categorical runs on CUDA only" % (name, t.device))
    if mask_bits.device != logits.device or actions.device != logits.device:
        raise ValueError("masked_log_prob: logits, mask_bits and actions must be on one device")
    rows = 1
    for n in lead:
        rows *= int(n)
    if rows >= 2 ** 31:
        raise ValueError("masked_log_prob: %d rows exceed the 2^31 - 1 a call handles" % rows)
    return rows, A


def _int32_actions(actions, A):
    if actions.dtype == torch.int64:   # values outside [0, A) are invalid actions (log_prob -inf) whatever their size
        actions = torch.where((actions >= 0) & (actions < A), actions, torch.full_like(actions, -1)).to(torch.int32)
    return actions.contiguous()


class _MaskedLogProb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, mask_bits, actions):
        rows, A = check_logits(logits, mask_bits, actions)
        lead = tuple(logits.shape[:-1])
        dev = logits.device
        lp = torch.empty(lead, dtype=torch.float32, device=dev)
        ent = torch.empty(lead, dtype=torch.float32, device=dev)
        lse = torch.empty(lead, dtype=torch.float32, device=dev)
        x = logits.detach().contiguous()
        m = mask_bits.contiguous()
        a = _int32_actions(actions, A)
        if rows:
            L = _native.lib()
            with torch.cuda.device(dev):
                _native.check(L.ge_masked_log_prob(_ptr(x), _DTYPES[x.dtype], rows, A, _ptr(m), _ptr(a), _ptr(lp), _ptr(ent),
                                                   _ptr(lse), _stream(dev)))
        ctx.save_for_backward(x, m, a, lse, ent)
        return lp, ent

    @staticmethod
    def backward(ctx, g_lp, g_ent):
        x, m, a, lse, ent = ctx.saved_tensors
        grad = torch.empty_like(x)
        rows, A = x.numel() // max(int(x.shape[-1]), 1), int(x.shape[-1])
        if rows:
            g_lp = None if g_lp is None else g_lp.to(torch.float32).contiguous()
            g_ent = None if g_ent is None else g_ent.to(torch.float32).contiguous()
            L = _native.lib()
            with torch.cuda.device(x.device):
                _native.check(L.ge_masked_log_prob_backward(_ptr(x), _DTYPES[x.dtype], rows, A, _ptr(m), _ptr(a), _ptr(lse), _ptr(ent),
                                                            _ptr(g_lp), _ptr(g_ent), _ptr(grad), _stream(x.device)))
        return grad, None, None


def masked_log_prob(logits, mask_bits, actions):
    """(log_prob, entropy) float32 [...] of `actions` under softmax(logits) restricted to the valid actions of `mask_bits`.

    Differentiable with respect to `logits` (one fused backward kernel, dense gradient in the logits' dtype, exactly 0 on
    invalid actions).  Empty mask rows give (0, 0); an action outside [0, A) or on a clear bit gives log_prob = -inf and no
    log_prob gradient.  For the logits, masks and actions of a BatchedGraphEnv.sample_logits call the values equal the
    sampler's bit for bit, so the PPO ratio of the first epoch is exactly 1."""
    return _MaskedLogProb.apply(logits, mask_bits, actions)
