"""Poisoned allocations for kernel tests.

``ops`` allocates every output, bf16 copy, LN-statistics and column-statistics buffer and the polar / GroupNorm workspaces with
``torch.empty`` / ``torch.empty_like``.  The caching allocator often hands back the very bytes a previous identical call left, so
a kernel that skips part of its output can still look right.  Inside ``poisoned()`` those allocations come back filled with 0xFF
bytes instead: NaN in fp32 / bf16 / fp16, 255 in uint8.  Anything a kernel leaves unwritten then stays NaN and fails a comparison.

Buffers that must start zeroed (the split-K workspace, the prior-trunk workspace) are made with ``torch.zeros`` and untouched.
"""
import contextlib

import torch

POISON_BYTE = 0xFF


def _poisonable(t):
    return t.dtype.is_floating_point or t.dtype == torch.uint8


def _poison(t):
    if _poisonable(t) and t.numel() > 0:
        t.untyped_storage().fill_(POISON_BYTE)
    return t


@contextlib.contextmanager
def poisoned():
    """``torch.empty`` and ``torch.empty_like`` return 0xFF-filled memory (floating-point and uint8 tensors) inside the block."""
    empty, empty_like = torch.empty, torch.empty_like
    torch.empty = lambda *a, **k: _poison(empty(*a, **k))
    torch.empty_like = lambda *a, **k: _poison(empty_like(*a, **k))
    try:
        yield
    finally:
        torch.empty, torch.empty_like = empty, empty_like


def is_poison(t):
    """elementwise: does ``t`` still hold the poison bytes (all bits set)?"""
    bits = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()]
    return t.contiguous().view(bits) == (POISON_BYTE if bits is torch.uint8 else -1)
