"""Guarded device buffers for kernel-level tests: an output tensor sits inside a larger allocation whose every byte is
a sentinel before the launch, so a write outside the tensor, or to a part of it the kernel must leave alone, shows up
as a changed byte."""
import ctypes

import numpy as np
import torch

SENTINEL = 0xFF          # every byte of an output allocation before the launch (fp16 / fp32 NaN, int32 -1)
GUARD = 4096


class Guarded:
    """A tensor inside a larger allocation: GUARD bytes of sentinel before and after it, base 1024-byte aligned
    (TMA), the whole allocation filled with the sentinel.  As an input buffer, the guards are NaN (fp32 / fp16)."""

    def __init__(self, shape, dtype, dev):
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        self.raw = torch.full((n + 2 * GUARD + 2048,), SENTINEL, dtype=torch.uint8, device=dev)
        self.lo = (-self.raw.data_ptr()) % 1024 + GUARD
        self.hi = self.lo + n
        self.t = self.raw[self.lo:self.hi].view(dtype).view(shape)

    def body(self):
        """The tensor's bytes (two Guarded buffers may sit at different offsets of their allocations)."""
        return self.raw[self.lo:self.hi]

    def guards_intact(self):
        return bool((self.raw[:self.lo] == SENTINEL).all()) and bool((self.raw[self.hi:] == SENTINEL).all())


def untouched(t):
    return t.numel() == 0 or bool((t.contiguous().view(torch.uint8) == SENTINEL).all())


def pos_zero(t):
    return t.numel() == 0 or bool((t.contiguous().view(torch.uint8) == 0).all())


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
