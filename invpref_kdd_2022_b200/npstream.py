"""numpy's global stream on the GPU: ``device_randint(high, n, device)`` returns, as an int64 CUDA tensor, exactly what
``np.random.randint(0, high, n)`` would have returned, and leaves ``np.random`` in exactly the state that call would
have left it in (``invpref_mt_randint``, csrc/nprng.cu).  The trainers' ``tie_break_rng="numpy_device"`` mode draws the
initial environments (train.py:711) and the tie-break rows (train.py:870-871) this way: the reference's stream, without
the ~10 ns per sample of numpy's sequential generator on the host."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

_MT_N = 624
_per_device = {}


class _DeviceState:
    """Per device: the jump table (built on first use), the call's scratch, and a pinned host / device pair for the
    generator state (key_in | key_out | pos_out)."""

    def __init__(self, device: torch.device):
        lib = _lib.load()
        jb, wb = C.c_size_t(0), C.c_size_t(0)
        _lib.check(lib.invpref_mt_jump_bytes(C.byref(jb), C.byref(wb)), "mt_jump_bytes")
        self.jumps = torch.empty(jb.value, dtype=torch.uint8, device=device)
        self.ws = torch.empty(wb.value, dtype=torch.uint8, device=device)
        self.state = torch.empty(2 * _MT_N + 2, dtype=torch.int32, device=device)
        self.host = torch.empty(2 * _MT_N + 2, dtype=torch.int32, pin_memory=True)
        _lib.check(lib.invpref_mt_build_jumps(_lib.ptr(self.jumps), jb.value, _lib.stream_ptr()), "mt_build_jumps")


def _state_for(device: torch.device) -> _DeviceState:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    st = _per_device.get(idx)
    if st is None:
        with torch.cuda.device(idx):
            st = _per_device[idx] = _DeviceState(torch.device("cuda", idx))
    return st


def jump_table_bytes(device=None) -> int:
    """Device bytes this module holds for `device` (jump table + scratch + state), 0 before its first draw there."""
    if device is None:
        return sum(s.jumps.numel() + s.ws.numel() + s.state.numel() * 4 for s in _per_device.values())
    d = torch.device(device)
    s = _per_device.get(d.index if d.index is not None else torch.cuda.current_device())
    return 0 if s is None else s.jumps.numel() + s.ws.numel() + s.state.numel() * 4


def device_randint(high: int, n: int, device, out: torch.Tensor = None) -> torch.Tensor:
    """``np.random.randint(0, high, n)`` drawn on `device` from numpy's global stream (1 <= high <= 2^32), which is
    advanced exactly as that call would advance it (``has_gauss`` / ``cached_gaussian`` are kept).  ``out``: optional
    contiguous int64 tensor of n elements on `device`.  One small copy each way and one stream synchronisation."""
    high, n = int(high), int(n)
    if not 1 <= high <= 1 << 32:
        raise ValueError(f"high must be in [1, 2^32] (numpy's 32-bit path), got {high}")
    if n < 0:
        raise ValueError(f"n must be >= 0, got {n}")
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("device_randint draws on a CUDA device only (no CPU fallback)")
    name, key, pos, has_gauss, gauss = np.random.get_state()
    if name != "MT19937":
        raise RuntimeError(f"numpy's global generator is {name}, not MT19937")
    st = _state_for(device)
    if out is None:
        out = torch.empty(n, dtype=torch.int64, device=device)
    elif out.dtype != torch.int64 or out.numel() != n or out.device != st.state.device:
        raise ValueError("out must be an int64 tensor of n elements on the device")
    with torch.cuda.device(st.state.device):
        st.host[:_MT_N].copy_(torch.from_numpy(np.ascontiguousarray(key, dtype=np.uint32).view(np.int32)))
        st.state[:_MT_N].copy_(st.host[:_MT_N], non_blocking=True)
        base = st.state.data_ptr()
        _lib.check(_lib.load().invpref_mt_randint(
            C.c_void_p(base), int(pos), high, n, _lib.ptr(out), C.c_void_p(base + 4 * _MT_N),
            C.c_void_p(base + 8 * _MT_N), _lib.ptr(st.jumps), _lib.ptr(st.ws), st.ws.numel(), _lib.stream_ptr()),
            "mt_randint")
        st.host[_MT_N:2 * _MT_N + 1].copy_(st.state[_MT_N:2 * _MT_N + 1], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        new_key = st.host[_MT_N:2 * _MT_N].numpy().view(np.uint32).copy()
        new_pos = int(st.host[2 * _MT_N])
    np.random.set_state((name, new_key, new_pos, has_gauss, gauss))
    return out
