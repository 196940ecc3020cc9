"""A context created with CSVB200_DBG_TIMELINE=1 runs its device-resident builds through the instrumented kernel and
grows a timeline buffer with them.  Growing it must leave the context's other buffers alone: the pinned staging of the
small zero-copy path (csvb200_index_build_to_host up to 256 KiB) has to stay valid for the next small call."""
import ctypes as C

import numpy as np
import pytest

import csv_simd_b200 as cs
from oracle import oracle as O
from tools import gen

pytestmark = pytest.mark.gpu


def small_builds_match_oracle(ctx, inputs, h_out):
    for a in inputs:
        want = O.read_sse(a)
        out = np.zeros(want.size + 8, dtype=np.uint64)
        ln = ctx.index_build_to_host(a.ctypes.data, a.size, out.ctypes.data, out.size)          # pageable destination
        assert ln == want.size and (out[:ln] == want).all(), a.size
        h_out.zero_()
        ln = ctx.index_build_to_host(a.ctypes.data, a.size, h_out.data_ptr(), h_out.numel())    # pinned: written in place
        assert ln == want.size and (h_out.numpy()[:ln].view(np.uint64) == want).all(), a.size


def test_timeline_growth_keeps_small_path_buffers(monkeypatch):
    import torch
    monkeypatch.setenv("CSVB200_DBG_TIMELINE", "1")   # read when the context is created
    ctx = cs.Context(0)
    try:
        lib = cs._lib.load()
        lib.csvb200_debug_timeline.restype = C.c_int
        lib.csvb200_debug_timeline.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        q, _ = gen.quoted(256 << 10, seed=61)
        small = [q[:size] for size in (64, 1000, 32769, 100000, 256 << 10)]
        h_out = torch.zeros((256 << 10) + 64, dtype=torch.int64).pin_memory()
        small_builds_match_oracle(ctx, small, h_out)   # the small path allocates its pinned buffers

        words = []
        for size in (1 << 20, 8 << 20):                # two device builds of growing size: the timeline grows twice
            data, _ = gen.quoted(size, seed=62)
            n = int(data.size)
            d = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
            d[:n].copy_(torch.from_numpy(data))
            torch.cuda.synchronize()
            idx = ctx.index_build_device(d.data_ptr(), n)
            assert (idx.to_host() == O.read_sse(data)).all()
            idx.free()
            w = C.c_size_t()
            lib.csvb200_debug_timeline(ctx._h, None, 0, C.byref(w))
            words.append(w.value)
            del d
        assert 0 < words[0] < words[1]

        small_builds_match_oracle(ctx, small, h_out)

        buf = np.zeros(words[-1], dtype=np.uint64)
        w = C.c_size_t()
        assert lib.csvb200_debug_timeline(ctx._h, buf.ctypes.data, buf.size, C.byref(w)) == 0
        assert w.value == words[-1]
        tiles = (n + (64 << 10) - 1) // (64 << 10)     # 64 KiB super-tiles of the TMA kernel
        t = buf[:tiles * 8].reshape(tiles, 8)
        assert (t[:, 0] != 0).all() and (t[:, 1] != 0).all()   # every super-tile stamped its aggregate and its prefix
    finally:
        ctx.close()
