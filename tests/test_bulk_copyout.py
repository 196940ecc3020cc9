"""The compact (u32) index build ships each sub-tile's run of entries with one bulk store of its 16-byte-aligned
middle and plain stores for the at most 3 + 3 entries around it, staging in the TMA ring slot it has just classified
(`compact_sub_bulk`, csrc/index_build_tma.cu).  Denser sub-tiles than one slot holds (8192 u32 entries) take several
rounds.  The stream below puts every sub-tile run length of interest at all four alignments of its first slot
(`g0 & 3`), at sub-tile 0 and 1 of a super-tile; the builds go through the default (u32) context, the one-tile kernel
and an 8-byte context, each against the oracle.  The stream's self-check runs without a GPU."""
import os

import numpy as np
import pytest

import csv_simd_b200 as cs
from oracle import oracle as O
from tests.test_build_regimes import G, SEPS, _device_bytes, make_subtile

SLOT = G.sub // 4                  # u32 entries a 32 KiB ring slot holds
DENSE = SLOT - 3                   # the most entries a sub-tile ships in one round at every alignment


def run_counts():
    """Runs without an aligned middle (0-8 entries), the sparse-loop edge, one round at its edge, and dense rounds at
    and around every multiple of a slot."""
    c = list(range(0, 9)) + [11, 12, G.sparse - 1, G.sparse, 5000]
    for k in range(1, 5):
        c += [k * SLOT - 4, k * SLOT - 3, k * SLOT - 2, k * SLOT - 1, k * SLOT, k * SLOT + 1]
    return sorted(x for x in set(c) if 0 <= x <= G.sub)


class AlignStream:
    """Each target sub-tile (count, first-slot alignment, quote parity on entry, placement) behind a filler sub-tile of
    1-4 entries that sets its alignment; half the targets at sub-tile 0 of a super-tile, half at sub-tile 1."""

    def __init__(self, seed=0, out_base=1):
        rng = np.random.default_rng(seed)
        parts, plan = [], []
        entries, pin, k = 0, 0, 0
        for count in run_counts():
            for head in range(4):
                for placement in ("spread", "end"):
                    want_pin = 0 if count == G.sub else k % 2
                    while (len(parts) + 1) % G.sub_per_super != k % G.sub_per_super:
                        b, pin = make_subtile(pin, 4, int(rng.integers(2)), "spread", rng)   # 4 entries: alignment kept
                        parts.append(b)
                        entries += 4
                    fill = 1 + (head - (out_base + entries + 1)) % 4
                    b, pin = make_subtile(pin, fill, want_pin, "spread", rng)
                    parts.append(b)
                    entries += fill
                    b, pin = make_subtile(want_pin, count, 0 if placement == "end" else (k // 2) % 2, placement, rng)
                    plan.append((len(parts), count, head))
                    parts.append(b)
                    entries += count
                    k += 1
        b, pin = make_subtile(pin, 3, 0, "spread", rng)
        parts.append(b)
        self.subtiles = np.stack(parts)
        self.data = self.subtiles.ravel()
        self.plan = plan
        self.out_base = out_base
        self.index = O.closed_form_numpy(self.data)

    def check(self):
        cnt = np.bincount((self.index[1:] // np.uint64(G.sub)).astype(np.int64), minlength=len(self.subtiles))
        g0 = (self.out_base + np.cumsum(cnt) - cnt) & 3
        for i, count, head in self.plan:
            assert (cnt[i], g0[i]) == (count, head), (i, count, head)
        return cnt, g0


@pytest.fixture(scope="module")
def stream():
    return AlignStream()


def test_align_stream_self_check(stream):
    cnt, g0 = stream.check()
    targets = np.array([i for i, *_ in stream.plan])
    got = set(zip(cnt[targets].tolist(), g0[targets].tolist()))
    assert got == {(c, h) for c in run_counts() for h in range(4)}
    ends = (g0[targets] + cnt[targets]) % 4 == 0
    assert ends.sum() >= len(run_counts())                      # runs that end on a 16-byte boundary
    assert (cnt[targets] + g0[targets] > SLOT).any()            # dense rounds
    assert set((targets % G.sub_per_super).tolist()) == set(range(G.sub_per_super))
    assert stream.data.size < (32 << 20)


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _make_ctx(kernel=None, entry_bytes=None):
    saved = {k: os.environ.get(k) for k in ("CSVB200_KERNEL", "CSVB200_INDEX_ENTRY_BYTES")}
    try:
        for k, v in (("CSVB200_KERNEL", kernel), ("CSVB200_INDEX_ENTRY_BYTES", entry_bytes)):
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        return cs.Context(0)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def ctxs():
    out = {"default": _make_ctx(), "simple": _make_ctx("simple"), "u64": _make_ctx(entry_bytes="8")}
    for c in out.values():
        c.set_reserve(1, 1)
    yield out
    for c in out.values():
        c.close()


def _check(c, data, want, what):
    idx = c.index_build(data)
    got = idx.to_host()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    assert np.array_equal(got, want), (what, int(np.flatnonzero(got != want)[0]))
    assert idx.end_parity == int(np.count_nonzero(data == 0x22) & 1), what
    idx.free()


@pytest.mark.gpu
def test_align_stream_vs_oracle(ctxs, stream):
    want = O.read_sse(stream.data)
    for name, c in ctxs.items():
        _check(c, stream.data, want, name)


@pytest.mark.gpu
def test_align_stream_device_build_several_waves(ctxs, stream):
    """Shuffled repetitions of the stream, four persistent waves and more: every CTA hands its ring slots back
    through many bulk stores, at every alignment."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 4 * G.wave_bytes(sms) + 333
    rng = np.random.default_rng(3)
    reps = -(-n // stream.data.size)
    order = np.concatenate([rng.permutation(len(stream.subtiles)) for _ in range(reps)])
    data = stream.subtiles[order].ravel()[:n].copy()
    want = O.read_sse(data)
    dev = torch.device("cuda", 0)
    for name, c in ctxs.items():
        buf, ptr = _device_bytes(data, dev, misalign=48)
        idx = c.index_build_device(ptr, data.size)
        got = idx.to_host()
        assert got.shape == want.shape and np.array_equal(got, want), name
        idx.free()
        del buf


@pytest.mark.gpu
def test_capacity_inside_bulk_range(stream):
    """A reservation that runs out inside a sub-tile's bulk range (at every alignment of the capacity): the first launch
    writes nothing at or past it, the rebuild is exact, and an index allocated before it stays intact."""
    dense = np.frombuffer(b",\n" * (3 << 20), dtype=np.uint8)     # one entry per byte: capacity n / 64 + 4096 overflows
    for name, kw in (("default", {}), ("u64", {"entry_bytes": "8"})):
        c = _make_ctx(**kw)
        try:
            keep = c.index_build(stream.data)
            keep_want = O.read_sse(stream.data)
            c.set_reserve(1, 64)
            for extra in range(4):
                data = np.concatenate([dense, np.full(64 * extra, ord(","), dtype=np.uint8)])
                _check(c, data, O.read_sse(data), (name, extra))
            assert np.array_equal(keep.to_host(), keep_want), name
            keep.free()
        finally:
            c.close()
