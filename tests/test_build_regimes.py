"""Index build at the edges of the TMA kernel's compaction regimes, and past its first persistent wave.

`compact_sub` (csrc/index_build_tma.cu) takes one of three paths per sub-tile, chosen by the number of entries the
sub-tile emits (`cnt`) and the parity of its first output slot (`head`): the sparse expansion loop (cnt below 3 entries
per 32-byte group), one staging round (cnt + head <= kStageCap) or several dense rounds of kStageCap entries.  CSV-shaped
inputs keep every sub-tile in one of the first two, so the regime stream below builds the input sub-tile by sub-tile
with an exact count at every regime edge, both head parities, both entry quote parities and three placements, and
asserts against the oracle that it did.  The multi-wave inputs are long enough for every resident CTA to process
several super-tiles, which cycles the hand-off rings and the barrier phases, compacts a pending super-tile while the
next is classified, and walks the look-back through several windows; they go through every build entry point.

The geometry is read from the CUDA sources, so a retune moves the targets with it.  The generator's self-check and the
geometry parse run without a GPU."""
import os
import re

import numpy as np
import pytest

import csv_simd_b200 as cs
from oracle import oracle as O
from tests import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "csv_simd_b200", "csrc")


# ---- geometry ------------------------------------------------------------------------------------------------------
def _grab(path, pattern):
    with open(os.path.join(CSRC, path)) as f:
        m = re.search(pattern, f.read(), re.M)
    if m is None:
        raise AssertionError(f"pattern {pattern!r} not found in {path}: the test geometry no longer matches the kernel")
    return m


class Geometry:
    """Tile geometry of the TMA kernel's production shape (ShapeB), parsed from the sources."""

    def __init__(self):
        self.threads = int(_grab("internal.h", r"^constexpr int kThreads = (\d+);").group(1))
        self.bytes_per_thread = int(_grab("internal.h", r"^constexpr int kBytesPerThread = (\d+);").group(1))
        args = _grab("index_build_tma.cu", r"^using ShapeB = TmaShape<([\d,\s]+)>;").group(1)
        vals = [int(v) for v in args.split(",")]
        # TmaShape<kMinBlocks, kStageBufs, kStageCap, kSub, kSkew = 1, kWorkers = 8, kExpand = 0, kLook = 1>
        vals += [1, 8, 0, 1][len(vals) - 4:]
        self.min_blocks, self.stage_bufs, self.cap, self.sub_per_super, self.skew, self.workers, self.expand, _ = vals
        self.warp_max = 32 * self.bytes_per_thread           # entries one warp's 4 KiB can emit
        self.sub = self.workers * self.warp_max              # bytes per sub-tile (one compact_sub call)
        self.super = self.sub_per_super * self.sub           # bytes per look-back descriptor
        self.sparse = 3 * (self.sub // 32)                   # compact_sub: cnt < 3 entries per 32-byte group

    def regime(self, cnt, head):
        """0 = sparse loop, 1 = one staging round, r >= 2 = r dense rounds (vectorised over numpy arrays)."""
        cnt = np.asarray(cnt, dtype=np.int64)
        rounds = -(-(cnt + head) // self.cap)
        return np.where(cnt < self.sparse, 0, np.maximum(rounds, 1))

    def wave_bytes(self, sms):
        return sms * self.min_blocks * self.super


G = Geometry()


def regime_name(r):
    return {0: "sparse", 1: "single round"}.get(int(r), f"dense, {int(r)} rounds")


def test_geometry_from_sources():
    assert G.threads * G.bytes_per_thread == cases.TILE         # the one-tile kernel's tile, which the suite sizes by
    assert G.sub <= 1 << 16 and G.cap + 8 <= 1 << 16           # 16-bit staging offsets and slots
    assert 0 < G.sparse < G.cap < G.sub                         # all three regimes exist
    assert G.super == G.sub_per_super * G.sub and G.expand == 2
    assert G.warp_max == 4096 and G.sub % G.warp_max == 0


# ---- regime generator ----------------------------------------------------------------------------------------------
SEPS = np.frombuffer(b",\n\r", dtype=np.uint8)
PLACEMENTS = ("spread", "packed", "end")


def _quoted_content(length, rng):
    """`length` bytes that stay inside a quoted span: separators, "" escapes, CR LF, text (an even number of quotes)."""
    toks = [b",", b'""', b"\r", b"\n", b"x", b'""', b",", b"\r\n"]
    out = bytearray()
    i = int(rng.integers(len(toks)))
    while len(out) < length:
        t = toks[i % len(toks)]
        i += 1
        out += t if len(out) + len(t) <= length else b"x"
    return np.frombuffer(bytes(out), dtype=np.uint8)


def make_subtile(pin, count, end_par, placement, rng):
    """One sub-tile entered with quote parity `pin` that emits exactly `count` entries and leaves with `end_par`
    (forced to 0 when there is no byte left for an opening quote).  Quoted spans at the start (pin = 1), at the end
    (end_par = 1) and in the middle hold separators that are not emitted; the emitted separators go where `placement`
    says among the remaining bytes.  Returns (bytes, end parity)."""
    S = G.sub
    room = S - count
    assert count <= S and room >= pin, (count, pin)
    if end_par and room - pin < 1:
        end_par = 0
    spare = room - pin - end_par
    lead = min(14, spare // 3) if pin else 0
    trail = min(14, spare // 3) if end_par else 0
    mid = 12 if spare - lead - trail >= 12 else 0
    b = np.full(S, ord("a"), dtype=np.uint8)
    free = np.ones(S, dtype=bool)
    if pin:                                  # the span the previous sub-tile opened, then its closing quote
        b[:lead] = _quoted_content(lead, rng)
        b[lead] = ord('"')
        free[:lead + 1] = False
    if end_par:                              # an opening quote whose span runs into the next sub-tile
        b[S - 1 - trail] = ord('"')
        b[S - trail:] = _quoted_content(trail, rng)
        free[S - 1 - trail:] = False
    if mid:
        m0 = S // 2 - mid // 2
        b[m0] = b[m0 + mid - 1] = ord('"')
        b[m0 + 1:m0 + mid - 1] = _quoted_content(mid - 2, rng)
        free[m0:m0 + mid] = False
    avail = np.flatnonzero(free)
    assert avail.size >= count
    if placement == "spread":
        at = avail[(np.arange(count, dtype=np.int64) * avail.size) // max(count, 1)]
    elif placement == "packed":              # the fewest warps' 4 KiB that hold them
        at = avail[:count]
    else:                                    # packed at the end: offset S - 1 when the sub-tile ends outside quotes
        at = avail[avail.size - count:]
    b[at] = SEPS[rng.integers(0, SEPS.size, size=count)]
    return b, end_par


def regime_counts():
    """Every count at a regime edge of compact_sub, every further multiple of kStageCap, and the full sub-tile."""
    c = [0, 1, 2, G.sparse - 1, G.sparse, G.sparse + 1, G.cap - 1, G.cap, G.cap + 1, 2 * G.cap - 1, 2 * G.cap, 2 * G.cap + 1]
    c += list(range(3 * G.cap, G.sub, G.cap)) + [G.sub - 1, G.sub]
    return sorted(set(c))


def tally(data, index=None, out_base=1):
    """Per sub-tile of `data` as the TMA kernel sees it in a build whose first entry goes to slot `out_base`:
    (entries emitted, head parity, entry quote parity, regime), from the oracle's index."""
    a = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    if index is None:
        index = O.closed_form_numpy(a)
    nsub = -(-a.size // G.sub)
    cnt = np.bincount((index[1:] // np.uint64(G.sub)).astype(np.int64), minlength=nsub)
    q = np.bincount(np.flatnonzero(a == 0x22) // G.sub, minlength=nsub)
    pin = (np.cumsum(q) - q) & 1
    head = (out_base + np.cumsum(cnt) - cnt) & 1
    return cnt, head, pin, G.regime(cnt, head)


def coverage_table(tallies):
    """Markdown table of sub-tiles per (regime, head) over several tallies."""
    rows = {}
    for _, head, _, reg in tallies:
        for r, h in zip(reg.tolist(), head.tolist()):
            rows.setdefault(r, [0, 0])[h] += 1
    lines = ["| regime | head 0 | head 1 |", "|---|---|---|"]
    for r in range(0, max(rows) + 1):
        h0, h1 = rows.get(r, [0, 0])
        lines.append(f"| {regime_name(r)} | {h0} | {h1} |")
    return "\n".join(lines)


class RegimeStream:
    """Sub-tiles at every (count, head, entry parity, placement) of regime_counts(), each behind a filler sub-tile of
    1 or 2 entries that sets its head, half of them at sub-tile 0 of a super-tile and half at a later one; quoted
    spans run across sub-tile and super-tile edges.  The constructor checks the result against the oracle."""

    def __init__(self, seed=0):
        rng = np.random.default_rng(seed)
        parts, plan = [], []
        entries, pin, k = 0, 0, 0       # entries so far (without the sentinel), quote parity, targets planned
        for count in regime_counts():
            for want_pin in (0, 1):
                if want_pin and count == G.sub:
                    continue            # every byte a separator: the sub-tile cannot be entered inside quotes
                for head in (0, 1):
                    for placement in PLACEMENTS:
                        want_sub = k % G.sub_per_super
                        while (len(parts) + 1) % G.sub_per_super != want_sub:   # pad to place the target
                            b, pin = make_subtile(pin, 7, int(rng.integers(2)), "spread", rng)
                            parts.append(b)
                            entries += 7
                        fill = 1 if (1 + entries + 1) & 1 == head else 2
                        b, pin = make_subtile(pin, fill, want_pin, "spread", rng)
                        assert pin == want_pin
                        parts.append(b)
                        entries += fill
                        end_par = 0 if placement == "end" else (k // 3) % 2
                        b, pin = make_subtile(want_pin, count, end_par, placement, rng)
                        plan.append((len(parts), count, head, want_pin, placement))
                        parts.append(b)
                        entries += count
                        k += 1
        b, pin = make_subtile(pin, 3, 0, "spread", rng)    # the last target is not the last sub-tile
        parts.append(b)
        self.subtiles = np.stack(parts)
        self.data = self.subtiles.ravel()
        self.plan = plan
        self.index = O.closed_form_numpy(self.data)
        self.check()

    def check(self):
        cnt, head, pin, reg = tally(self.data, self.index)
        total = np.bincount(np.flatnonzero(np.isin(self.data, SEPS)) // G.sub, minlength=cnt.size)
        last = set((self.index[1:][(self.index[1:] % np.uint64(G.sub)) == G.sub - 1] // np.uint64(G.sub)).tolist())
        for i, count, h, p, placement in self.plan:
            assert (cnt[i], head[i], pin[i]) == (count, h, p), (i, count, h, p, placement)
            if G.sub - count >= 40:
                assert total[i] > count, (i, count)          # separators inside quotes too: c0 != c1
            if placement == "end" and count > 0:
                assert i in last, (i, count)                 # an entry at offset sub-tile - 1
        return cnt, head, pin, reg


@pytest.fixture(scope="module")
def regime():
    return RegimeStream()


def test_regime_generator_self_check(regime):
    cnt, head, pin, reg = regime.check()
    targets = np.array([i for i, *_ in regime.plan])
    assert len(regime.plan) == len(regime_counts()) * 2 * 2 * len(PLACEMENTS) - 2 * len(PLACEMENTS)
    realised = set(zip(reg[targets].tolist(), head[targets].tolist(), pin[targets].tolist()))
    rounds = -(-(G.sub + 1) // G.cap)
    for r in range(0, rounds + 1):
        for h in (0, 1):
            for p in (0, 1):
                assert (r, h, p) in realised, (regime_name(r), h, p)
    subpos = targets % G.sub_per_super
    assert set(subpos[pin[targets] == 1].tolist()) == set(range(G.sub_per_super))
    assert (pin[::G.sub_per_super] == 1).any()                    # a quoted span across a super-tile edge
    assert regime.data.size % 128 == 0 and regime.data.size < (24 << 20)


def test_regime_stream_shuffled_keeps_regimes(regime):
    data = shuffled_stream(regime, 2 * regime.data.size + 77, seed=1)
    cnt, head, pin, reg = tally(data)
    assert data.size % 128 != 0
    assert set(zip(reg.tolist(), head.tolist())) == {(r, h) for r in range(-(-(G.sub + 1) // G.cap) + 1) for h in (0, 1)}


def shuffled_stream(regime, nbytes, seed):
    """The regime stream's sub-tiles repeated in shuffled order (heads and entry parities change with the order),
    cut to `nbytes`."""
    rng = np.random.default_rng(seed)
    reps = -(-nbytes // regime.data.size)
    order = np.concatenate([rng.permutation(len(regime.subtiles)) for _ in range(reps)])
    return regime.subtiles[order].ravel()[:nbytes].copy()


# ---- GPU: the regime stream through both kernels ------------------------------------------------------------------
def _build(c, data, flags=0):
    idx = c.index_build(data, flags)
    out = idx.to_host().copy()
    par = idx.end_parity
    idx.free()
    return out, par


@pytest.fixture(scope="module")
def forced_ctxs():
    out = {}
    for k in ("simple", "tma"):
        os.environ["CSVB200_KERNEL"] = k
        out[k] = cs.Context(0)
    os.environ.pop("CSVB200_KERNEL", None)
    yield out
    for c in out.values():
        c.close()


@pytest.mark.gpu
def test_regime_stream_vs_oracle(ctx, forced_ctxs, regime):
    data = np.concatenate([regime.data, np.frombuffer(b'x,"y\n",z\r\n' * 4 + b"tail,", dtype=np.uint8)])
    want = O.read_sse(data)
    par = int(np.count_nonzero(data == 0x22) & 1)
    for name, c in [("default", ctx)] + list(forced_ctxs.items()):
        got, p = _build(c, data)
        assert got.shape == want.shape and (got == want).all(), name
        assert p == par, name


# ---- GPU: inputs several persistent waves long, through every entry point -------------------------------------------
def _device_bytes(a, dev, misalign=0):
    """A device copy of `a` at an address that is 16-byte aligned and `misalign` bytes past a 128-byte boundary."""
    import torch
    buf = torch.zeros(a.size + 256, dtype=torch.uint8, device=dev)
    off = (-buf.data_ptr()) % 128 + misalign
    buf[off:off + a.size].copy_(torch.from_numpy(np.require(a, requirements="W")))
    torch.cuda.synchronize(dev)
    return buf, buf.data_ptr() + off


def _quoted_cut(a, near):
    """The first odd offset at or after `near` that lies inside a quoted span (None if there is none nearby)."""
    lo, hi = near, min(a.size, near + (1 << 20))
    before = int(np.count_nonzero(a[:lo] == 0x22))
    par = (before + np.cumsum(a[lo:hi] == 0x22) - (a[lo:hi] == 0x22)) & 1
    hits = np.flatnonzero((par == 1) & ((np.arange(lo, hi) & 1) == 1))
    return lo + int(hits[0]) if hits.size else None


class MultiWave:
    def __init__(self, regime, sms):
        self.wave = G.wave_bytes(sms)
        n = 4 * self.wave                          # the first wave and three more
        alt = np.zeros(n + 101, dtype=np.uint8)
        sep = np.random.default_rng(5).choice(SEPS, size=alt.size)
        body = np.full(alt.size, ord("b"), dtype=np.uint8)
        full = ((np.arange(alt.size) // G.super) & 1) == 0
        alt[:] = np.where(full, sep, body)          # alternating all-separator and separator-free super-tiles
        for k, pos in enumerate(range(G.super + 1000, alt.size - 8, alt.size // 7)):
            alt[pos:pos + 2] = (0xC3, 0xA9)         # a few valid two-byte sequences: some non-ASCII bitmap bits set
        alt[3 * self.wave + 12345] = 0xFF           # and one invalid byte in the last wave
        self.inputs = {
            "regime shuffled": shuffled_stream(regime, n + 45, seed=2),
            "random alphabet": np.frombuffer(cases.rand_bytes(n + 77, 61), dtype=np.uint8),
            "full random": np.frombuffer(cases.full_random(n + 13, 62), dtype=np.uint8),
            "separator super-tiles": alt,
        }
        self.want = {k: O.read_sse(a) for k, a in self.inputs.items()}


@pytest.fixture(scope="module")
def big_ctx():
    """Reserve one entry per byte: no capacity-overflow rebuild, so the chunked host pipeline stays on its own path."""
    c = cs.Context(0)
    c.set_reserve(1, 1)
    yield c
    c.close()


@pytest.fixture(scope="module")
def multi(regime):
    import torch
    return MultiWave(regime, torch.cuda.get_device_properties(0).multi_processor_count)


def _same(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    assert np.array_equal(got, want), (what, int(np.flatnonzero(got != want)[0]))


@pytest.mark.gpu
def test_multi_wave_host_and_device_builds(big_ctx, multi):
    import torch
    dev = torch.device("cuda", big_ctx.device)
    for name, a in multi.inputs.items():
        assert a.size >= 4 * multi.wave and a.size % 128 != 0
        want = multi.want[name]
        par = int(np.count_nonzero(a == 0x22) & 1)
        got, p = _build(big_ctx, a)
        _same(got, want, (name, "host"))
        assert p == par
        buf, ptr = _device_bytes(a, dev, misalign=16)
        idx = big_ctx.index_build_device(ptr, a.size)
        _same(idx.to_host(), want, (name, "device, 16 bytes past a 128-byte boundary"))
        assert idx.end_parity == par
        idx.free()
        del buf


@pytest.mark.gpu
def test_multi_wave_build_validate(big_ctx, multi):
    import torch
    dev = torch.device("cuda", big_ctx.device)
    nl = np.array([0x0D, 0x0A], dtype=np.uint8)
    for name, a in multi.inputs.items():
        want = multi.want[name]
        buf, ptr = _device_bytes(a, dev)
        idx = big_ctx.index_build_device(ptr, a.size, cs.BUILD_VALIDATE)
        _same(idx.to_host(), want, (name, "validate"))
        is_ascii, newlines = idx.validation()
        assert is_ascii == O.is_ascii(a), name
        assert newlines == int(np.isin(a[want[1:].astype(np.int64)], nl).sum()), name
        assert idx.validate_utf8() == O.utf8_valid_up_to(a), name    # reads only the tiles the bitmap flags
        idx.free()
        del buf


@pytest.mark.gpu
def test_multi_wave_build_to_host(big_ctx, multi):
    for name, a in multi.inputs.items():
        want = multi.want[name]
        out = np.zeros(want.size + 16, dtype=np.uint64)
        ln = big_ctx.index_build_to_host(a.ctypes.data, a.size, out.ctypes.data, out.size)   # 64 MiB chunks
        assert ln == want.size, name
        _same(out[:ln], want, (name, "to_host"))


@pytest.mark.gpu
def test_multi_wave_shard_chain(big_ctx, multi):
    import torch
    dev = torch.device("cuda", big_ctx.device)
    carried = 0
    for name, a in multi.inputs.items():
        n = a.size
        c1 = (n // 3) // G.sub * G.sub + (1 if len(name) & 1 else -1)      # a sub-tile edge +- 1
        c2 = _quoted_cut(a, 2 * n // 3) or (2 * n // 3) | 1
        cuts = [0, c1, c2, n]
        segs, par = [], 0
        for k in range(3):
            lo, hi = cuts[k], cuts[k + 1]
            buf, ptr = _device_bytes(a[lo:hi], dev)
            p = big_ctx.shard_quote_parity(ptr, hi - lo)
            assert p == int(np.count_nonzero(a[lo:hi] == 0x22) & 1)
            if k == 2:
                carried += par
            idx = big_ctx.index_build_shard_device(ptr, hi - lo, par, lo, emit_sentinel=(k == 0))
            segs.append(idx.to_host().copy())
            assert idx.end_parity == par ^ p
            idx.free()
            del buf
            par ^= p
        _same(np.concatenate(segs), multi.want[name], (name, "shards", cuts))
    assert carried == 3          # the cut inside a quoted span: carry 1 at an odd global offset


@pytest.mark.gpu
def test_multi_wave_exchange_emulated_ranks(multi):
    """The exchange form (prediction, build, in-kernel exchange, conditional redo) with two ranks on one GPU; rank 1's
    shard is more than three waves long."""
    import torch
    dev = torch.device("cuda", 0)
    name = "regime shuffled"
    a = multi.inputs[name]
    cut = _quoted_cut(a, a.size // 8)
    assert cut is not None and a.size - cut >= 3 * multi.wave
    cuts = [0, cut, a.size]
    ctxs = [cs.Context(0) for _ in range(2)]
    exs = [c.exchange(k, 2) for k, c in enumerate(ctxs)]
    cs.Exchange.connect_local(exs)
    try:
        idxs, infos, keep = [], [], []
        for k in range(2):
            buf, ptr = _device_bytes(a[cuts[k]:cuts[k + 1]], dev)
            keep.append(buf)
            idx = ctxs[k].index_build_shard_exchange(exs[k], ptr, cuts[k + 1] - cuts[k], cuts[k])
            infos.append(idx.shard_info())       # synchronises: rank 0 has posted before rank 1 starts
            idxs.append(idx)
        got = np.concatenate([i.to_host() for i in idxs])
        _same(got, multi.want[name], "exchange")
        assert [i["carry_in"] for i in infos] == [0, 1]
        assert [i["base"] for i in infos] == [0, infos[0]["entries"]]
        assert sum(i["entries"] for i in infos) == multi.want[name].size
        for i in idxs:
            i.free()
    finally:
        for e in exs:
            e.close()
        for c in ctxs:
            c.close()


@pytest.mark.gpu
def test_unsynchronised_chain_on_one_context(regime, multi):
    """Five device builds enqueued back to back on one context with nothing synchronised in between: B has A's size
    and finds A's descriptors in the shared scratch under A's tag, D is larger than everything before it so the
    scratch is reallocated mid-chain, E rebuilds A's bytes."""
    import torch
    dev = torch.device("cuda", 0)
    c = cs.Context(0)
    c.set_reserve(1, 1)            # an overflow rebuild would synchronise
    try:
        size = (96 << 20) + 45
        ins = {"A": shuffled_stream(regime, size, seed=7), "B": shuffled_stream(regime, size, seed=8),
               "C": np.frombuffer(cases.rand_bytes((20 << 20) + 3, 63), dtype=np.uint8),
               "D": multi.inputs["regime shuffled"]}
        assert ins["D"].size > size
        bufs = {k: _device_bytes(a, dev) for k, a in ins.items()}
        ins["E"], bufs["E"] = ins["A"], bufs["A"]
        idxs = {k: c.index_build_device(bufs[k][1], ins[k].size) for k in "ABCDE"}
        for k in "ABCDE":
            want = multi.want["regime shuffled"] if k == "D" else O.read_sse(ins[k])
            _same(idxs[k].to_host(), want, k)
            assert idxs[k].end_parity == int(np.count_nonzero(ins[k] == 0x22) & 1), k
        for i in idxs.values():
            i.free()
    finally:
        c.close()
