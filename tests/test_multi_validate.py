"""csvb200_multi_tape_validate, csvb200_multi_validate_utf8 and csvb200_multi_tape_chunks: validation and chunks of a
distributed index.  Every result must equal, field for field, what the one-GPU call gives on an index of the same bytes,
and what the oracle gives where it has a definition.  Device 0 listed several times runs the whole path on one GPU; the
cross-device variants run it over real devices.  The cuts go where the seams must be handled exactly: between a CR and
its LF, on either side of a bad separator, across empty shards and shards of 0-3 bytes, inside multi-byte sequences and
right before a lead whose continuation bytes lie in the next shard."""
import ctypes as C

import numpy as np
import pytest

import csv_simd_b200 as cs
from csv_simd_b200 import _lib
from csv_simd_b200.errors import InvalidState
from oracle import oracle as O
from tests.conftest import golden_bytes
from tools import gen

pytestmark = pytest.mark.gpu

U64MAX = 0xFFFFFFFFFFFFFFFF


class Multis:
    """One csvb200_multi per shard count, reused over the cases.  The input goes in from pinned memory, so that no
    context of them sets up a staging ring for pageable uploads."""

    def __init__(self, devices_for):
        self.devices_for, self.cache, self.pinned = devices_for, {}, None

    def index(self, raw, cuts):
        import torch
        g = 4 if cuts is None else len(cuts) - 1
        if g not in self.cache:
            self.cache[g] = cs.Multi(self.devices_for(g))
        if len(raw):
            self.pinned = torch.frombuffer(bytearray(raw), dtype=torch.uint8).pin_memory()
            raw = self.pinned.numpy()
        return self.cache[g].index_build_distributed(raw, cuts)

    def close(self):
        for m in self.cache.values():
            m.close()


@pytest.fixture
def one_gpu(ctx):
    ms = Multis(lambda g: [ctx.device] * g)
    yield ms
    ms.close()


@pytest.fixture
def across_gpus(ctx):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs at least 2 GPUs")
    ms = Multis(lambda g: [k % ndev for k in range(g)])
    yield ms
    ms.close()


# ---- tape validation --------------------------------------------------------------------------------------------------
def _check_tape(ctx, ms, raw, cuts, field_cnt, crlf, oracle=True):
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    want = idx.tape_validate(field_cnt, crlf)
    host = idx.to_host()
    idx.free()
    mi = ms.index(raw, cuts)
    assert (mi.to_host() == host).all()
    got = mi.tape_validate(field_cnt, crlf)
    mi.free()
    assert got == want, (cuts, got, want)
    if oracle:
        assert got["first_bad_slot"] == O.tape_first_bad_slot(raw, host, field_cnt, crlf)
    return got, host


def _rows(n, nl):
    return nl.join([b"c0,c1,c2"] + [b"%d,%d,%d" % (i, i * 7, i * 13) for i in range(n)]) + nl


def _crlf_cuts(raw, at):
    """cuts between the CR and the LF of the line ends found after each byte offset in `at`"""
    return [raw.index(b"\r\n", a) + 1 for a in at]


def _run_tape_seams(ctx, ms):
    for crlf in (False, True):
        nl = b"\r\n" if crlf else b"\n"
        good = _rows(400, nl)
        n = len(good)
        if crlf:
            c = _crlf_cuts(good, [n // 5, n // 2, 3 * n // 4])
            cut_sets = [[0] + c + [n], [0, c[0], c[0], c[1], c[1], c[1], c[2], n], [0, c[0] - 1, c[0], c[0] + 1, n]]
        else:
            cut_sets = [None, [0, n // 3, n // 3, 2 * n // 3, n], [0, 1, 2, 2, 3, n // 2, n]]
        for cuts in cut_sets:
            rep, _ = _check_tape(ctx, ms, good, cuts, 3, crlf)
            assert rep["ok"] == 1
        if crlf:
            # the pair broken: "\r \n" keeps the separator count, and the LF no longer follows its CR; cut between the CR
            # and the space, between the space and the LF, and with empty shards in between
            row = good.index(b"\r\n", n // 2)
            broken = good[:row] + b"\r \n" + good[row + 2:]
            nb = len(broken)
            for cuts in ([0, row + 1, nb], [0, row + 2, nb], [0, row + 1, row + 1, row + 2, row + 2, nb],
                         [0, row + 1, row + 2, row + 3, nb], None):
                rep, _ = _check_tape(ctx, ms, broken, cuts, 3, True)
                assert rep["ok"] == 0 and rep["first_bad_slot"] != U64MAX
        # the trailing partial row, without and with a bad slot before it
        tail = good + b"7,8"
        for cuts in (None, [0, len(good) - 1, len(good), len(good) + 1, len(tail)]):
            rep, _ = _check_tape(ctx, ms, tail, cuts, 3, crlf)
            assert rep["problem"] != 0 and rep["first_bad_slot"] == U64MAX and rep["ok"] == 0
            swapped = tail.replace(b"10,70,130", b"10\n70,130", 1)
            rep, _ = _check_tape(ctx, ms, swapped, cuts, 3, crlf)
            assert rep["problem"] != 0 and rep["first_bad_slot"] != U64MAX


def _swap(raw, host, s):
    """raw with the separator of slot s swapped between ',' and LF (the index stays the same)"""
    b = bytearray(raw)
    p = int(host[s])
    b[p] = 0x0A if b[p] == 0x2C else 0x2C
    return bytes(b)


def _run_bad_slot_places(ctx, ms):
    for crlf in (False, True):
        good = _rows(500, b"\r\n" if crlf else b"\n")
        idx = ctx.index_build(good)
        host = idx.to_host()
        idx.free()
        n, jump = len(good), 4 if crlf else 3
        s = 150 * jump + 2                                      # a field separator in the middle of the file
        e = 300 * jump + 1
        for name, bad_slots, cuts in (
            ("first of a segment", [s], [0, int(host[s]), n]),
            ("first of a segment behind empty ones", [s], [0, int(host[s]), int(host[s]), int(host[s]), n]),
            ("last of a segment", [s], [0, int(host[s]) + 1, n]),
            ("slot 1", [1], [0, 1, int(host[1]) + 1, n // 2, n]),
            ("slot 1, alone in its segment", [1], [0, int(host[1]), int(host[1]) + 1, n]),
            ("several segments: the lowest wins", [e, s, e + 50 * jump],
             [0, int(host[s]) - 3, int(host[e]), int(host[e + 50 * jump]) + 1, n]),
            ("several segments, lowest as first of a segment", [s, e], [0, int(host[s]), int(host[e]), n]),
        ):
            raw = good
            for b in bad_slots:
                raw = _swap(raw, host, b)
            rep, _ = _check_tape(ctx, ms, raw, cuts, 3, crlf)
            assert rep["first_bad_slot"] == min(bad_slots), name
            assert rep["first_bad_pos"] == int(host[min(bad_slots)]), name


def _run_large_random(ctx, ms):
    data, _ = gen.unquoted(8 << 20, seed=9)
    raw = bytearray(data.tobytes())
    idx = ctx.index_build(bytes(raw))
    host = idx.to_host()
    idx.free()
    rng = np.random.default_rng(3)
    for t in range(4):
        s = int(rng.integers(1, host.size))
        cuts = None if t % 2 == 0 else [0] + sorted(int(x) for x in rng.integers(0, len(raw), 5)) + [len(raw)]
        bad = _swap(bytes(raw), host, s)
        rep, _ = _check_tape(ctx, ms, bad, cuts, 16, False)
        assert rep["first_bad_slot"] == s


def test_tape_seams_on_one_gpu(ctx, one_gpu):
    _run_tape_seams(ctx, one_gpu)


def test_tape_seams_across_gpus(ctx, across_gpus):
    _run_tape_seams(ctx, across_gpus)


def test_tape_bad_slot_places_on_one_gpu(ctx, one_gpu):
    _run_bad_slot_places(ctx, one_gpu)


def test_tape_bad_slot_places_across_gpus(ctx, across_gpus):
    _run_bad_slot_places(ctx, across_gpus)


def test_tape_large_random_swaps(ctx, one_gpu):
    _run_large_random(ctx, one_gpu)


def test_tape_validate_status_codes(ctx, one_gpu):
    raw = _rows(50, b"\n")
    mi = one_gpu.index(raw, [0, 10, len(raw)])
    with pytest.raises(ValueError):
        mi.tape_validate(0, False)
    assert b"field_cnt" in mi._lib.csvb200_multi_last_error(mi.multi._h)
    mi.free()
    # CRLF with no fields (jump 1): the one-GPU kernel and the oracle already disagree on this degenerate row shape (they
    # report slots 3 and 1), so the distributed call is held to the one-GPU call alone
    _check_tape(ctx, one_gpu, raw, [0, 10, len(raw)], 0, True, oracle=False)


# ---- UTF-8 ------------------------------------------------------------------------------------------------------------
def _check_utf8(ctx, ms, raw, cuts):
    want = ctx.validate_utf8(raw)
    assert want == (O.utf8_valid_up_to(raw), O.is_ascii(raw))
    mi = ms.index(raw, cuts)
    got = mi.validate_utf8()
    mi.free()
    assert got == want, (cuts, got, want, raw[:200])
    return got


# boundary code points of every sequence length
SEQS = [chr(c).encode() for c in (0x80, 0x7FF, 0x800, 0xFFF, 0x1000, 0xD7FF, 0xE000, 0xFFFD, 0xFFFF, 0x10000, 0x3FFFF,
                                    0x40000, 0xFFFFF, 0x100000, 0x10FFFF, 0xE9, 0x20AC, 0x1F642)]


def _run_utf8_seams(ctx, ms):
    # every valid 2-, 3- and 4-byte sequence kind, with a cut at each of its interior positions and at both edges
    for seq in SEQS:
        for pad in (0, 1, 2, 3, 5):
            raw = b"a" * pad + seq + b"z,"
            for p in range(len(seq) + 1):
                assert _check_utf8(ctx, ms, raw, [0, pad + p, len(raw)])[0] is None
            inner = [pad + p for p in range(1, len(seq))]
            assert _check_utf8(ctx, ms, raw, [0] + inner + [len(raw)])[0] is None          # every interior cut at once
            assert _check_utf8(ctx, ms, raw, [0] + sorted(inner * 2) + [len(raw)])[0] is None
    # every code point of every length in one text, cut at random places
    text = "".join(chr(c) for c in range(0x80, 0x110000) if not 0xD800 <= c <= 0xDFFF).encode()
    rng = np.random.default_rng(21)
    for _ in range(2):
        assert _check_utf8(ctx, ms, text, [0] + sorted(int(x) for x in rng.integers(0, len(text), 15)) + [len(text)])[0] is None
    # the crafted invalid cases of the one-GPU test, with a cut at every byte around them
    crafted = [b"ab\xe2\x82", b"ab\xc0\xaf", b"\xed\xa0\x80", b"a\x80", b"\xf4\x90\x80\x80", b"\xf0\x8f\xbf\xbf",
               b"\xe0\x9f\xbf", b"\xc2", b"x\xf0\x9f\x99", b"\xf5\x80\x80\x80", b"\xff", b"\xc2\x80\x80",
               b"\xe1\x80\xc2\x80", b"ok\xe2\x82\xac\xe2\x82\xac\x80", b"\xf0\x9f\x99\x82" * 5 + b"\xbf"]
    for c in crafted:
        for pad, tail in ((0, b""), (13, b"tail,more\n"), (33, b"")):
            raw = b"x" * pad + c + tail
            n = len(raw)
            around = [p for p in range(max(0, pad - 3), min(n, pad + len(c) + 4))]
            for p in around:
                _check_utf8(ctx, ms, raw, [0, p, n])
            _check_utf8(ctx, ms, raw, [0] + [p for p in around if p > 0][:14] + [n])            # shards of one byte
            _check_utf8(ctx, ms, raw, [0] + sorted([p for p in around if p > 0][:7] * 2) + [n])   # and empty ones
    # a sequence truncated at the end of the last shard
    for raw in (b"abc\xe2\x82", b"abc\xf0\x9f\x99", b"abc\xc3"):
        for cuts in ([0, 3, len(raw)], [0, len(raw) - 1, len(raw)], [0, 2, 3, 4, 4, len(raw)]):
            assert _check_utf8(ctx, ms, raw, cuts)[0] == 3
    # a shard made only of continuation bytes: completing a sequence (valid), and stray after a complete one
    smile = "\U0001F642".encode()
    raw = b"x" + smile + b"y"
    assert _check_utf8(ctx, ms, raw, [0, 2, 5, len(raw)])[0] is None
    raw = b"x" + smile + b"\x80\x80\x80" + b"y"
    assert _check_utf8(ctx, ms, raw, [0, 5, 8, len(raw)])[0] == 5
    assert _check_utf8(ctx, ms, raw, [0, 2, 5, 8, len(raw)])[0] == 5
    # an ASCII shard followed by a lead whose continuation bytes lie past the 3-byte halo of that shard: the lead is the
    # next shard's to judge, here it is look-ahead only
    for seq in (smile, "€".encode(), "é".encode()):
        raw = b"ab,cd" + seq + seq + b"\n"
        assert _check_utf8(ctx, ms, raw, [0, 5, len(raw)]) == (None, False)
        assert _check_utf8(ctx, ms, raw, [0, 5, 5 + len(seq), len(raw)]) == (None, False)
        assert _check_utf8(ctx, ms, raw, [0, 3, 5, len(raw)]) == (None, False)
    # a non-ASCII byte just outside a shard that is itself ASCII
    raw = b"abc" + "é".encode() + b"def"
    assert _check_utf8(ctx, ms, raw, [0, 3, len(raw)]) == (None, False)
    assert _check_utf8(ctx, ms, raw, [0, 5, len(raw)]) == (None, False)
    assert _check_utf8(ctx, ms, b"plain,ascii\n" * 100, [0, 7, 7, 600, 1200]) == (None, True)


def _run_utf8_fuzz(ctx, ms):
    rng = np.random.default_rng(5)
    alphabet = np.array([0x41, 0x2C, 0x0A, 0x80, 0xBF, 0xC2, 0xC1, 0xE0, 0xA0, 0x9F, 0xED, 0xEF, 0xF0, 0x90, 0x8F, 0xF4,
                         0xF5, 0xE2, 0x82, 0xAC], dtype=np.uint8)
    for seed in range(60):
        n = int(rng.integers(1, 3000))
        data = np.full(n, 0x61, dtype=np.uint8)
        for p_ in rng.integers(0, n, size=int(rng.integers(0, 12))):
            seg = alphabet[rng.integers(0, alphabet.size, size=int(rng.integers(1, 6)))]
            data[p_:p_ + seg.size] = seg[:max(0, min(seg.size, n - p_))]
        raw = data.tobytes()
        g = int(rng.integers(1, 13))
        # cuts mostly packed around the non-ASCII bytes, so that shards of 0-3 bytes sit next to multi-byte sequences
        hot = np.flatnonzero(data >= 0x80)
        centre = int(hot[0]) if hot.size else n // 2
        pts = [int(x) for x in np.clip(centre + rng.integers(-4, 5, size=g - 1), 0, n)] if seed % 2 else \
              [int(x) for x in rng.integers(0, n + 1, size=g - 1)]
        _check_utf8(ctx, ms, raw, [0] + sorted(pts) + [n])
    # valid multi-byte text stays valid wherever the cuts fall
    txt = ("αβγ,δεζ\nκόσμε,\U0001F642\n".encode()) * 5000
    for _ in range(4):
        assert _check_utf8(ctx, ms, txt, [0] + sorted(int(x) for x in rng.integers(0, len(txt), 7)) + [len(txt)])[0] is None


def test_utf8_seams_on_one_gpu(ctx, one_gpu):
    _run_utf8_seams(ctx, one_gpu)


def test_utf8_seams_across_gpus(ctx, across_gpus):
    _run_utf8_seams(ctx, across_gpus)


def test_utf8_fuzz_on_one_gpu(ctx, one_gpu):
    _run_utf8_fuzz(ctx, one_gpu)


def test_utf8_fuzz_across_gpus(ctx, across_gpus):
    _run_utf8_fuzz(ctx, across_gpus)


# ---- chunks -----------------------------------------------------------------------------------------------------------
def _run_chunks(ctx, ms):
    for name, fc, crlf in (("sample.csv", 3, False), ("sample_rx.csv", 8, True)):
        raw = golden_bytes(name)
        n = len(raw)
        idx = ctx.index_build(raw)
        rc, jump = idx.tape_init(fc, crlf)
        host = idx.to_host()
        want = {num: idx.tape_chunks(num) for num in (1, 2, 3, 5, 12, 200)}
        idx.free()
        # cuts on the bytes of chunk edges (their slots then open a segment), one byte after them, and empty shards
        edges = sorted({int(host[c["start"]]) for c in want[5]} | {int(host[c["end"]]) for c in want[3]})
        cut_sets = [None, [0] + edges + [n], [0] + [e + 1 for e in edges] + [n],
                    [0] + sorted(edges[:3] * 3) + [n], [0, 1, 1, n // 2, n // 2, n]]
        for cuts in cut_sets:
            mi = ms.index(raw, cuts)
            assert mi.tape_init(fc, crlf) == (rc, jump)
            for num, w in want.items():
                got = mi.tape_chunks(num)
                assert got == w, (name, cuts, num)
                o = O.chunks(rc, jump, num)
                assert [(c["id"], c["start"], c["end"], c["record_cnt"]) for c in got] == \
                       [(c["id"], c["start"], c["end"], c["record_cnt"]) for c in o]
            mi.free()


def test_chunks_on_one_gpu(ctx, one_gpu):
    _run_chunks(ctx, one_gpu)


def test_chunks_across_gpus(ctx, across_gpus):
    _run_chunks(ctx, across_gpus)


def test_chunks_status_codes(ctx, one_gpu):
    raw = golden_bytes("sample.csv")
    mi = one_gpu.index(raw, [0, len(raw) // 3, len(raw) // 3, len(raw)])
    with pytest.raises(InvalidState):
        mi.tape_chunks(3)                                   # before tape_init
    rc, _ = mi.tape_init(3, False)
    with pytest.raises(InvalidState):
        mi.tape_chunks(0)
    arr = (_lib.Chunk * 2)()
    n = C.c_size_t()
    code = mi._lib.csvb200_multi_tape_chunks(mi._h, 5, arr, 2, C.byref(n))
    assert code == 9 and n.value == (1 if rc < 5 else 5)   # CSVB200_ERR_CAPACITY with the count set
    assert b"too small" in mi._lib.csvb200_multi_last_error(mi.multi._h)
    mi.free()
