"""Values past 4 GiB: column materialisation, the values behind lookups and the distributed index on inputs whose values,
or whose 256-record tiles, add up to 2^32 bytes or more.  Every input is built with numpy from a fixed seed, and the
builder knows every blob's length under every flag; the oracle (read_sse for the index, materialize_column and the
C field_value for the values, u64 throughout) is checked against those lengths and then against the library.

- A: about 6 GiB, 300 rows of ~20 MiB blobs in four shapes (plain, padded, quoted with escapes, padded and quoted):
  under every flag a 256-record tile holds more than 2^32 bytes of blob values.
- B: one padded, quoted value of 2^32 + 4099 bytes with a "" pair across its own byte 2^32.  One thread walks it
  whenever it is unquoted or written as a column, which takes minutes: one test makes the few calls that do.
- C: n = 2^32 exactly (a default context keeps 4-byte entries, the last is 0xFFFFFFFF), and 256 blobs that add up to
  just under 2^32: the top of the compact range and of the multi-column kernels' exact range.

Every test starts with an offsets-only comparison of the device form, which launches no write pass."""
import gc

import numpy as np
import pytest

import csv_simd_b200 as cs
from oracle import oracle as O

pytestmark = pytest.mark.gpu

B32 = 1 << 32
MIB = 1 << 20
FLAGS = [0, 1, 2, 3]
FIELD_SETS = ([1], [1, 0], [1, 0, 2, 0, 2, 0, 2, 1])   # the single-column kernels, the plain and the batched multi-column
ALPHA = np.frombuffer(b"ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/", dtype=np.uint8)
# peaks measured on one B200 (input A is the largest): 45 GB of device memory and 39 GB of host memory (input, oracle
# column, the host columns of the 8-column call and the copies of device buffers)
DEVICE_NEED = 56 << 30
HOST_NEED = 64 << 30


# ---- inputs ------------------------------------------------------------------------------------------------------
class Blob:
    """pl / pr: padding bytes (space, tab) on each side; body: the L bytes between the quotes (or the whole value
    when unquoted), made of base64 characters; pairs: body positions of "" escapes; comma / lf: body positions of
    a ',' and an LF inside a quoted body."""

    def __init__(self, shape, L, pl=0, pr=0, pairs=(), comma=None, lf=None, pool_off=0):
        self.shape, self.L, self.pl, self.pr = shape, L, pl, pr
        self.pairs, self.comma, self.lf, self.pool_off = list(pairs), comma, lf, pool_off

    @property
    def quoted(self):
        return self.shape in (2, 3)

    @property
    def raw(self):
        return self.pl + self.pr + self.L + (2 if self.quoted else 0)

    def length(self, flags):
        """the value's length under flags, from the shape alone"""
        trimmed = self.raw - self.pl - self.pr
        unquoted = self.L - len(self.pairs)
        if flags & 1 and self.quoted and (flags & 2 or self.pl + self.pr == 0):
            return unquoted
        return trimmed if flags & 2 else self.raw


def _blob(rng, shape, L):
    padded = shape in (1, 3)
    pl, pr = (int(rng.integers(1, 5)), int(rng.integers(1, 5))) if padded else (0, 0)
    pairs, comma, lf = (), None, None
    if shape in (2, 3):
        slots = np.sort(rng.choice(np.arange(2, L // 64 - 2), 8, replace=False)) * 64 + 8
        pairs, comma, lf = [int(s) for s in slots[:6]], int(slots[6]), int(slots[7])
    return Blob(shape, L, pl, pr, pairs, comma, lf, int(rng.integers(0, 1 << 20)))


def _copy_cyclic(dst, pool, off):
    i = min(dst.size, pool.size - off)
    dst[:i] = pool[off:off + i]
    while i < dst.size:
        k = min(dst.size - i, pool.size)
        dst[i:i + k] = pool[:k]
        i += k


class Input:
    def __init__(self, name, rows, pool, fill_to=None):
        """rows: (id bytes, Blob, tag bytes); fill_to: pad the last row's tag with 'z' to make the input that long"""
        self.name = name
        head = b"id,blob,tag\n"
        sizes = [len(i) + 1 + b.raw + 1 + len(t) + 1 for i, b, t in rows]
        n = len(head) + sum(sizes)
        if fill_to is not None:
            i, b, t = rows[-1]
            rows[-1] = (i, b, t + b"z" * (fill_to - n))
            n = fill_to
        data = np.empty(n, dtype=np.uint8)
        data[:len(head)] = np.frombuffer(head, dtype=np.uint8)
        at = len(head)
        self.bodies = []       # [start, end) of every blob body
        for i, b, t in rows:
            for piece in (i, b","):
                data[at:at + len(piece)] = np.frombuffer(piece, dtype=np.uint8)
                at += len(piece)
            data[at:at + b.pl] = np.frombuffer(b" \t", dtype=np.uint8)[np.arange(b.pl) % 2]
            at += b.pl
            if b.quoted:
                data[at] = 0x22
                at += 1
            body = data[at:at + b.L]
            _copy_cyclic(body, pool, b.pool_off)
            for p in b.pairs:
                body[p:p + 2] = 0x22
            if b.comma is not None:
                body[b.comma] = 0x2C
                body[b.lf] = 0x0A
            self.bodies.append((at, at + b.L))
            at += b.L
            if b.quoted:
                data[at] = 0x22
                at += 1
            data[at:at + b.pr] = np.frombuffer(b"\t ", dtype=np.uint8)[np.arange(b.pr) % 2]
            at += b.pr
            for piece in (b",", t, b"\n"):
                data[at:at + len(piece)] = np.frombuffer(piece, dtype=np.uint8)
                at += len(piece)
        assert at == n
        self.data, self.n, self.blobs = data, n, [b for _, b, _ in rows]
        self.rows = len(rows)
        self.offs = {}         # (field, flags) -> oracle offsets over every data row

    def blob_lens(self, flags):
        return np.array([b.length(flags) for b in self.blobs], dtype=np.uint64)

    def in_body(self, a, b):
        return any(s <= a and b <= e for s, e in self.bodies)


def _tag(i):
    return (b"t%d" % i, b" t%d\t" % i, b'"q""%d"' % i, b'" s,%d "' % i)[i % 4]


def input_a():
    rng = np.random.default_rng(20261022)
    pool = ALPHA[rng.integers(0, 64, 2 * MIB, dtype=np.uint8)]
    rows = [(b"%d" % i, _blob(rng, i % 4, 20 * MIB + int(rng.integers(-65536, 65536))), _tag(i)) for i in range(300)]
    inp = Input("A", rows, pool)
    # a 2-byte UTF-8 character across byte 2^32, and one invalid byte after it, inside a blob body
    inp.bad = B32 + 777
    assert inp.in_body(B32 - 9, inp.bad + 9) and np.isin(inp.data[B32 - 9:inp.bad + 9], ALPHA).all()
    inp.data[B32 - 1:B32 + 1] = (0xC3, 0xA9)
    inp.data[inp.bad] = 0xFF
    for flags in FLAGS:
        lens = inp.blob_lens(flags)
        assert lens[:256].sum() > B32 and lens[7:263].sum() > B32, flags
    return inp


def input_b():
    rng = np.random.default_rng(4099)
    pool = ALPHA[rng.integers(0, 64, 2 * MIB, dtype=np.uint8)]
    pl, pr = 2, 3
    L = B32 + 4099 - pl - pr - 2
    mid = B32 - 1 - (pl + 1)       # the pair sits on the value's own bytes 2^32 - 1 and 2^32
    big = Blob(3, L, pl, pr, pairs=[5000, mid, L - 5000], comma=70000, lf=140000)
    small = [_blob(rng, s, 4096 + 64 * s) for s in (0, 1, 2, 3, 2, 1)]
    rows = [(b"%d" % i, small[i], _tag(i)) for i in range(3)] + [(b"3", big, _tag(3))]
    rows += [(b"%d" % (i + 4), small[3 + i], _tag(i + 4)) for i in range(3)]
    inp = Input("B", rows, pool)
    assert big.raw == B32 + 4099 and inp.n > B32
    return inp


def input_c():
    rng = np.random.default_rng(1 << 32)
    pool = ALPHA[rng.integers(0, 64, 2 * MIB, dtype=np.uint8)]
    total = B32 - 32768
    raw = (total // 256) + rng.integers(-4096, 4096, 256)
    raw[-1] += total - raw.sum()
    rows = []
    for i in range(256):
        b = _blob(rng, i % 4, 1 << 20)
        b.L = int(raw[i]) - (b.raw - b.L)          # the same shape, stretched to the raw length drawn above
        rows.append((b"%d" % i, b, _tag(i)))
    rows += [(b"%d" % i, _blob(rng, i % 4, 1024), _tag(i)) for i in range(256, 272)]
    inp = Input("C", rows, pool, fill_to=B32)
    assert inp.data[-1] == 0x0A
    for flags in FLAGS:
        s = int(inp.blob_lens(flags)[:256].sum())
        assert B32 - (64 << 10) <= s < B32, flags
    return inp


BUILDERS = {"A": input_a, "B": input_b, "C": input_c}


def _host_available():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) << 10
    return 0


@pytest.fixture(scope="module")
def inp(request, ctx):
    """one input at a time: pytest groups the tests by this module-scoped parameter and tears the last one down first"""
    import torch
    free, _ = torch.cuda.mem_get_info(torch.device("cuda", ctx.device))
    if free < DEVICE_NEED:
        pytest.skip(f"needs ~{DEVICE_NEED >> 30} GB of free device memory")
    if _host_available() < HOST_NEED:
        pytest.skip(f"needs ~{HOST_NEED >> 30} GB of free host memory")
    x = BUILDERS[request.param]()
    x.idx = ctx.index_build(x.data, cs.BUILD_KEEP_BYTES | cs.BUILD_VALIDATE)
    x.host = O.read_sse(x.data)
    assert (x.idx.to_host() == x.host).all()
    x.rc, x.jump = x.idx.tape_init(3, False)
    assert x.rc - 1 == x.rows and x.jump == 3
    x.windows = [(0, x.rc - 1)] + ([(7, 260), (250, 10)] if x.rows >= 260 else [(3, 1), (4, 3)])
    yield x
    x.idx.free()
    del x.idx, x.data, x
    gc.collect()
    torch.cuda.empty_cache()


ON_A = pytest.mark.parametrize("inp", ["A"], indirect=True)
ON_ALL = pytest.mark.parametrize("inp", ["A", "B", "C"], indirect=True)


# ---- oracle ------------------------------------------------------------------------------------------------------
def _oracle_offsets(x, field, flags):
    """offsets of every data row from the oracle's sizing pass (O.materialize_column without the output)"""
    key = (field, flags)
    if key not in x.offs:
        offs = np.zeros(x.rows + 1, dtype=np.uint64)
        O.lib().oracle_materialize_column(x.data.ctypes.data, x.n, x.host.ctypes.data, x.host.size, x.rc, 3, 0, field,
                                          0, x.rows, flags, offs.ctypes.data, None)
        if field == 1:      # the lengths the builder knows
            assert (np.diff(offs) == x.blob_lens(flags)).all(), flags
        x.offs[key] = offs
    return x.offs[key]


def _oracle_values(x, field, flags):
    offs, vals = O.materialize_column(x.data, x.host, x.rc, 3, False, field, 0, x.rows, flags)
    assert (offs == _oracle_offsets(x, field, flags)).all()
    return offs, np.frombuffer(vals, dtype=np.uint8)


def _win(offs, first, nrec):
    return offs[first:first + nrec + 1] - offs[first]


def _same_bytes(got, want, what):
    """byte equality of two large arrays, 256 MiB at a time (no full-size temporaries)"""
    assert got.size == want.size, what
    step = 256 * MIB
    for i in range(0, got.size, step):
        assert np.array_equal(got[i:i + step], want[i:i + step]), (what, i)


# ---- device form, offsets only -----------------------------------------------------------------------------------
def _offsets_device(x, fields, first, nrec, flags):
    import torch
    dev = torch.device("cuda", x.idx.ctx.device)
    d_off = [torch.full((nrec + 1,), -1, dtype=torch.int64, device=dev) for _ in fields]
    torch.cuda.synchronize(dev)     # the library works on its own stream: the fills must land first
    x.idx.materialize_columns_device(fields, first, nrec, flags, [t.data_ptr() for t in d_off])
    torch.cuda.synchronize(dev)
    return [t.cpu().numpy().view(np.uint64) for t in d_off]


def _check_offsets(x, fields, first, nrec, flags):
    got = _offsets_device(x, fields, first, nrec, flags)
    for f, g in zip(fields, got):
        w = _win(_oracle_offsets(x, f, flags), first, nrec)
        bad = np.flatnonzero(g != w)
        assert bad.size == 0, (x.name, fields, first, nrec, flags, f, int(bad[0]) if bad.size else None)


def _gate(x):
    """the first assertion of every test: the offsets of the blob and id columns without a write pass"""
    _check_offsets(x, [1, 0], 0, x.rows, 0)


@ON_ALL
def test_offsets_device_form(inp):
    x = inp
    _gate(x)
    # the length pass walks B's 4 GiB value with one thread when it unquotes it (flags 3), which takes minutes
    for flags in (FLAGS if x.name != "B" else [0, 1, 2]):
        for fields in FIELD_SETS:
            for first, nrec in x.windows:
                _check_offsets(x, fields, first, nrec, flags)
    # the tile sums that make these inputs what they are
    o = _oracle_offsets(x, 1, 3)
    if x.name == "A":
        assert o[256] - o[0] > B32 and o[263] - o[7] > B32
    if x.name == "B":
        assert o[4] - o[3] > B32
    if x.name == "C":
        assert B32 - (64 << 10) <= o[256] - o[0] < B32
        # the last entry, the final LF, is 0xFFFFFFFF: the largest a 4-byte entry holds.  The binding does not expose
        # the entry width, so that a default context stores n = 2^32 in 4-byte entries rests on
        # test_compact_index.py::test_4gib_edge; here the entries and the lookups are checked against the oracle
        assert x.n == B32 and int(x.host[-1]) == 0xFFFFFFFF
        rec, fld = np.array([x.rows - 1, x.rows - 1, 255, 256], dtype=np.uint32), np.array([2, 1, 1, 1], dtype=np.uint32)
        rg = x.idx.seek_fields(rec, fld)
        assert int(rg[0, 1]) == 0xFFFFFFFF
        for q in range(rec.size):
            assert (int(rg[q, 0]), int(rg[q, 1])) == O.seek_field(x.host, x.n, x.rc, 3, False, int(rec[q]), int(fld[q]))


# ---- host forms, the device form with values, lookups ------------------------------------------------------------
def _check_host_columns(x, fields, first, nrec, flags, want):
    got = x.idx.materialize_columns(fields, first, nrec, flags) if len(fields) > 1 else \
        [x.idx.materialize_column(fields[0], first, nrec, flags)]
    for f, (g_off, g_val) in zip(fields, got):
        w_off, w_val = want[f]
        assert (g_off == _win(w_off, first, nrec)).all(), (x.name, fields, first, nrec, flags, f)
        _same_bytes(g_val, w_val[int(w_off[first]):int(w_off[first + nrec])], (x.name, fields, first, nrec, flags, f))


def _check_device_cap(x, flags, want, k):
    """fields [1, 0] with values; column 1's cap falls inside record k's value: every value before it is written whole,
    record k's and every later one is skipped, and the sentinel bytes from its start on stay untouched"""
    import torch
    dev = torch.device("cuda", x.idx.ctx.device)
    (o1, v1), (o0, v0) = want[1], want[0]
    cap1 = int(o1[k] + o1[k + 1]) // 2
    assert int(o1[k]) < cap1 < int(o1[k + 1])
    caps = [cap1, int(o0[-1])]
    d_off = [torch.full((x.rows + 1,), -1, dtype=torch.int64, device=dev) for _ in range(2)]
    d_out = [torch.full((c + 4096,), 0xEE, dtype=torch.uint8, device=dev) for c in caps]
    torch.cuda.synchronize(dev)
    x.idx.materialize_columns_device([1, 0], 0, x.rows, flags, [t.data_ptr() for t in d_off], [t.data_ptr() for t in d_out],
                                     caps)
    torch.cuda.synchronize(dev)
    assert (d_off[0].cpu().numpy().view(np.uint64) == o1).all() and (d_off[1].cpu().numpy().view(np.uint64) == o0).all()
    out1 = d_out[0].cpu().numpy()
    _same_bytes(out1[:int(o1[k])], v1[:int(o1[k])], (x.name, flags, "cap"))
    assert (out1[int(o1[k]):] == 0xEE).all(), (x.name, flags)
    out0 = d_out[1].cpu().numpy()
    _same_bytes(out0[:caps[1]], v0, (x.name, flags, "ids"))
    assert (out0[caps[1]:] == 0xEE).all()


def _lookups(x):
    """every data row's blob, then probes: past the last record, at r = 0xFFFFFFFF (r + 1 wraps to the header row in
    u32, as in the reference), past the last field"""
    rec = np.concatenate([np.arange(x.rows), [x.rows, x.rows + 5, 0xFFFFFFFF, 0, 2]]).astype(np.uint32)
    fld = np.concatenate([np.ones(x.rows), [1, 1, 1, 3, 0xFFFFFFFF]]).astype(np.uint32)
    return rec, fld


def _check_lookup_values(got, x, rec, fld, flags, w_off, w_val, what):
    """the data rows against the oracle's column, the probes against the oracle's seek_field and field_value"""
    g_off, g_val, g_found = got
    assert (g_off[:x.rows + 1] == w_off).all() and g_found[:x.rows].all(), what
    _same_bytes(g_val[:int(w_off[-1])], w_val, what)
    at = int(w_off[-1])
    for q in range(x.rows, rec.size):
        rg = O.seek_field(x.host, x.n, x.rc, 3, False, int(rec[q]), int(fld[q]))
        v = O.field_value(x.data[rg[0]:rg[1]].tobytes(), flags) if rg else b""
        assert bool(g_found[q]) == (rg is not None) and int(g_off[q + 1]) - int(g_off[q]) == len(v), (what, q)
        assert g_val[at:at + len(v)].tobytes() == v, (what, q)
        at += len(v)
    assert g_found[x.rows + 2] and not g_found[[x.rows, x.rows + 1, x.rows + 3, x.rows + 4]].any(), what
    assert (g_val[at:] == 0xEE).all(), what     # the device form's sentinel bytes past the values


def _seek_values_device(x, rec, fld, flags, cap):
    import torch
    dev = torch.device("cuda", x.idx.ctx.device)
    nq = rec.size
    d_rec = torch.from_numpy(rec.view(np.int32).copy()).to(dev)
    d_fld = torch.from_numpy(fld.view(np.int32).copy()).to(dev)
    d_off = torch.full((nq + 1,), -1, dtype=torch.int64, device=dev)
    d_found = torch.full(((nq + 63) // 64,), -1, dtype=torch.int64, device=dev)
    d_out = torch.full((cap + 4096,), 0xEE, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)     # the library works on its own stream: the fills must land first
    x.idx.seek_values_device(d_rec.data_ptr(), d_fld.data_ptr(), nq, flags, d_off.data_ptr(), d_out.data_ptr(), cap,
                             d_found.data_ptr())
    torch.cuda.synchronize(dev)
    words = d_found.cpu().numpy().view(np.uint64)
    found = np.unpackbits(words.view(np.uint8), bitorder="little")[:nq].astype(bool)
    return d_off.cpu().numpy().view(np.uint64), d_out.cpu().numpy(), found


def _check_records(x, got, rec):
    g_off, g_val, g_found = got
    for q in range(rec.size):
        rg = O.seek_record(x.host, x.n, x.rc, x.jump, 3, int(rec[q]))
        assert bool(g_found[q]) == (rg is not None), (x.name, "record", q)
        want = x.data[rg[0]:rg[1]] if rg else x.data[:0]
        _same_bytes(g_val[int(g_off[q]):int(g_off[q + 1])], want, (x.name, "record", q))


@ON_ALL
def test_values(inp):
    x = inp
    _gate(x)
    k = {"A": 150, "B": 3, "C": 128}[x.name]
    rec, fld = _lookups(x)
    # one thread walks B's 4 GiB value in every column write and in every trimmed or unquoted lookup, which takes
    # minutes: on B the values come from the 32-lane raw copies of the lookups, and the device form with a cap inside
    # that value (skipped whole, so never walked) checks every other value
    subset = {"column": FLAGS, "columns": FLAGS, "batched": (0, 3), "seek": FLAGS}
    if x.name == "B":
        subset = {"column": (), "columns": (), "batched": (), "seek": (0,)}
    for flags in FLAGS:
        want = {f: _oracle_values(x, f, flags) for f in (0, 1, 2)}
        for w, (first, nrec) in enumerate(x.windows if x.name != "B" else x.windows[::2]):
            if flags in subset["column"]:
                _check_host_columns(x, [1], first, nrec, flags, want)
            if flags in subset["columns"] and (w == 0 or flags == 3):
                _check_host_columns(x, [1, 0, 2], first, nrec, flags, want)
        if flags in subset["batched"]:
            _check_host_columns(x, list(FIELD_SETS[2]), 0, x.rows, flags, want)
        if x.name != "B" or flags in (0, 2):
            _check_device_cap(x, flags, want, k)
        if flags in subset["seek"]:
            w_off, w_val = want[1]
            _check_lookup_values(x.idx.seek_values(rec, fld, flags), x, rec, fld, flags, w_off, w_val,
                                 (x.name, flags, "seek"))
            if flags in (0, 3):
                _check_lookup_values(_seek_values_device(x, rec, fld, flags, int(w_off[-1]) + 64), x, rec, fld, flags,
                                     w_off, w_val, (x.name, flags, "seek device"))
        if flags == 0:
            w_off, w_val = want[1]
            g_off, g_val = x.idx.gather_fields(rec[:x.rows], fld[:x.rows])
            assert (g_off == w_off).all()
            _same_bytes(g_val, w_val, (x.name, "gather"))
            _check_records(x, x.idx.seek_values(rec), rec)
        del want


# ---- input A: chunks, UTF-8, the distributed index ---------------------------------------------------------------
@ON_A
def test_chunks_and_utf8(inp, ctx):
    x = inp
    _gate(x)
    got = x.idx.tape_chunks(4)
    want = O.chunks(x.rc, x.jump, 4)
    assert [(c["id"], c["start"], c["end"], c["record_cnt"]) for c in got] == \
           [(c["id"], c["start"], c["end"], c["record_cnt"]) for c in want]
    for c in got:
        assert c["byte_start"] == int(x.host[c["start"]]) + 1 and c["byte_end"] == int(x.host[c["end"]]) + 1
    assert got[-1]["byte_end"] == x.n and any(c["byte_start"] > B32 for c in got)
    # the oracle decodes the blob that holds byte 2^32, from its body's first byte (ASCII, so a character boundary)
    s, e = next((s, e) for s, e in x.bodies if s < B32 < e)
    assert s + O.utf8_valid_up_to(x.data[s:e]) == x.bad
    assert ctx.validate_utf8(x.data) == (x.bad, False)
    assert x.idx.validate_utf8() == x.bad
    assert x.idx.validation()[0] is False


def _cut_sets(x):
    """two shards cut inside the first blob that starts past 4.3 GiB (shard 0 holds more than 2^32 bytes), and three
    with a second cut inside record 2's blob"""
    j = next(i for i, (s, _) in enumerate(x.bodies) if s > int(4.3 * (1 << 30)))
    s, e = x.bodies[j]
    c = (s + e) // 2 + 3
    s2, e2 = x.bodies[2]
    c2 = (s2 + e2) // 2 + 1
    assert c > B32
    return {"two": ([0, c, x.n], [j]), "three": ([0, c2, c, x.n], [2, j])}


@ON_A
@pytest.mark.parametrize("placement", ["one_gpu", "across_gpus"])
def test_distributed(inp, ctx, placement):
    import torch
    x = inp
    _gate(x)
    ndev = torch.cuda.device_count()
    if placement == "across_gpus" and ndev < 2:
        pytest.skip("needs at least 2 GPUs")
    for name, (cuts, crossing) in _cut_sets(x).items():
        g = len(cuts) - 1
        devices = [ctx.device] * g if placement == "one_gpu" else [k % ndev for k in range(g)]
        for d in set(devices) - {ctx.device}:     # the fixture checked ctx.device; a shard may land on another GPU
            if torch.cuda.mem_get_info(torch.device("cuda", d))[0] < DEVICE_NEED:
                pytest.skip(f"needs ~{DEVICE_NEED >> 30} GB of free device memory on device {d}")
        m = cs.Multi(devices)
        mi = m.index_build_distributed(x.data, cuts)
        assert (mi.to_host() == x.host).all()
        assert mi.tape_init(3, False) == (x.rc, x.jump)
        # two shards: 1 and 2 columns under every flag, 8 under one; three shards: 2 columns under two flags
        runs = {"two": [(f, cols) for f in FLAGS for cols in FIELD_SETS if len(cols) < 8 or f == 3],
                "three": [(f, [1, 0]) for f in (0, 3)]}[name]
        for flags in sorted({f for f, _ in runs}):
            want = {f: _oracle_values(x, f, flags) for f in (0, 1, 2)}
            for fields in [cols for f, cols in runs if f == flags]:
                for f, (g_off, g_val) in zip(fields, mi.materialize_columns(fields, 0, x.rows, flags)):
                    assert (g_off == want[f][0]).all(), (name, fields, flags, f)
                    _same_bytes(g_val, want[f][1], (name, fields, flags, f))
            # the values that contain a cut, and the records that do
            rec = np.array(crossing, dtype=np.uint32)
            offs, vals, found = mi.seek_values(rec, np.ones_like(rec), flags)
            w_off, w_val = want[1]
            assert found.all()
            for q, r in enumerate(crossing):
                _same_bytes(vals[int(offs[q]):int(offs[q + 1])], w_val[int(w_off[r]):int(w_off[r + 1])], (name, flags, r))
            del want
        rec = np.array(crossing, dtype=np.uint32)
        offs, vals, found = mi.seek_values(rec)
        assert found.all()
        for q, r in enumerate(crossing):
            a, b = O.seek_record(x.host, x.n, x.rc, x.jump, 3, r)
            _same_bytes(vals[int(offs[q]):int(offs[q + 1])], x.data[a:b], (name, "record", r))
        mi.free()
        m.close()


# ---- input B: its value past 2^32 walked by one thread ---------------------------------------------------------
@pytest.mark.parametrize("inp", ["B"], indirect=True)
def test_one_value_past_2_pow_32(inp):
    """B's value unquoted and written by the kernels that walk it with one thread: the single-column length pass
    (value_len_range's u64 counter), the lookup values' length and write passes, and the column write kernel.  Each
    walk of its 2^32 + 4099 bytes is slow, so these are the only calls that make one."""
    import time
    x = inp
    _gate(x)
    b = x.blobs[3]
    w = _oracle_offsets(x, 1, 3)
    assert int(w[4] - w[3]) == b.length(3) == b.L - len(b.pairs) > B32
    t0 = time.time()
    _check_offsets(x, [1], 3, 1, 3)
    t1 = time.time()
    print(f"\nB, one-thread walk in the column length pass (flags 3): {t1 - t0:.1f} s", flush=True)
    a, e = O.seek_field(x.host, x.n, x.rc, 3, False, 3, 1)
    want = np.frombuffer(O.field_value(x.data[a:e].tobytes(), 3), dtype=np.uint8)
    mid = B32 - 1 - (b.pl + 1)      # the body position of the "" pair on the value's own bytes 2^32 - 1 and 2^32
    assert mid in b.pairs and bytes(x.data[a + B32 - 1:a + B32 + 1]) == b'""'
    q = mid - sum(p < mid for p in b.pairs)      # where it lands once unquoted: one '"', then the next body byte
    assert want.size == b.length(3) and want[q] == 0x22 and want[q + 1] == x.data[a + B32 + 1]
    t2 = time.time()
    offs, out, found = _seek_values_device(x, np.array([3], dtype=np.uint32), np.array([1], dtype=np.uint32), 3, want.size)
    t3 = time.time()
    print(f"B, one-thread walks in the lookup length and write passes (flags 3): {t3 - t2:.1f} s", flush=True)
    assert found[0] and int(offs[0]) == 0 and int(offs[1]) == want.size
    _same_bytes(out[:want.size], want, ("B", "seek device", 3))
    assert (out[want.size:] == 0xEE).all()
    del out, want
    t4 = time.time()
    g_off, g_val = x.idx.materialize_column(1, 3, 1, 0)
    t5 = time.time()
    assert g_off.tolist() == [0, e - a] and e - a == b.raw
    _same_bytes(g_val, x.data[a:e], ("B", "column", 3))
    print(f"B, one-thread walk in the column write pass (flags 0): {t5 - t4:.1f} s", flush=True)
