"""csvb200_multi_materialize_columns: columns materialised straight from a distributed index.  Every result must equal,
byte for byte, what csvb200_materialize_columns gives on a one-GPU index of the same bytes, and what the oracle's scalar
definition gives.  Device 0 listed several times runs the whole path on one GPU; the multi-GPU test runs it across real
devices.  The cuts are placed where the interior / boundary split has to get things right: inside a quoted value holding
"" and separators, on a separator and one byte either side of it, inside the header row, around a shard shorter than a
row (a record spanning three segments), and on an empty shard."""
import ctypes as C

import numpy as np
import pytest

import csv_simd_b200 as cs
from csv_simd_b200.errors import InvalidState
from oracle import oracle as O
from tools import gen

pytestmark = pytest.mark.gpu

FLAGS = [0, 1, 2, 3]
TRICKY = b'"x "", y\n z ""q"""'   # a quoted value holding "", a comma and a newline


def _text():
    vals = [b'plain', b'"quoted"', b'  padded\t', b'"with ""escapes"" inside"', b'""', b'', b' "q, and\nnewline" ',
            b'""""', b'\t\t', b'" "', b' "pad" ', b'"a,b"', TRICKY]
    rows = [b'identifier,name,note']
    for i in range(600):
        rows.append(b"%d,%s,%s" % (i, vals[i % len(vals)], vals[(i * 5 + 3) % len(vals)]))
    return b"\n".join(rows) + b"\n"


def _cut_sets(raw, index):
    """{name: cuts} over the text of _text(), 3 fields per row."""
    n = len(raw)
    q = raw.index(TRICKY, n // 3) + 4                 # inside the quoted value, between the quotes of its first ""
    row_ends = index[3::3]                            # slots 3, 6, ...: the line ends
    mid = [int(index[s]) for s in range(3 * 200 + 1, 3 * 200 + 3)]   # the two field separators of a row
    sep = int(row_ends[300])
    s1 = int(index[3 * 400 + 1])                      # the first comma of a row: a shard [s1 - 1, s1 + 1) holds only it
    return {
        "header_and_quote": [0, 5, q, n],
        "on_separator": [0, mid[0], sep - 1, sep, sep + 1, n],
        "three_segments": [0, s1 - 1, s1 + 1, n],
        "empty_shard": [0, q, q, sep, n],
        "all": sorted([0, 5, q, mid[1], sep - 1, sep + 1, s1 - 1, s1 + 1, s1 + 1, n]),
    }


def _boundary_records(mi, jump, record_cnt):
    """records whose slots run over more than one segment (what the split stages on one device)"""
    base = np.array([s["base"] for s in mi.segments()] + [len(mi)], dtype=np.int64)
    out = []
    for r in range(record_cnt - 1):
        lo, hi = (r + 1) * jump, (r + 2) * jump
        if np.searchsorted(base, lo, side="right") != np.searchsorted(base, hi, side="right"):
            out.append(r)
    return out


def _check(mi, idx, raw, host, rc, field_cnt, crlf, fields, first, nrec, flags, oracle=True):
    got = mi.materialize_columns(fields, first, nrec, flags)
    want = idx.materialize_columns(fields, first, nrec, flags)
    assert len(got) == len(fields)
    for f, (g_off, g_val), (w_off, w_val) in zip(fields, got, want):
        assert (g_off == w_off).all(), (fields, f, first, nrec, flags)
        assert g_val.tobytes() == w_val.tobytes(), (fields, f, first, nrec, flags)
        if oracle:
            o_off, o_val = O.materialize_column(raw, host, rc, field_cnt, crlf, f, first, nrec, flags)
            assert (g_off == o_off).all() and g_val.tobytes() == o_val, (fields, f, first, nrec, flags)


def _run_cut_sets(ctx, devices_for):
    raw = _text()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, jump = idx.tape_init(3, False)
    host = idx.to_host()
    column_sets = ([1], [2, 0, 1, 1], [(i * 7) % 4 for i in range(32)])   # field 3 does not exist: empty values
    for name, cuts in _cut_sets(raw, host).items():
        m = cs.Multi(devices_for(len(cuts) - 1))
        mi = m.index_build_distributed(raw, cuts)
        assert (mi.to_host() == host).all(), name
        assert mi.tape_init(3, False) == (rc, jump)
        segs = mi.segments()
        bnd = _boundary_records(mi, jump, rc)
        assert bnd, name
        if name == "three_segments":
            assert any(s["entries"] == 1 for s in segs)
        if name == "empty_shard":
            assert any(s["entries"] == 0 for s in segs)
        windows = [(0, rc - 1), (0, 0), (rc - 6, 20), (rc + 3, 4)]
        for b in bnd:
            windows += [(b, 1), (b, 7), (max(0, b - 9), 10), (b - 1, 2)]
        for flags in FLAGS:
            for fields in column_sets:
                for first, nrec in windows:
                    if first < 0:
                        continue
                    _check(mi, idx, raw, host, rc, 3, False, fields, first, nrec, flags, oracle=len(fields) < 32)
        mi.free()
        m.close()
    idx.free()


def test_cut_placements_on_one_gpu(ctx):
    _run_cut_sets(ctx, lambda g: [ctx.device] * g)


def test_cut_placements_across_gpus(ctx):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs at least 2 GPUs")
    _run_cut_sets(ctx, lambda g: [k % ndev for k in range(g)])


@pytest.mark.parametrize("kind", ["unquoted", "quoted"])
def test_generated_inputs(ctx, kind):
    """The synthetic generators at a few MiB: default cuts and cuts at random (mostly unaligned) offsets, all 16 columns
    and a few subsets, against the one-GPU call and the oracle."""
    import torch
    data, _ = gen.unquoted(3 << 20, seed=5) if kind == "unquoted" else gen.quoted(3 << 20, seed=6)
    raw = data.tobytes()
    hdr = O.header_new(raw)
    field_cnt, crlf = hdr.field_cnt, hdr.crlf
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, jump = idx.tape_init(field_cnt, crlf)
    host = idx.to_host()
    rng = np.random.default_rng(11)
    ndev = torch.cuda.device_count()
    for cuts in (None, [0] + sorted(int(x) for x in rng.integers(0, len(raw), 6)) + [len(raw)]):
        g = 4 if cuts is None else len(cuts) - 1
        m = cs.Multi([k % ndev for k in range(g)])
        mi = m.index_build_distributed(raw, cuts)
        mi.tape_init(field_cnt, crlf)
        for flags in FLAGS:
            _check(mi, idx, raw, host, rc, field_cnt, crlf, list(range(field_cnt)), 0, rc - 1, flags, oracle=False)
            _check(mi, idx, raw, host, rc, field_cnt, crlf, [field_cnt - 1], 0, rc - 1, flags)
            _check(mi, idx, raw, host, rc, field_cnt, crlf, [3, 0, 3, 9], rc // 3, rc // 2, flags)
        mi.free()
        m.close()
    idx.free()


def test_window_wrapping_past_record_0xffffffff(ctx):
    """Record numbers are u32 and wrap as in the one-GPU call: record 0xFFFFFFFF reads the header row's slots."""
    raw = _text()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, _ = idx.tape_init(3, False)
    m = cs.Multi([ctx.device] * 3)
    mi = m.index_build_distributed(raw, _cut_sets(raw, idx.to_host())["header_and_quote"])
    mi.tape_init(3, False)
    for flags in FLAGS:
        got = mi.materialize_columns([0, 1, 2], 0xFFFFFFFF - 3, 12, flags)
        want = idx.materialize_columns([0, 1, 2], 0xFFFFFFFF - 3, 12, flags)
        for (g_off, g_val), (w_off, w_val) in zip(got, want):
            assert (g_off == w_off).all() and g_val.tobytes() == w_val.tobytes()
    mi.free()
    m.close()
    idx.free()


def _raw_call(mi, fields, first, nrec, flags, offs, outs, caps):
    k = len(fields)
    f = np.ascontiguousarray(fields, dtype=np.uint32)
    p_off = (C.c_void_p * k)(*[o.ctypes.data if o is not None else None for o in offs]) if offs is not None else None
    p_out = (C.c_void_p * k)(*[v.ctypes.data if v is not None and v.size else None for v in outs]) if outs is not None else None
    c_caps = (C.c_size_t * k)(*caps) if caps is not None else None
    lens = (C.c_size_t * max(k, 1))()
    rc = mi._lib.csvb200_multi_materialize_columns(mi._h, f.ctypes.data, k, first, nrec, flags, p_off, p_out, c_caps, lens)
    return rc, [int(lens[c]) for c in range(k)]


def test_status_codes(ctx):
    """INVALID_STATE before tape_init; INVALID_ARG for 0 or 33 columns, unknown flags and null arrays; CAPACITY when one
    column does not fit, with every column's offsets and length still correct."""
    raw = _text()
    idx = ctx.index_build(raw, cs.BUILD_KEEP_BYTES)
    rc, _ = idx.tape_init(3, False)
    host = idx.to_host()
    m = cs.Multi([ctx.device] * 4)
    mi = m.index_build_distributed(raw, _cut_sets(raw, host)["on_separator"][:4] + [len(raw)])
    with pytest.raises(InvalidState):
        mi.materialize_columns([0], 0, 5)
    mi.tape_init(3, False)
    nrec, flags = rc - 1, cs.FIELD_UNQUOTE | cs.FIELD_TRIM
    with pytest.raises(ValueError):
        mi.materialize_columns([], 0, nrec, flags)
    with pytest.raises(ValueError):
        mi.materialize_columns([0] * 33, 0, nrec, flags)
    with pytest.raises(ValueError):
        mi.materialize_columns([0], 0, nrec, 4)
    offs = [np.zeros(nrec + 1, dtype=np.uint64) for _ in range(2)]
    assert _raw_call(mi, [1, 2], 0, nrec, flags, None, None, None)[0] == 1
    assert _raw_call(mi, [1, 2], 0, nrec, flags, [offs[0], None], None, None)[0] == 1
    want = [O.materialize_column(raw, host, rc, 3, False, f, 0, nrec, flags) for f in (1, 2)]
    # the sizing call, then values present for one column only
    code, lens = _raw_call(mi, [1, 2], 0, nrec, flags, offs, None, None)
    assert code == 9 and lens == [len(w[1]) for w in want]
    outs = [np.zeros(len(w[1]), dtype=np.uint8) for w in want]
    assert _raw_call(mi, [1, 2], 0, nrec, flags, offs, [outs[0], None], lens)[0] == 1
    # CAPACITY on the second column only: lengths and all offsets are still right, the values are not written
    offs = [np.zeros(nrec + 1, dtype=np.uint64) for _ in range(2)]
    outs = [np.full(len(w[1]), 0xEE, dtype=np.uint8) for w in want]
    code, lens = _raw_call(mi, [1, 2], 0, nrec, flags, offs, outs, [len(want[0][1]), len(want[1][1]) - 1])
    assert code == 9 and lens == [len(w[1]) for w in want]
    for o, (w_off, _) in zip(offs, want):
        assert (o == w_off).all()
    assert (outs[0] == 0xEE).all()
    # and the exact capacities fill both
    code, lens = _raw_call(mi, [1, 2], 0, nrec, flags, offs, outs, [len(w[1]) for w in want])
    assert code == 0
    for o, v, (w_off, w_val) in zip(offs, outs, want):
        assert (o == w_off).all() and v.tobytes() == w_val
    mi.free()
    m.close()
    idx.free()
