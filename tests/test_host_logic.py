"""CPU: host-side mirror of the reference API (Header, boundaries, chunks, error mapping) and the
multi-rank exchange logic (gloo, world_size 2) checked against the oracle."""
import os
import socket
import sys

import numpy as np
import pytest

import csv_simd_b200 as cs
from csv_simd_b200 import dist as csd
from oracle import oracle as O
from tests import cases
from tests.conftest import ROOT, golden_bytes


@pytest.mark.parametrize("name", ["reader_test01.csv", "sample.csv", "sample_rx.csv"])
def test_header_new_matches_oracle(golden, name):
    data = golden_bytes(name)
    h = cs.Header.new(cs.Mmap(data=data))
    g = golden[name]
    assert h.header == g["header"] and h.field_cnt == g["field_cnt"] and h.record_offset == g["record_offset"]
    assert (h.new_line is cs.NewLine.CRLF) == g["crlf"] and h.delimiter == 0x2C


def test_header_new_fuzz_vs_oracle():
    for seed in range(200):
        data = cases.rand_bytes(40 + seed, 5000 + seed, weights=[5, 5, 5, 2, 1, 0.3, 0.3, 2, 1, 0.2, 0.2])
        try:
            want = O.header_new(data)
        except O.OraclePanic:
            with pytest.raises(cs.ReferencePanic):
                cs.Header.new(cs.Mmap(data=data))
            continue
        got = cs.Header.new(cs.Mmap(data=data))
        assert got.field_cnt == want.field_cnt and got.record_offset == want.record_offset
        assert (got.new_line is cs.NewLine.CRLF) == want.crlf


def test_header_bom_and_long_first_line():
    data = b"\xef\xbb\xbf" + b",".join(b"col%d" % i for i in range(3000)) + b"\r\nrest\r\n"
    h = cs.Header.new(cs.Mmap(data=data))
    assert h.field_cnt == 3000 and h.header[0] == "col0" and h.new_line is cs.NewLine.CRLF
    assert h.field_cnt == O.header_new(data).field_cnt


def test_boundaries_doctest_and_oracle():
    # src/tape.rs:362-384
    r = cs.boundaries(8, 3)
    assert [(b.start, b.len) for b in r] == [(0, 3), (3, 3), (6, 2)]
    r = cs.boundaries(1000, 12)
    assert (r[0].start, r[0].len) == (0, 84) and (r[1].start, r[1].len) == (84, 84)
    assert (r[11].start, r[11].len) == (917, 83) and sum(b.len for b in r) == 1000
    assert [(b.start, b.len) for b in cs.boundaries(8, 12)] == [(0, 8)]
    assert cs.boundaries(0, 3) is None
    for task in (1, 2, 7, 255, 256, 257, 1000, 65537, 2 ** 32 - 1):
        for jobs in (1, 2, 3, 12, 255):
            got = cs.boundaries(task, jobs)
            assert [(b.start, b.len) for b in got] == O.boundaries(task, jobs), (task, jobs)


def test_chunks_matches_oracle():
    for rc, jump, num in ((15, 3, 4), (8, 9, 3), (1000, 16, 12), (3, 5, 7)):
        t = cs.Tape(cs.Header(["a"], cs.NewLine.LF, jump, 0x2C, 0), rc, jump, cs.Mmap(data=b""), None)
        got = [dict(id=c.id, start=c.start, end=c.end, record_cnt=c.record_cnt) for c in t.chunks(num)]
        assert got == O.chunks(rc, jump, num)
    t = cs.Tape(cs.Header(["a"], cs.NewLine.LF, 1, 0x2C, 0), 0, 1, cs.Mmap(data=b""), None)
    with pytest.raises(cs.InvalidState):
        t.chunks(3)


def test_create_missing_file_is_io_error():
    with pytest.raises(cs.Io):
        cs.create("/nonexistent/definitely_missing.csv")


def test_carry_and_base_scans_match_oracle():
    data = np.frombuffer(cases.rand_bytes(20000, 77), dtype=np.uint8)
    cuts = [0, 4999, 5000, 12345, 20000]
    summ = [O.shard_summary(data[cuts[k]:cuts[k + 1]]) for k in range(4)]
    carries = csd.carry_in_parities([s[0] for s in summ])
    counts = [(s[2] - s[1]) if c else s[1] for s, c in zip(summ, carries)]
    counts[0] += 1  # sentinel on rank 0
    bases = csd.exclusive_bases(counts)
    full = O.closed_form_numpy(data)
    assert sum(counts) == full.size
    for k in range(4):
        seg = O.closed_form_numpy(data[cuts[k]:cuts[k + 1]], carries[k], cuts[k], with_sentinel=(k == 0))
        assert (seg == full[bases[k]:bases[k] + counts[k]]).all()


def test_speculative_verify_math_matches_oracle():
    """Any guessed carries: verify_speculation recovers the true carries and entry counts (c0 + c1 = total)."""
    data = np.frombuffer(cases.rand_bytes(40000, 5), dtype=np.uint8)
    cuts = [0, 7001, 7002, 19999, 33333, 40000]
    full = O.closed_form_numpy(data)
    for guess_bits in range(32):
        gathered = []
        for k in range(5):
            shard = data[cuts[k]:cuts[k + 1]]
            p, c0, s = O.shard_summary(shard)
            used = 0 if k == 0 else (guess_bits >> k) & 1
            gathered.append(((s - c0) if used else c0, p ^ used, used, s))
        carries, counts, redo = csd.verify_speculation(gathered)
        assert carries == csd.carry_in_parities([O.shard_summary(data[cuts[k]:cuts[k + 1]])[0] for k in range(5)])
        assert redo == [carries[k] != gathered[k][2] for k in range(5)]
        assert 1 + sum(counts) == full.size
        bases = csd.exclusive_bases([counts[0] + 1] + counts[1:])
        for k in range(5):
            seg = O.closed_form_numpy(data[cuts[k]:cuts[k + 1]], carries[k], cuts[k], with_sentinel=(k == 0))
            assert (seg == full[bases[k]:bases[k] + seg.size]).all()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        data = np.frombuffer(cases.rand_bytes(30001, 99), dtype=np.uint8)
        cut = 14567  # arbitrary, unaligned
        lo, hi = (0, cut) if rank == 0 else (cut, data.size)
        shard = data[lo:hi]
        p, c0, s = O.shard_summary(shard)                     # stands in for pass A on this rank
        carry, ps = csd.exchange_parity(p)                    # the real exchange code, gloo backend
        seg = O.closed_form_numpy(shard, carry, lo, with_sentinel=(rank == 0))   # stands in for pass B
        base, total = csd.exchange_counts(seg.size)
        full = O.closed_form_numpy(data)
        ok = total == full.size and (seg == full[base:base + seg.size]).all() and len(ps) == world
        # speculative protocol: both ranks guess 0, ONE all_gather of 4 words, verify on every rank
        import torch
        mine = torch.tensor([c0, p, 0, s], dtype=torch.int64)
        allr = torch.empty(4 * world, dtype=torch.int64)
        dist.all_gather_into_tensor(allr, mine)
        carries, counts, redo = csd.verify_speculation(allr.view(world, 4).tolist())
        seg2 = O.closed_form_numpy(shard, carries[rank], lo, with_sentinel=(rank == 0))
        ok = ok and carries[rank] == carry and counts[rank] + (rank == 0) == seg2.size and (seg2 == seg).all()
        ok = ok and redo[rank] == (carry != 0) and 1 + sum(counts) == full.size
        # replicated index: gather_segments puts the whole index on every rank (gloo stands in for NCCL)
        seg_t = torch.from_numpy(seg.view(np.int64).copy())
        cnts = [counts[0] + 1, counts[1]]
        full_t = csd.gather_segments(seg_t, cnts)
        ok = ok and full_t.numel() == full.size and (full_t.numpy().view(np.uint64) == full).all()
        q.put((rank, bool(ok), carry))
    finally:
        dist.destroy_process_group()


def test_two_rank_exchange_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert [r[1] for r in res] == [True, True]
    assert res[0][2] == 0


def test_bench_reference_arm_contract():
    """bench.py --impl reference runs the reference's CPU path (the oracle) without a GPU and prints ONE JSON
    line with the contract's keys; under a multi-rank launch only rank 0 prints."""
    import json
    import subprocess
    env = dict(os.environ, RANK="0", LOCAL_RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "25",
                          "--warmup", "1", "--size", str(8 << 20)], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "csv_bytes_indexed_per_sec" and d["unit"] == "GB/s"
    assert d["steps"] == 25   # --steps is the number of timed steps, whatever it is
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["config"]["workload"]
    env["RANK"] = "1"
    env["WORLD_SIZE"] = "2"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--size", str(1 << 20)], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_dump_stays_within_budget_for_every_world_size(tmp_path):
    """bench.py --dump-outputs: every rank writes its own segment, and all ranks' files together stay within 64 MB
    (each rank takes 1/world of the sample and the edges); the values are the index's own."""
    import bench

    class FakeIndex:
        end_parity = 1

        def __init__(self, k):
            self.host = np.arange(3_000_000, dtype=np.uint64) * np.uint64(7) + np.uint64(k)

        def to_host(self):
            return self.host

    for world in (1, 2, 8):
        d = tmp_path / f"w{world}"
        written = sum(bench.dump_index(FakeIndex(k), str(d), k, world) for k in range(world))
        files = sorted(os.listdir(d))
        assert written == sum(os.path.getsize(d / f) for f in files) <= bench.DUMP_MAX_BYTES, world
        assert len(files) == 7 * world and all(f.endswith(".npy") for f in files)
        for k in range(world):
            sfx = f"_rank{k}" if world > 1 else ""
            host = FakeIndex(k).host
            pos = np.load(d / f"index_sample_pos{sfx}.npy").astype(np.int64)
            assert np.load(d / f"index_len{sfx}.npy").tolist() == [host.size]
            assert pos.size > 0 and (np.load(d / f"index_sample{sfx}.npy") == host[pos]).all()
            sums = np.load(d / f"index_block_sums{sfx}.npy")
            assert sums.dtype == np.float64 and int(sums.astype(np.uint64).sum(dtype=np.uint64)) == int(host.sum(dtype=np.uint64))


def test_numa_helpers():
    from csv_simd_b200 import numa
    assert numa._parse_cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11]
    assert numa._parse_cpulist("") == []
    assert numa.device_numa_node("0000:ff:1f.7") in (None, 0, 1, 2, 3, 4, 5, 6, 7)
