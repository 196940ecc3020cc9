#!/usr/bin/env python
"""bench.py -- CSV bytes indexed per second (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--no-also]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (csv bytes -> structural index) over one batch of synthetic
CSV.  N=1: BASELINE config 2 (1 GiB unquoted, 16 numeric fields/row, LF).  N>1: BASELINE config 4
(quote-heavy CRLF grammar sharded at arbitrary byte offsets, 1 GiB per GPU, weak scaling: the logical file
is the concatenation of N seeded 1 GiB row streams cut at start + 37k + 13) with the cross-shard
quote-parity exchange inside every step.

  value      whole-job CSV GB/s with the input already resident in HBM (max over ranks, CUDA events)
  e2e        the same metric through the public host-buffer C-ABI call: pinned host bytes in,
             host index out, H2D + kernels + D2H all inside the timed region
  roofline   dominant kernel (index_build_tma_kernel): algorithmic bytes N + 8E per launch / average
             launch duration (CUDA events around each launch) vs the measured HBM copy peak
  parity     (N>1) every rank's device-resident segment AND its end-to-end host segment compared element-wise
             with the oracle's closed form of the same shard under the ORACLE's carry chain
  also       the other BASELINE configs measured in the same run: config 3 (1 GiB quote-heavy, the one the
             north-star target is stated on) and config 5 (10 M lookups over a 4 GiB 256-field file) at N=1;
             at N>1 the same-grammar solo rate of rank 0's shard (-> efficiency_same_grammar) and, for
             N < 8, config 4 as written: ONE 8 GiB file cut N ways (strong scaling)
  cpu_baseline / --impl reference
             the reference's CPU path (oracle/csv_oracle.c: the literal SSE restatement, 1 thread
             because the reference is a single serial loop) on the box's host cores

--impl reference times exactly --steps passes like the CUDA arm; at about 1 GB/s on one core the default 100 steps
over 1 GiB take about 100 s, so pass a smaller --steps for a quicker reference line.

--dump-outputs DIR writes the index of the last timed step (all ranks' segments, sampled: dump_index) as float64
.npy files, at most 64 MB in all, so that two builds of the project can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GiB = 1 << 30
METRIC = "csv_bytes_indexed_per_sec"
UNIT = "GB/s"
STRONG_TOTAL_PIECES = 8     # config 4 as written: an 8 GiB file


# ---------------------------------------------------------------------------------------------
# workloads (deterministic generators, tools/gen_csv.c; SURVEY.md 8d)
# ---------------------------------------------------------------------------------------------
def _cut(k: int, world: int) -> int:
    """Shard k starts this many bytes past the start of its first row stream: NOT at a record boundary and not
    16-byte aligned in the file (SURVEY 8d config 4)."""
    return 0 if k == 0 or k >= world else 37 * k + 13


def make_workload(name: str, rank: int, world: int, size: int, pieces: int = 1):
    """Returns (bytes ndarray for this rank, description).  cfg4: the logical file is the concatenation of
    world * pieces seeded row streams of `size` bytes; rank k owns streams [k * pieces, (k + 1) * pieces) shifted
    by the cut offsets, i.e. G[kP][cut_k:] ++ ... ++ G[(k+1)P][:cut_{k+1}]."""
    from tools import gen
    if name == "cfg2_unquoted":
        data, _ = gen.unquoted(size, seed=42, first_row=rank << 32, with_header=(rank == 0))
        desc = "synthetic unquoted CSV, 16 numeric fields/row, LF (BASELINE config 2)"
    elif name == "cfg3_quoted":
        data, _ = gen.quoted(size, seed=43, first_row=rank << 32, with_header=(rank == 0))
        desc = "synthetic quote-heavy CSV: embedded commas, CRLF, newlines and \"\" escapes (BASELINE config 3)"
    elif name == "cfg4_sharded":
        first = rank * pieces
        out = [None] * pieces

        def one(j):
            out[j], _ = gen.quoted(size, seed=44, first_row=(first + j) << 32, with_header=(first + j == 0))
        ts = [threading.Thread(target=one, args=(j,)) for j in range(pieces)]   # the generator releases the GIL
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        parts = [out[0][_cut(rank, world):]] + out[1:]
        if rank + 1 < world:
            nxt, _ = gen.quoted(4096, seed=44, first_row=(first + pieces) << 32, with_header=False)
            parts.append(nxt[:_cut(rank + 1, world)])
        data = np.concatenate(parts) if len(parts) > 1 else parts[0]
        desc = ("synthetic quote-heavy CSV sharded at arbitrary byte offsets with cross-shard quote-parity "
                "fix-up (BASELINE config 4)")
    else:
        raise SystemExit(f"unknown workload {name}")
    return np.ascontiguousarray(data), desc


def config_block(wl, desc, n_rank0, total_bytes, entries, world, numa_node=None, **extra):
    """The `config` object of a bench line: the same keys for the repo arm and the reference arm."""
    cfg = {"workload": wl, "description": desc, "bytes_per_gpu": int(n_rank0), "total_bytes": int(total_bytes),
           "index_entries": int(entries), "index_entry_bytes": 8,
           "l2_policy": "input (1 GiB) and index (>= 0.5 GB) are far larger than the 126 MB L2; no flush",
           "parallelism": f"byte-range shards x{world}" if world > 1 else "single GPU",
           "host_numa_node_rank0": numa_node}
    cfg.update(extra)
    return cfg


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed regions (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                util = float(r[4])
                if util < 5 and len(self.rows) > 3:
                    continue
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                power.append(float(r[3]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload: str, n: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the hot kernel, from the committed
    ncu --set full capture of the same 1 GiB workload (profiles/); (None, why) when no capture matches.
    cfg4 shards are 1 GiB of the cfg3 grammar (another seed), so the cfg3 capture stands in for them."""
    for name in ("r02_traffic.json", "r01_v6_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                t = json.load(f)
            key = "cfg2" if workload == "cfg2_unquoted" else "cfg3"
            if abs(n - GiB) > (1 << 20):
                return None, "no ncu capture at this size"
            note = t[key]["source"] + ("; cfg4 shard = same grammar and size as cfg3" if workload == "cfg4_sharded" else "")
            return t[key]["traffic_bytes_per_launch"], note
        except Exception:  # noqa: BLE001
            continue
    return None, "profiles/*traffic.json unreadable"


def host_cpu():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return model, os.cpu_count()


def cpu_reference_gbs(data: np.ndarray, reps: int):
    """The reference's CPU path (literal SSE restatement, single thread) on this host."""
    from oracle import oracle as O
    buf = O.aligned_copy(data)
    buf.sum()  # pre-fault (the reference's mmap page faults are excluded, as BASELINE.md states)
    best, E = 0.0, 0
    for _ in range(reps):
        t = time.perf_counter()
        E, _ = O.read_sse_timed(buf)
        dt = time.perf_counter() - t
        best = max(best, buf.size / dt / 1e9)
    return best, E


# ---------------------------------------------------------------------------------------------
def run_reference(args, rank: int, world: int):
    """The reference arm: the reference's own CPU algorithm (the SSE restatement) on the SAME bytes rank 0 of the
    repo arm indexes (N=1: the cfg2 file; N>1: rank 0's cfg4 shard, seed 44), same config keys."""
    if rank != 0:
        return
    wl = args.workload or ("cfg2_unquoted" if world == 1 else "cfg4_sharded")
    size = args.size or GiB
    data, desc = make_workload(wl, 0, world, size)
    from oracle import oracle as O
    buf = O.aligned_copy(data)
    buf.sum()
    for _ in range(min(args.warmup, 1)):
        O.read_sse_timed(buf)
    t = time.perf_counter()
    for _ in range(args.steps):
        E, _ = O.read_sse_timed(buf)
    dt = time.perf_counter() - t
    gbs = buf.size * args.steps / dt / 1e9
    model, ncpu = host_cpu()
    sample = (f"{buf.size} bytes per step = rank 0's shard of the repo arm's workload ({wl}), single thread: the "
              f"reference is one serial loop (src/reader.rs:229-258); host {model}, {ncpu} logical cpus")
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config_block(wl, desc, buf.size, buf.size * world if wl == "cfg4_sharded" else buf.size, E, world,
                               note="the reference is single-threaded: one shard per step on one host core"),
        "cpu_baseline": {"value": gbs, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": gbs, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


DUMP_SAMPLE = 1 << 21        # entries of the seeded random sample of the index, shared by all ranks
DUMP_EDGE = 1 << 16          # entries kept whole at each end of the index, shared by all ranks
DUMP_BLOCK = 1 << 16         # entries per block sum: every entry counts, each sum exact in float64
DUMP_MAX_BYTES = 64 << 20    # all ranks' files together


def dump_index(idx, out_dir: str, rank: int = 0, world: int = 1) -> int:
    """Writes what a caller of the build receives (the host index and its end quote parity) as float64 .npy files;
    returns the bytes written.  The index itself is too large to store whole, so it is kept as its length, its first
    and last entries, a sample at positions drawn from a fixed seed, and exact sums of consecutive blocks of
    DUMP_BLOCK entries (a difference anywhere in the index changes one of them).  Positions are < 2^53, so float64
    holds them exactly.  With world > 1 every rank writes its own segment (suffix _rank<k>) with 1/world of the
    sample, the edges and the byte budget, so that all ranks' files together stay within DUMP_MAX_BYTES."""
    host = idx.to_host()
    E = host.size
    sample, edge = DUMP_SAMPLE // world, DUMP_EDGE // world
    assert E == 0 or int(host.max()) * DUMP_BLOCK < (1 << 53), "index positions too large for exact float64 block sums"
    pos = np.unique(np.random.default_rng(rank).integers(0, E, size=min(E, sample))) if E else np.zeros(0, np.int64)
    full = E - E % DUMP_BLOCK
    sums = host[:full].reshape(-1, DUMP_BLOCK).sum(axis=1, dtype=np.uint64)
    if full < E:
        sums = np.append(sums, host[full:].sum(dtype=np.uint64))
    arrays = {
        "index_len": np.array([E], dtype=np.float64),
        "end_parity": np.array([idx.end_parity], dtype=np.float64),
        "index_head": host[:edge].astype(np.float64),
        "index_tail": host[max(E - edge, 0):].astype(np.float64),
        "index_sample_pos": pos.astype(np.float64),
        "index_sample": host[pos].astype(np.float64),
        "index_block_sums": sums.astype(np.float64),
    }
    budget = DUMP_MAX_BYTES // world
    assert sum(a.nbytes for a in arrays.values()) <= budget, f"dump of rank {rank} exceeds its {budget} bytes"
    os.makedirs(out_dir, exist_ok=True)
    written = 0
    for name, a in arrays.items():
        path = os.path.join(out_dir, name + (f"_rank{rank}" if world > 1 else "") + ".npy")
        np.save(path, a)
        written += os.path.getsize(path)
    return written


def pcie_probe(torch, dev, mb: int = 256, reps: int = 3):
    """Pinned H2D and D2H running at the same time (what bounds the end-to-end path): GB/s per direction."""
    n = mb << 20
    h_a = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_b = torch.empty(n, dtype=torch.uint8).pin_memory()
    d_a = torch.empty(n, dtype=torch.uint8, device=dev)
    d_b = torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def run(up, down):
        torch.cuda.synchronize(dev)
        t = time.perf_counter()
        for _ in range(reps):
            if up:
                with torch.cuda.stream(s1):
                    d_a.copy_(h_a, non_blocking=True)
            if down:
                with torch.cuda.stream(s2):
                    h_b.copy_(d_b, non_blocking=True)
        torch.cuda.synchronize(dev)
        return n * reps / (time.perf_counter() - t) / 1e9
    run(True, True)
    return {"h2d_alone_gbs": run(True, False), "d2h_alone_gbs": run(False, True), "duplex_each_gbs": run(True, True),
            "copy_mb": mb}


def run_ours(args, rank: int, local_rank: int, world: int):
    import torch
    import torch.distributed as dist

    import csv_simd_b200 as cs
    from csv_simd_b200 import dist as csd
    from oracle import oracle as O   # the checker (parity blocks, cpu_baseline); never on the measured path

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from csv_simd_b200 import numa
    numa_node = numa.bind_to_device(local_rank)   # pinned staging buffers on the GPU's own NUMA node
    numa_why = None if numa_node is not None else numa.why_unbound(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = args.workload or ("cfg2_unquoted" if world == 1 else "cfg4_sharded")
    size = args.size or GiB
    peak, peak_src = hbm_peak()

    ctx = cs.Context(local_rank)
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)  # our kernels run on torch's current stream: torch events bracket them
    # the cross-shard exchange: peer-mapped mailboxes written from inside the build launch (default), or the round-1
    # path (NCCL all_gather + verify launch) with --exchange nccl for an A/B on the same box
    ex = csd.make_exchange(ctx) if (world > 1 and args.exchange == "p2p") else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def all_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_sum_int(*xs):
        if world == 1:
            return [int(x) for x in xs]
        t = torch.tensor(list(xs), dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [int(v) for v in t.tolist()]

    def gather_obj(x):
        if world == 1:
            return [x]
        out = [None] * world
        dist.all_gather_object(out, x)
        return out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # -----------------------------------------------------------------------------------------
    def measure(wl_name, data, sharded, steps, e2e_steps_cap=10, check=True, ex_=None, dump_dir=None):
        """One workload on this rank's bytes: device-resident steps (value), per-launch kernel time (roofline),
        end-to-end host->host steps (e2e), and -- sharded -- element-wise parity against the oracle.  With dump_dir,
        the index of the last timed step is written there (dump_index) once the timing is over."""
        n = int(data.size)
        sizes = [int(v) for v in gather_obj(n)] if sharded else [n]
        goff = sum(sizes[:rank]) if sharded else 0
        total_bytes = sum(sizes)
        d_in = torch.empty(n + 64, dtype=torch.uint8, device=dev)
        d_in[:n].copy_(torch.from_numpy(data))
        torch.cuda.synchronize(dev)

        def step_device(resolve=True):
            # resolve=False: nothing in the step waits on the host (the timed loops); the index, its length
            # and (sharded) every rank's counts are complete in HBM when the stream reaches the end event
            if not sharded:
                idx = ctx.index_build_device(d_in.data_ptr(), n)
                if resolve:
                    idx.sync()
                return idx
            return csd.sharded_index_build(ctx, d_in.data_ptr(), n, goff, resolve=resolve, exchange=ex_).local

        E, carry_in = 0, 0
        for _ in range(max(args.warmup, 3)):
            idx = step_device()
            E = len(idx)
            idx.free()
        res = {"n": n, "total_bytes": total_bytes, "goff": goff}
        parity = None
        if sharded:
            sh = csd.sharded_index_build(ctx, d_in.data_ptr(), n, goff, exchange=ex_)
            carry_in, E = sh.carry_in, len(sh.local)
            if check:
                # the oracle's own carry chain: shard parities -> exclusive XOR scan; closed form of this shard
                op, _c0, _s = O.shard_summary(data)
                pars = gather_obj(int(op))
                ocarry = 0
                for p_ in pars[:rank]:
                    ocarry ^= p_ & 1
                want, _ = O.read_closed_form(data, ocarry, goff, with_sentinel=(rank == 0))
                obase = sum(int(c) for c in gather_obj(int(want.size))[:rank])
                got = sh.local.to_host()
                parity = {"dev_ok": bool(sh.carry_in == ocarry and sh.base == obase and got.size == want.size
                                         and np.array_equal(got, want)),
                          "want": want}
            sh.local.free()

        # ---- value: K device-resident steps, CUDA events, max over ranks ----
        for _ in range(3):   # unsynchronised steps right before the timed ones: the pool blocks of this shape exist
            step_device(resolve=False).free()
        launches0 = ctx.launch_count()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = []
        e0.record(stream)
        for i in range(steps):
            idx = step_device(resolve=False)
            if dump_dir is None or i + 1 < steps:
                idx.free()
            if i < 64:   # per-step marks (diagnostic: a stall of one step shows up as max >> median)
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(stream)
                marks.append(ev)
            if sharded and (i + 1) % 512 == 0 and i + 1 < steps:
                barrier()   # the mailbox ring holds 1024 builds: no rank may run further ahead of the slowest one
        e1.record(stream)
        barrier()
        ms_mine = e0.elapsed_time(e1)
        per = [a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks)]
        res["step_ms_median_max_rank"] = [float(statistics.median(per)), float(max(per))] if per else None
        res["ms_per_step_by_rank"] = [float(v) / steps for v in gather_obj(ms_mine)]
        ms_total = all_max(ms_mine)
        launches = ctx.launch_count() - launches0
        launches, E_total = all_sum_int(launches, E)
        res.update(ms_per_step=ms_total / steps, launches=launches, E_total=E_total)
        res["value"] = total_bytes / (res["ms_per_step"] * 1e-3) / 1e9
        if dump_dir is not None:
            written = dump_index(idx, dump_dir, rank, world)
            idx.free()
            written = all_sum_int(written)[0]   # every rank's files: the directory as a whole stays within the budget
            assert written <= DUMP_MAX_BYTES, f"--dump-outputs wrote {written} bytes, more than {DUMP_MAX_BYTES}"

        # ---- roofline of the dominant kernel: per-launch duration from events around each launch ----
        kms = []
        E_local = E
        for _ in range(min(steps, 50)):
            if not sharded:
                idx = ctx.index_build_device(d_in.data_ptr(), n)
            else:
                idx = ctx.index_build_shard_device(d_in.data_ptr(), n, carry_in, goff, rank == 0)
            idx.sync()
            kms.append(ctx.last_build_ms())
            E_local = len(idx)
            idx.free()
        k_ms = sum(kms) / len(kms)
        alg_bytes = n + 8 * E_local
        res.update(kernel_ms=k_ms, alg_bytes=alg_bytes, E_local=E_local,
                   achieved=alg_bytes / (k_ms * 1e-3) / 1e9)
        # same-grammar solo rate of THIS rank's bytes (no exchange, no other rank involved): device steps
        if sharded:
            barrier()
            e0.record(stream)
            for _ in range(min(steps, 50)):
                idx = ctx.index_build_shard_device(d_in.data_ptr(), n, carry_in, goff, rank == 0)
                idx.free()
            e1.record(stream)
            torch.cuda.synchronize(dev)
            res["solo_ms_per_step"] = all_max(e0.elapsed_time(e1) / min(steps, 50))

        # ---- e2e: pinned host bytes -> C-ABI -> host index (H2D + kernels + D2H inside the timed region) ----
        h_in = torch.from_numpy(data).pin_memory()
        h_out = torch.empty(E_local + 1024, dtype=torch.int64).pin_memory()
        e2e_steps = max(3, min(steps, e2e_steps_cap))
        redone_any = []

        def step_e2e():
            if not sharded:
                return ctx.index_build_to_host(h_in.data_ptr(), n, h_out.data_ptr(), h_out.numel())
            ln_, _base, _total, redone = csd.sharded_index_build_to_host(ctx, h_in.data_ptr(), n, goff, h_out.data_ptr(),
                                                                         h_out.numel(), exchange=ex_)
            if redone:
                redone_any.append(rank)
            return ln_

        barrier()   # page-locking the buffers above takes a different time on every rank: line the ranks up first
        for _ in range(2):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            ln = step_e2e()
        barrier()
        e2e_s = all_max((time.perf_counter() - t0) / e2e_steps)
        assert ln == E_local, (ln, E_local)
        res.update(e2e_s=e2e_s, e2e_steps=e2e_steps, e2e_gbs=total_bytes / e2e_s / 1e9)
        if parity is not None:
            want = parity.pop("want")
            got = h_out.numpy()[:ln].view(np.uint64)
            parity["e2e_ok"] = bool(got.size == want.size and np.array_equal(got, want))
            oks = gather_obj((parity["dev_ok"], parity["e2e_ok"], sorted(set(redone_any))))
            res["parity"] = {"checked": True,
                             "what": "element-wise: device-resident segment and end-to-end host segment of every rank "
                                     "== oracle closed form of the shard under the oracle's own carry chain; carry-in "
                                     "and segment base == oracle's",
                             "ranks_ok": sum(1 for a, b, _ in oks if a and b), "ranks": world,
                             "device_path_ok": [bool(a) for a, _, _ in oks], "e2e_path_ok": [bool(b) for _, b, _ in oks],
                             "redone": sorted({r for _, _, rs in oks for r in rs})}
        res["_h_in"], res["_h_out"], res["_d_in"] = h_in, h_out, d_in
        return res

    # ---- the headline workload -------------------------------------------------------------------------
    data, desc = make_workload(wl, rank, world, size)
    sharded = world > 1 and wl == "cfg4_sharded"
    m = measure(wl, data, sharded, args.steps, ex_=ex, dump_dir=args.dump_outputs)
    n, E_local = m["n"], m["E_local"]

    # the same call on ordinary (pageable) memory, as a caller holding an mmap and a Vec would make it: informational
    e2e_pageable = None
    if world == 1:
        out_pg = np.empty(E_local + 1024, dtype=np.uint64)
        out_pg[::512] = 0
        ctx.index_build_to_host(data.ctypes.data, n, out_pg.ctypes.data, out_pg.size)
        t0 = time.perf_counter()
        for _ in range(3):
            ctx.index_build_to_host(data.ctypes.data, n, out_pg.ctypes.data, out_pg.size)
        e2e_pageable = n / ((time.perf_counter() - t0) / 3) / 1e9
        del out_pg
    for k in ("_h_in", "_h_out", "_d_in"):
        m.pop(k, None)
    torch.cuda.empty_cache()

    # PCIe ceiling of this box, measured now (all ranks at once when N>1): what bounds e2e
    barrier()
    pcie = pcie_probe(torch, dev)
    pcie_all = gather_obj(pcie)
    h2d_t = n / (pcie["duplex_each_gbs"] * 1e9)
    d2h_t = 8 * E_local / (pcie["duplex_each_gbs"] * 1e9)
    e2e_bound_s = all_max(max(h2d_t, d2h_t))

    clocks = sampler.stop() if rank == 0 else None

    # ---- also: the other BASELINE configs, same run ------------------------------------------------------
    also = {}
    if not args.no_also:
        if world == 1 and wl == "cfg2_unquoted":
            d3, desc3 = make_workload("cfg3_quoted", 0, 1, GiB)
            m3 = measure("cfg3_quoted", d3, False, min(args.steps, 50), e2e_steps_cap=5)
            for k in ("_h_in", "_h_out", "_d_in"):
                m3.pop(k, None)
            torch.cuda.empty_cache()
            cpu3, E3 = cpu_reference_gbs(d3, reps=2)
            assert E3 == m3["E_local"], (E3, m3["E_local"])
            also["cfg3_quoted_1gib"] = {
                "description": desc3, "bytes": m3["n"], "index_entries": m3["E_local"], "value": m3["value"], "unit": UNIT,
                "ms_per_step": m3["ms_per_step"], "kernel_ms": m3["kernel_ms"],
                "roofline": {"achieved": m3["achieved"], "peak": peak, "frac": m3["achieved"] / peak,
                             "algorithmic_bytes_per_launch": m3["alg_bytes"], "traffic": ncu_traffic("cfg3_quoted", m3["n"])[0]},
                "e2e": {"value": m3["e2e_gbs"], "unit": UNIT, "h2d_bytes_per_step": m3["n"],
                        "d2h_bytes_per_step": 8 * m3["E_local"]},
                "cpu_baseline": {"value": cpu3, "unit": UNIT, "cores": 1, "kind": "port",
                                 "sample": "full input, best of 2 passes, single thread"},
                "entries_equal_oracle": True}
            del d3
            also["cfg5_lookup"] = bench_cfg5(ctx, torch, dev, stream, O, peak)
        if sharded:
            # same-grammar efficiency: the slowest rank's solo step on its own shard / the sharded step
            also["solo_same_grammar"] = {"ms_per_step": m["solo_ms_per_step"],
                                         "csv_gbs_per_gpu": n / (m["solo_ms_per_step"] * 1e-3) / 1e9,
                                         "what": "index_build_shard_device on each rank's own shard with the true carry, no "
                                                 "exchange (max over ranks), device-resident"}
            also["efficiency_same_grammar"] = m["solo_ms_per_step"] / m["ms_per_step"]
            also["exchange"] = {
                "kind": "peer-mapped mailboxes, rows stored over NVLink from inside the build launch" if ex is not None
                        else "NCCL all_gather_into_tensor + verify launch (round 1)",
                "bytes_posted_per_rank_per_step": 40 * world, "bytes_read_per_rank_per_step": 40 * rank_count_below(world),
                "step_overhead_ms": m["ms_per_step"] - m["solo_ms_per_step"]}
            if ex is not None and not args.no_ab:
                # the round-1 exchange on the same bytes, same box: what the mailboxes replace
                m_old = measure("cfg4_sharded", data, True, min(args.steps, 30), e2e_steps_cap=3, check=False, ex_=None)
                for k in ("_h_in", "_h_out", "_d_in"):
                    m_old.pop(k, None)
                torch.cuda.empty_cache()
                also["exchange"]["nccl_allgather_ms_per_step"] = m_old["ms_per_step"]
                also["exchange"]["nccl_allgather_efficiency_same_grammar"] = m_old["solo_ms_per_step"] / m_old["ms_per_step"]
            if world < STRONG_TOTAL_PIECES and STRONG_TOTAL_PIECES % world == 0 and size == GiB:
                pieces = STRONG_TOTAL_PIECES // world
                ds, _ = make_workload("cfg4_sharded", rank, world, GiB, pieces=pieces)
                ms_ = measure("cfg4_sharded", ds, True, min(args.steps, 30), e2e_steps_cap=3, ex_=ex)
                for k in ("_h_in", "_h_out", "_d_in"):
                    ms_.pop(k, None)
                torch.cuda.empty_cache()
                also["strong_8gib"] = {
                    "what": "config 4 as written: ONE 8 GiB file (the same 8 row streams as the N=8 weak run) cut "
                            f"{world} ways at start + 37k + 13",
                    "total_bytes": ms_["total_bytes"], "bytes_per_gpu": ms_["n"], "index_entries": ms_["E_total"],
                    "ms_per_step": ms_["ms_per_step"], "ms_per_step_by_rank": ms_["ms_per_step_by_rank"],
                    "step_ms_median_max_rank0": ms_["step_ms_median_max_rank"],
                    "value": ms_["value"], "unit": UNIT,
                    "kernel_ms": ms_["kernel_ms"], "roofline_frac": ms_["achieved"] / peak,
                    "solo_ms_per_step": ms_["solo_ms_per_step"],
                    "efficiency_same_grammar": ms_["solo_ms_per_step"] / ms_["ms_per_step"],
                    "e2e": {"value": ms_["e2e_gbs"], "unit": UNIT}, "parity": ms_.get("parity")}
                del ds

    # ---- CPU baseline (rank 0, N=1 only): the reference's CPU path on this box's host cores ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        gbs, E_cpu = cpu_reference_gbs(data, reps=5)
        model, ncpu = host_cpu()
        assert E_cpu == E_local, (E_cpu, E_local)  # the oracle checks the GPU's entry count
        cpu = {"value": gbs, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": (f"full {n}-byte input, best of 5 passes, single thread (the reference is one serial loop, "
                          f"src/reader.rs:229-258); input pre-faulted in RAM, println!s omitted; host {model}, "
                          f"{ncpu} logical cpus")}

    if rank == 0:
        traffic = ncu_traffic(wl, n)
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config_block(wl, desc, n, m["total_bytes"], m["E_total"], world, numa_node,
                                   host_numa_unbound_reason=numa_why, ms_per_step_by_rank=m["ms_per_step_by_rank"],
                                   step_ms_median_max_rank0=m["step_ms_median_max_rank"]),
            "roofline": {"bound": "hbm", "kernel": "index_build_tma_kernel", "achieved": m["achieved"], "peak": peak,
                         "unit": "GB/s", "frac": m["achieved"] / peak, "traffic": traffic[0], "traffic_source": traffic[1],
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": m["alg_bytes"], "kernel_ms": m["kernel_ms"],
                         "csv_gbs_kernel_only": n / (m["kernel_ms"] * 1e-3) / 1e9},
            "cpu_baseline": cpu,
            "e2e": {"value": m["e2e_gbs"], "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": 8 * E_local,
                    "ms_per_step": m["e2e_s"] * 1e3, "steps": m["e2e_steps"], "pageable_buffers_gbs": e2e_pageable,
                    "pcie_probe_rank0": pcie, "pcie_duplex_each_gbs_all_ranks": [p_["duplex_each_gbs"] for p_ in pcie_all],
                    "pcie_bound_ms": e2e_bound_s * 1e3, "frac_of_pcie_bound": e2e_bound_s / m["e2e_s"],
                    "api": "csvb200_index_build_to_host" if not sharded else
                           "csvb200_shard_build_to_host + exchange + csvb200_shard_job_verify (csv_simd_b200.dist.sharded_index_build_to_host)"},
            "gpu_launches": m["launches"],
            "clocks": clocks,
        }
        if "parity" in m:
            line["parity"] = m["parity"]
        if also:
            line["also"] = also
        print(json.dumps(line), flush=True)
    if ex is not None:
        barrier()
        ex.close()
    if world > 1:
        dist.destroy_process_group()
    ctx.close()


def rank_count_below(world: int) -> float:
    """Average number of lower ranks whose rows a rank reads (rank k waits for k rows)."""
    return (world - 1) / 2.0


def bench_cfg5(ctx, torch, dev, stream, O, peak):
    """BASELINE config 5: 10 M random (record, field) lookups against the index of a 4 GiB 256-field CSV."""
    from tools import gen
    nq, steps = 10_000_000, 20
    data, rows = gen.unquoted(4 * GiB, seed=45, nfields=256, modulus=10 ** 15)
    n = int(data.size)
    d = torch.empty(n + 64, dtype=torch.uint8, device=dev)
    d[:n].copy_(torch.from_numpy(data))
    idx = ctx.index_build_device(d.data_ptr(), n)
    E = len(idx)
    build_ms = ctx.last_build_ms()
    rc, jump = idx.tape_init(256, False)
    assert rc == rows + 1 and jump == 256
    rec, fld = gen.queries(nq, rc, 256, seed=46)
    d_rec, d_fld = torch.from_numpy(rec.view(np.int32)).to(dev), torch.from_numpy(fld.view(np.int32)).to(dev)
    d_out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    for _ in range(3):
        idx.seek_fields_device(d_rec.data_ptr(), d_fld.data_ptr(), nq, d_out.data_ptr())
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        idx.seek_fields_device(d_rec.data_ptr(), d_fld.data_ptr(), nq, d_out.data_ptr())
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    got = d_out.cpu().numpy().view(np.uint64)
    # end to end: pinned host query arrays in, pinned host ranges out (chunked H2D / kernel / D2H pipeline)
    h_rec, h_fld = torch.from_numpy(rec.view(np.int32)).pin_memory(), torch.from_numpy(fld.view(np.int32)).pin_memory()
    h_out = torch.empty((nq, 2), dtype=torch.int64).pin_memory()
    import ctypes as C
    best = 1e9
    for _ in range(3):
        t = time.perf_counter()
        rcode = idx._lib.csvb200_seek_fields(idx._h, C.c_void_p(h_rec.data_ptr()), C.c_void_p(h_fld.data_ptr()), nq,
                                             C.c_void_p(h_out.data_ptr()))
        best = min(best, time.perf_counter() - t)
        assert rcode == 0
    assert (h_out.numpy().view(np.uint64) == got).all()
    host = idx.to_host()
    t = time.perf_counter()
    cs_cpu, hits = O.seek_fields_timed(host, n, rc, 256, False, rec, fld)
    cpu_s = time.perf_counter() - t
    live = got[:, 0] != np.uint64(0xFFFFFFFFFFFFFFFF)
    cs_gpu = int((got[live, 0] ^ (got[live, 1] << np.uint64(1))).sum(dtype=np.uint64))
    ok = bool(hits == int(live.sum()) and cs_cpu == cs_gpu)
    assert ok, "GPU lookups differ from the oracle"
    idx.free()
    del d, d_out
    torch.cuda.empty_cache()
    return {"metric": "batched_field_lookups_per_sec", "value": nq / (ms * 1e-3) / 1e6, "unit": "Mqueries/s",
            "config": {"csv_bytes": n, "fields_per_row": 256, "rows": int(rows), "index_entries": int(E), "queries": nq},
            "ms_per_batch": ms, "index_build_ms": build_ms,
            "roofline": {"bound": "hbm", "achieved": 40 * nq / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": 40 * nq / (ms * 1e-3) / 1e9 / peak,
                         "note": "40 algorithmic bytes per query (8 in, 16 gathered, 16 out); random 16-byte gathers "
                                 "over a 2.2 GB index are sector-bound"},
            "e2e": {"value": nq / best / 1e6, "unit": "Mqueries/s", "h2d_bytes_per_step": 8 * nq, "d2h_bytes_per_step": 16 * nq},
            "cpu_baseline": {"value": nq / cpu_s / 1e6, "unit": "Mqueries/s", "cores": 1, "kind": "port",
                             "sample": "all 10 M queries, scalar seek_field restatement without the println!s"},
            "parity": {"checked": True, "ok": ok, "what": "hit count and checksum of all (start, end) pairs == oracle seek_field"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=[None, "cfg2_unquoted", "cfg3_quoted", "cfg4_sharded"])
    ap.add_argument("--size", type=int, default=None, help="bytes per GPU (default 1 GiB)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the `also` block (the other BASELINE configs)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: cross-shard exchange over peer-mapped mailboxes (default) or the round-1 NCCL all_gather")
    ap.add_argument("--no-ab", action="store_true", help="N>1: skip the A/B run of the round-1 exchange")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the index of the last timed step to DIR/<name>.npy (float64; sampled, see dump_index) "
                         "so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N")
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
