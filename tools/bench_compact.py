"""What the storage form of the device-resident index costs and saves, for one context (run it once with
CSVB200_INDEX_ENTRY_BYTES=8 and once without, in the same session, to compare the two forms):
  * the build kernel's time (csvb200_ctx_last_build_ms, mean of --steps builds) and its true bytes, N + 4E for 4-byte
    entries and N + 8E for 8-byte ones, over that time, as a fraction of a device-to-device copy rate measured here
    (torch copy of a --size buffer: read + write bytes over time);
  * csvb200_index_copy_out into a pinned buffer (for a compact index: widened on the device in chunks on the way);
  * the first csvb200_index_device_ptr call (for a compact index: the one-time conversion to u64 entries).
Prints one JSON line per workload, with the card's name and power limit.

    python tools/bench_compact.py [--size BYTES] [--steps K]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import csv_simd_b200 as cs  # noqa: E402
from tools import gen  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the numbers stay valid, the label is missing
        return f"unknown ({e})"


def copy_rate_gbs(dev, nbytes, steps=20):
    a = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize(dev)
    return 2 * nbytes * steps / (e0.elapsed_time(e1) * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1 << 30)
    ap.add_argument("--steps", type=int, default=30)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    ctx = cs.Context(0)
    entry_bytes = 8 if os.environ.get("CSVB200_INDEX_ENTRY_BYTES") == "8" else 4
    copy_gbs = copy_rate_gbs(dev, args.size)
    for name, make in (("cfg2_unquoted", lambda: gen.unquoted(args.size, seed=42)[0]),
                       ("cfg3_quoted", lambda: gen.quoted(args.size, seed=43)[0])):
        data = make()
        n = int(data.size)
        d_in = torch.empty(n + 64, dtype=torch.uint8, device=dev)
        d_in[:n].copy_(torch.from_numpy(data))
        torch.cuda.synchronize(dev)
        kms = []
        for i in range(args.steps + 3):
            idx = ctx.index_build_device(d_in.data_ptr(), n)
            idx.sync()
            if i >= 3:
                kms.append(ctx.last_build_ms())
            E = len(idx)
            idx.free()
        k_ms = sum(kms) / len(kms)
        true_bytes = n + (4 if entry_bytes == 4 and n <= (1 << 32) else 8) * E
        h_out = torch.empty(E, dtype=torch.int64).pin_memory()
        copy_ms, conv_ms = [], []
        for _ in range(5):
            idx = ctx.index_build_device(d_in.data_ptr(), n)
            idx.sync()
            t0 = time.perf_counter()
            idx.copy_out_ptr(h_out.data_ptr(), E)
            copy_ms.append((time.perf_counter() - t0) * 1e3)
            t0 = time.perf_counter()
            assert idx.device_ptr != 0
            conv_ms.append((time.perf_counter() - t0) * 1e3)   # ends in a synchronisation of the context's stream
            idx.free()
        print(json.dumps({
            "workload": name, "n": n, "entries": E, "entry_bytes": entry_bytes, "card": card(),
            "kernel_ms": k_ms, "kernel_ms_min_max": [min(kms), max(kms)],
            "true_bytes_per_launch": true_bytes, "true_gbs": true_bytes / (k_ms * 1e-3) / 1e9,
            "copy_rate_gbs": copy_gbs, "frac_of_copy_rate": true_bytes / (k_ms * 1e-3) / 1e9 / copy_gbs,
            "frac_of_6453_4_gbs": true_bytes / (k_ms * 1e-3) / 1e9 / 6453.4,
            "copy_out_pinned_ms": sorted(copy_ms)[len(copy_ms) // 2], "first_device_ptr_ms": sorted(conv_ms)[len(conv_ms) // 2],
        }), flush=True)
        del d_in
    ctx.close()


if __name__ == "__main__":
    main()
