"""Validation of a distributed index (csvb200_multi_tape_validate, csvb200_multi_validate_utf8), config 4: G GiB of
quote-heavy CRLF CSV, 1 GiB per GPU, default cuts, at G = 1, 2 and 8.  One JSON line per (G, call):

  - wall time of the host call (every device checks its own segment / shard, the host joins the answers);
  - kernel time from torch.profiler in a separate run: per device the summed duration of the call's kernels, then the
    max over devices;
  - the one-GPU call on one GPU's 1 GiB share (the first part) as the reference point: csvb200_tape_validate on an index
    with 8-byte entries (CSVB200_INDEX_ENTRY_BYTES=8, as the distributed segments hold), and K7 on that share already on
    the device (csvb200_validate_utf8_device, so that the upload of csvb200_validate_utf8 is not in its time);
  - parity: the distributed answer equals the one-GPU answer on the share (both inputs are well-formed, so both report
    no bad slot and no ill-formed sequence, and the same is_ascii).

Config 4 is ASCII and only exercises K7's fast path, so a third line per G runs csvb200_multi_validate_utf8 on multi-byte
UTF-8 text (1 GiB per GPU, 87 % non-ASCII bytes).  The name and power limit of the cards are read with nvidia-smi in the
same run.  With fewer GPUs than G, device 0 is listed G times; its shards then run one after another and the line says
so ("emulated").

    python tools/bench_multi_validate.py [--gpus 1,2,8] [--steps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

os.environ["CSVB200_INDEX_ENTRY_BYTES"] = "8"   # before any context exists: the one-GPU K5 reads 8-byte entries too

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import csv_simd_b200 as cs  # noqa: E402
from tools import gen  # noqa: E402

GiB = 1 << 30
TEXT = "αβγ,δεζ\nκόσμε,\U0001F642\n".encode()
NONASCII = sum(b >= 0x80 for b in TEXT) / len(TEXT)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout
    return [line.strip() for line in out.splitlines() if line.strip()]


def make_data(G):
    parts = [None] * G
    ts = [threading.Thread(target=lambda j=j: parts.__setitem__(j, gen.quoted(GiB, seed=44, first_row=j << 32,
                                                                              with_header=(j == 0))[0].copy()))
          for j in range(G)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return np.concatenate(parts), int(parts[0].size)


def timed(fn, steps):
    fn()
    best = 1e9
    for _ in range(steps):
        t = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t)
    return best


def kernel_ms(fn, key):
    """per device: summed ms of the kernels whose name holds `key` in one call (torch.profiler, CUPTI)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and key in e.name:
            per[e.device_index] = per.get(e.device_index, 0.0) + e.time_range.elapsed_us() / 1e3
    return per


def line(G, devs, ndev, cards, call, workload, nbytes, wall, per, ref):
    return {"bench": "multi_validate", "call": call, "gpus": G, "devices": devs, "emulated": ndev < G, "cards": cards,
            "workload": workload, "bytes": nbytes, "wall_s": wall,
            "kernel_ms_max_over_devices": max(per.values()) if per else None,
            "per_device_kernel_ms": {str(k): v for k, v in sorted(per.items())}, "one_gpu_reference": ref}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,8")
    ap.add_argument("--steps", type=int, default=5)
    a = ap.parse_args()
    cards = gpu_info()
    ndev = torch.cuda.device_count()
    ctx = cs.Context(0)
    for G in [int(x) for x in a.gpus.split(",")]:
        devs = list(range(G)) if ndev >= G else [0] * G
        data, share = make_data(G)
        wl = "cfg4 grammar (quoted, CRLF, 16 fields), 1 GiB per GPU, default cuts"
        # reference: the first 1 GiB part on one GPU
        idx = ctx.index_build(data[:share], cs.BUILD_KEEP_BYTES)
        ref_rep = idx.tape_validate(16, True)
        d_share = torch.from_numpy(data[:share]).to(f"cuda:{ctx.device}")
        d_res = torch.empty(2, dtype=torch.int64, device=f"cuda:{ctx.device}")

        def ref_utf8():
            ctx.validate_utf8_device(d_share.data_ptr(), share, d_res.data_ptr())
            torch.cuda.synchronize(ctx.device)
            r = d_res.cpu().numpy().view(np.uint64)
            return (None if r[0] == 0xFFFFFFFFFFFFFFFF else int(r[0])), not bool(r[1])

        ref_u = ref_utf8()
        m = cs.Multi(devs)
        mi = m.index_build_distributed(data)
        rep = mi.tape_validate(16, True)
        ok = rep["ok"] == ref_rep["ok"] == 1 and rep["first_bad_slot"] == ref_rep["first_bad_slot"] and rep["problem"] == 0
        out = line(G, devs, ndev, cards, "csvb200_multi_tape_validate", wl, int(data.size),
                   timed(lambda: mi.tape_validate(16, True), a.steps), kernel_ms(lambda: mi.tape_validate(16, True), "tape_validate"),
                   {"call": "csvb200_tape_validate (8-byte entries)", "bytes": share,
                    "wall_s": timed(lambda: idx.tape_validate(16, True), a.steps),
                    "kernel_ms": sum(kernel_ms(lambda: idx.tape_validate(16, True), "tape_validate").values())})
        out["parity"] = {"ok": bool(ok), "what": "ok and first_bad_slot equal the one-GPU report on the share"}
        print(json.dumps(out), flush=True)
        u = mi.validate_utf8()
        out = line(G, devs, ndev, cards, "csvb200_multi_validate_utf8", wl, int(data.size),
                   timed(mi.validate_utf8, a.steps), kernel_ms(mi.validate_utf8, "utf8_validate"),
                   {"call": "csvb200_validate_utf8_device", "bytes": share, "wall_s": timed(ref_utf8, a.steps),
                    "kernel_ms": sum(kernel_ms(ref_utf8, "utf8_validate").values())})
        out["parity"] = {"ok": u == ref_u == (None, True), "what": "(valid_up_to, is_ascii) equal the one-GPU answer on the share"}
        print(json.dumps(out), flush=True)
        mi.free()
        idx.free()
        del d_share, data
        # multi-byte text: the slow path of K7 on every group
        # whole copies of TEXT only, so that neither the input nor the share ends inside a sequence
        text = np.resize(np.frombuffer(TEXT, dtype=np.uint8), G * GiB - G * GiB % len(TEXT))
        mi = m.index_build_distributed(text)
        share = GiB - GiB % len(TEXT)
        d_share = torch.from_numpy(text[:share]).to(f"cuda:{ctx.device}")
        ref_u = ref_utf8()
        u = mi.validate_utf8()
        out = line(G, devs, ndev, cards, "csvb200_multi_validate_utf8", f"multi-byte UTF-8 text ({NONASCII:.0%} non-ASCII bytes), "
                   "1 GiB per GPU, default cuts", int(text.size), timed(mi.validate_utf8, a.steps),
                   kernel_ms(mi.validate_utf8, "utf8_validate"),
                   {"call": "csvb200_validate_utf8_device", "bytes": share, "wall_s": timed(ref_utf8, a.steps),
                    "kernel_ms": sum(kernel_ms(ref_utf8, "utf8_validate").values())})
        out["parity"] = {"ok": u == ref_u == (None, False), "what": "(valid_up_to, is_ascii) equal the one-GPU answer on the share"}
        print(json.dumps(out), flush=True)
        mi.free()
        m.close()
        del d_share, text
    ctx.close()


if __name__ == "__main__":
    main()
