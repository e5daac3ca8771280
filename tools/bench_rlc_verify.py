"""Throughput of batch signature verification with per-item statuses by one random linear combination
(bbs_rlc_verify_batch_status) against the per-item call (bbs_verify_batch) and the one-verdict call (bbs_rlc_verify_batch),
on one GPU.

Workloads: bench.py's signature workload (bench.make_workload: distinct 32-byte messages at L = 10, signed on the GPU) at
65,536 and 524,288 items, in three variants: all valid (bench's corrupted items replaced by their valid neighbours); one
item per 4,096 failing only at the pairing (e ^ 1); and bench's own mix, every 16th item corrupted.  The three host-buffer
calls are warmed up, then alternated; the statuses of the rlc call must equal the per-item call's (and the variant's
expectation), `combined` must be ACCEPT for the all-valid variant and REJECT for the others, and so must the one-verdict
call's verdict.  Prints one JSON line: rates (signatures/s, median over the timed calls), the profiled stage times of one
status call per variant, and the GPU's name and power limit."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from bbs_sign_b200 import _native, api  # noqa: E402

ptr = bench.ptr
L = 10
STAGES = ["upload_h2s_first_chunk", "h2s_prep", "scan_scatter", "bucket", "reduce", "finish", "combined_pairing",
          "accept_or_g1", "per_item_pairing"]


def variants(ctx, lib, n):
    """{name: (msgs, offs, sigs, expect, combined expected)}"""
    msgs, offs, sigs, expect = bench.make_workload(ctx, lib, n, L, seed=2024)
    out = {"mix_1_16": (msgs, offs, sigs, expect, 0)}
    bad = np.where(expect == 0)[0]
    m = msgs.copy().reshape(n, L * bench.MSG_BYTES)
    s = sigs.copy().reshape(n, bench.SIG_BYTES)
    m[bad], s[bad] = m[bad - 1], s[bad - 1]                      # bench corrupts items 3 mod 16: neighbours are intact
    valid = (np.ascontiguousarray(m.reshape(-1)), offs, np.ascontiguousarray(s.reshape(-1)), np.ones(n, np.uint8), 1)
    out["all_valid"] = valid
    s1 = s.copy()
    items = np.arange(2048, n, 4096)
    s1[items, 48] ^= 1                                           # LE32 e: bit 0
    e1 = np.ones(n, np.uint8)
    e1[items] = 0
    out["pairing_only_1_4096"] = (valid[0], offs, np.ascontiguousarray(s1.reshape(-1)), e1, 0)
    return out


def run_size(lib, n, rounds, warmup, seed):
    ctx = api.BatchContext(api.BLS12_381, bench.IRTF_PK, header=b"", n_messages=L)
    st_a = np.zeros(n, dtype=np.uint8)
    st_b = np.zeros(n, dtype=np.uint8)
    comb = np.zeros(1, dtype=np.uint8)
    verdict = np.zeros(1, dtype=np.uint8)
    res = {}
    for name, (msgs, offs, sigs, expect, want) in variants(ctx, lib, n).items():
        def per_item():
            rc = lib.bbs_verify_batch(ctx.handle, n, ptr(sigs), ptr(msgs), ptr(offs), L, ptr(st_a))
            assert rc == 0, lib.bbs_last_error().decode()

        def status():
            rc = lib.bbs_rlc_verify_batch_status(ctx.handle, n, ptr(sigs), ptr(msgs), ptr(offs), L, ptr(seed), ptr(st_b),
                                                 ptr(comb))
            assert rc == 0, lib.bbs_last_error().decode()

        def one_verdict():
            rc = lib.bbs_rlc_verify_batch(ctx.handle, n, ptr(sigs), ptr(msgs), ptr(offs), L, ptr(seed), ptr(verdict))
            assert rc == 0, lib.bbs_last_error().decode()

        calls = (per_item, status, one_verdict)
        for _ in range(warmup):
            for fn in calls:
                fn()
        times = {fn.__name__: [] for fn in calls}
        for _ in range(rounds):
            for fn in calls:
                t0 = time.perf_counter()
                fn()
                times[fn.__name__].append(time.perf_counter() - t0)
            if not np.array_equal(st_a, expect) or not np.array_equal(st_b, expect):
                raise RuntimeError(f"{name}: status vectors differ from the workload's expectation")
            if int(comb[0]) != want or int(verdict[0]) != want:
                raise RuntimeError(f"{name}: combined = {int(comb[0])}, verdict = {int(verdict[0])}, expected {want}")
        lib.bbs_ctx_set_profiling(ctx.handle, 1)
        status()
        ms = np.zeros(len(STAGES), dtype=np.float32)
        lib.bbs_ctx_kernel_times(ctx.handle, ms.ctypes.data_as(bench.C.POINTER(bench.C.c_float)), len(STAGES))
        lib.bbs_ctx_set_profiling(ctx.handle, 0)
        rate = {k: round(n / float(np.median(v))) for k, v in times.items()}
        res[name] = {"per_item_sigs_per_s": rate["per_item"], "rlc_status_sigs_per_s": rate["status"],
                     "rlc_verdict_sigs_per_s": rate["one_verdict"],
                     "status_over_per_item": round(rate["status"] / rate["per_item"], 3),
                     "status_over_verdict": round(rate["status"] / rate["one_verdict"], 3),
                     "combined": int(comb[0]), "status_stage_ms": {k: round(float(v), 3) for k, v in zip(STAGES, ms)}}
    ctx.close()
    return res


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return name.strip(), power.strip()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the batch sizes (rehearsal runs)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    lib = _native.load()
    seed = np.frombuffer(hashlib.sha256(b"tools/bench_rlc_verify.py").digest(), dtype=np.uint8).copy()
    name, power = gpu_identity()
    res = {"gpu": name, "power_limit": power, "rounds": a.rounds, "L": L}
    for n in (65536, 524288):
        m = max(8192, int(n * a.scale))
        res[f"n{n}"] = dict(n=m, **run_size(lib, m, a.rounds, a.warmup, seed))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
