"""Throughput of batch proof verification with the pairing half by one random linear combination
(bbs_rlc_proof_verify_batch) against the per-item pairing path (bbs_proof_verify_batch), on one GPU.

Workloads: bench.py's proof workloads (bench.make_proof_workload: distinct proofs made on the GPU, every 16th corrupted so
that it fails at the challenge), 262,144 proofs at L = 32 / R = 16 and 524,288 at L = 10 / R = 5.  Both host-buffer calls
are warmed up, then alternated; both must return the same status vector (equal to the workload's expectation) and the rlc
call must report combined == ACCEPT.  The same is repeated on a variant in which one proof per 4,096 fails ONLY at the
pairing (made by bbs_proof_gen_batch from a signature whose e has bit 0 flipped: the prover checks no signature, so its
challenge is consistent): there the combined check fails and the per-item pairing decides, the worst case of the mode.
Prints one JSON line: rates (proofs/s, median over the timed calls), the profiled stage times of one rlc call, and the
GPU's name and power limit."""
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
STAGES = ["h2s", "g1", "prep", "scan_scatter", "bucket", "reduce", "finish", "combined_pairing", "accept_or_fallback"]


def pairing_only_variant(ctx, lib, w, every=4096):
    """copies of the workload's proof buffers in which items every/2, every/2 + every, ... are proofs of signatures with e
    flipped in bit 0; returns (fixed, commit, expect)"""
    L, R = w["L"], w["R"]
    U = L - R
    n = len(w["expect"])
    items = np.arange(every // 2, n, every)
    k = len(items)
    sigs = w["sigs"].reshape(n, bench.SIG_BYTES)[items].copy()
    sigs[:, 48] ^= 1                                   # LE32 e: bit 0
    msgs = np.ascontiguousarray(w["msgs"].reshape(n, L * bench.MSG_BYTES)[items]).reshape(-1)
    offs = np.arange(k * L + 1, dtype=np.uint64) * bench.MSG_BYTES
    rand = np.ascontiguousarray(w["rand"].reshape(n, (5 + U) * 32)[items]).reshape(-1)
    sigs = np.ascontiguousarray(sigs).reshape(-1)
    idx = np.tile(np.arange(0, L, 2, dtype=np.uint32)[:R], k)
    steps = np.arange(k + 1, dtype=np.uint64)
    dis_off, rand_off, commit_off = steps * R, steps * (5 + U), steps * U       # bench.ptr keeps no reference: name them
    fx = np.zeros(k * bench.PROOF_FIXED, dtype=np.uint8)
    cm = np.zeros(k * U * 32, dtype=np.uint8)
    st = np.zeros(k, dtype=np.uint8)
    rc = lib.bbs_proof_gen_batch(ctx.handle, k, ptr(sigs), ptr(msgs), ptr(offs), L, ptr(idx), ptr(dis_off), ptr(rand),
                                 ptr(rand_off), ptr(commit_off), None, 0, ptr(fx), ptr(cm), ptr(st))
    if rc != 0 or not (st == 1).all():
        raise RuntimeError(f"bbs_proof_gen_batch failed: {lib.bbs_last_error().decode()}")
    fixed = w["fixed"].copy().reshape(n, bench.PROOF_FIXED)
    commit = w["commit"].copy().reshape(n, U * 32)
    fixed[items] = fx.reshape(k, bench.PROOF_FIXED)
    commit[items] = cm.reshape(k, U * 32)
    expect = w["expect"].copy()
    expect[items] = 0
    return fixed.reshape(-1), commit.reshape(-1), expect


def run_workload(lib, n, L, R, rounds, warmup, seed):
    ctx = api.BatchContext(api.BLS12_381, bench.IRTF_PK, header=b"", n_messages=L)
    w = bench.make_proof_workload(ctx, lib, n, 77, L, R)
    st_a = np.zeros(n, dtype=np.uint8)
    st_b = np.zeros(n, dtype=np.uint8)
    comb = np.zeros(1, dtype=np.uint8)

    def per_item(fixed, commit):
        rc = lib.bbs_proof_verify_batch(ctx.handle, n, ptr(fixed), ptr(commit), ptr(w["commit_off"]), ptr(w["idx"]),
                                        ptr(w["dmsg"]), ptr(w["moff"]), ptr(w["dis_off"]), None, 0, ptr(st_a))
        assert rc == 0, lib.bbs_last_error().decode()

    def rlc(fixed, commit):
        rc = lib.bbs_rlc_proof_verify_batch(ctx.handle, n, ptr(fixed), ptr(commit), ptr(w["commit_off"]), ptr(w["idx"]),
                                            ptr(w["dmsg"]), ptr(w["moff"]), ptr(w["dis_off"]), None, 0, ptr(seed), ptr(st_b),
                                            ptr(comb))
        assert rc == 0, lib.bbs_last_error().decode()

    def measure(fixed, commit, expect, want_combined):
        for _ in range(warmup):
            per_item(fixed, commit)
            rlc(fixed, commit)
        ta, tb = [], []
        for _ in range(rounds):
            for fn, acc in ((per_item, ta), (rlc, tb)):
                t0 = time.perf_counter()
                fn(fixed, commit)
                acc.append(time.perf_counter() - t0)
                if not np.array_equal(st_a if fn is per_item else st_b, expect):
                    raise RuntimeError(f"{fn.__name__}: status vector differs from the workload's expectation")
            if int(comb[0]) != want_combined:
                raise RuntimeError(f"combined = {int(comb[0])}, expected {want_combined}")
        return n / float(np.median(ta)), n / float(np.median(tb))

    def stages(fixed, commit):
        lib.bbs_ctx_set_profiling(ctx.handle, 1)
        rlc(fixed, commit)
        ms = np.zeros(len(STAGES), dtype=np.float32)
        lib.bbs_ctx_kernel_times(ctx.handle, ms.ctypes.data_as(bench.C.POINTER(bench.C.c_float)), len(STAGES))
        lib.bbs_ctx_set_profiling(ctx.handle, 0)
        return {k: round(float(v), 3) for k, v in zip(STAGES, ms)}

    a, b = measure(w["fixed"], w["commit"], w["expect"], 1)
    out = {"per_item_proofs_per_s": round(a), "rlc_proofs_per_s": round(b), "speedup": round(b / a, 3),
           "rlc_stage_ms": stages(w["fixed"], w["commit"])}
    fixed, commit, expect = pairing_only_variant(ctx, lib, w)
    a2, b2 = measure(fixed, commit, expect, 0)
    out.update({"fallback_per_item_proofs_per_s": round(a2), "fallback_rlc_proofs_per_s": round(b2),
                "fallback_rlc_stage_ms": stages(fixed, commit)})
    ctx.close()
    return out


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
    seed = np.frombuffer(hashlib.sha256(b"tools/bench_rlc_proof.py").digest(), dtype=np.uint8).copy()
    name, power = gpu_identity()
    res = {"gpu": name, "power_limit": power, "rounds": a.rounds}
    for key, n, L, R in (("L32_R16", 262144, 32, 16), ("L10_R5", 524288, 10, 5)):
        m = max(4096, int(n * a.scale))
        res[key] = dict(n=m, **run_workload(lib, m, L, R, a.rounds, a.warmup, seed))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
