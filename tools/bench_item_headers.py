#!/usr/bin/env python3
"""Throughput of the per-item header / presentation header calls (bbs_*_hdr) against the shared-header calls, on one GPU.

Workloads (BLS12-381, scalar messages, host-buffer calls: copies included, every call ends in a device synchronise):
  verify       L = 10, 65,536 items: shared-header context; flagged context (BBS_CTX_PER_ITEM_HEADER) with 65,536 distinct
               64-byte headers; flagged context with one header repeated
  proof verify L = 32, R = 16, 262,144 proofs: shared ph; a 32-byte ph per proof with the context's header; a header and a
               ph per proof
  sign         L = 10, 262,144 items: shared header; a header per item
Every input is seeded and made on the GPU by the _hdr sign / proof-gen calls, so every item verifies; inputs are packed
once and only the library call is timed.  Variants are run alternately, `--rounds` times each after a warm-up; the result
is the median.  Per-kernel times (CUDA events, bbs_ctx_kernel_times) come from one extra profiled call per variant.
Prints one JSON line with the GPU's name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bbs_sign_b200 import _native, api as A  # noqa: E402
from oracle import bbs_oracle as O  # noqa: E402

SUITE, OCS = A.BLS12_381, O.BLS12_381


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"name": name.strip(), "power_limit": power.strip()}


def scalars(rng, count):
    s = rng.integers(0, 256, size=(count, 32), dtype=np.uint8)
    s[:, 31] &= 0x0f                     # below r
    return s


def kernel_times(ctx, call):
    """[msg_to_scalars, G1, pairing, item_domain] for verify / proof verify, [h2s, sign, item_domain] for sign (ms)"""
    lib = ctx.lib
    lib.bbs_ctx_set_profiling(ctx.handle, 1)
    call()
    ms = (C.c_float * 4)()
    lib.bbs_ctx_kernel_times(ctx.handle, ms, 4)
    lib.bbs_ctx_set_profiling(ctx.handle, 0)
    return [round(x, 3) for x in ms]


def run(variants, n, rounds):
    """variants: name -> (ctx, call returning statuses); alternated, median items/s"""
    for name, (ctx, call) in variants.items():
        st = call()
        assert (st == 1).all(), (name, np.bincount(st))
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for name, (ctx, call) in variants.items():
            t = time.perf_counter()
            call()
            times[name].append(time.perf_counter() - t)
    out = {}
    for name, (ctx, call) in variants.items():
        med = statistics.median(times[name])
        out[name] = {"items_per_s": round(n / med), "seconds": [round(t, 4) for t in times[name]],
                     "kernel_ms": kernel_times(ctx, call)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="batch sizes times this (smaller for a quick look)")
    args = ap.parse_args()
    if args.rounds < 3:
        ap.error("--rounds must be at least 3")
    lib = _native.load()
    info = gpu_info()
    rng = np.random.default_rng(2024)
    sk = O.key_gen(OCS, bytes(range(32)), b"", b"BBS-SIG-KEYGEN-SALT-")
    skb, pkb = sk.to_bytes(32, "little"), OCS.g2_compress(O.sk_to_pk(OCS, sk))
    h = b"shared header of the batch"
    result = {"gpu": info, "curve": "BLS12_381", "rounds": args.rounds, "calls": "host-buffer, synchronised"}

    P = A._ptr
    # ---- verify, L = 10 ----
    n, L = int(65536 * args.scale), 10
    shared = A.BatchContext(SUITE, pkb, h, L)
    flag = A.BatchContext(SUITE, pkb, b"", L, per_item_headers=True)
    hdrs = [rng.bytes(64) for _ in range(n)]
    hb, hoff = A._pack_items(hdrs, n, "header")
    sb, soff = A._pack_items([h] * n, n, "header")
    sc = scalars(rng, n * L)
    s_dist = flag.core_sign_batch(skb, sc, n, L, headers=hdrs)[0]
    s_same = flag.core_sign_batch(skb, sc, n, L, headers=[h] * n)[0]      # also the shared-header context's signatures
    st = np.zeros(n, np.uint8)

    def ok(rc):
        assert rc == 0
        return st

    # inputs are packed once: the timed calls are the library's host-buffer entry points only
    result["verify_L10"] = {"n": n, **run({
        "shared_header": (shared, lambda: ok(lib.bbs_core_verify_batch(shared.handle, n, P(s_same), P(sc), L, P(st)))),
        "per_item_distinct": (flag, lambda: ok(lib.bbs_core_verify_batch_hdr(flag.handle, n, P(s_dist), P(sc), L, P(hb), P(hoff), P(st)))),
        "per_item_identical": (flag, lambda: ok(lib.bbs_core_verify_batch_hdr(flag.handle, n, P(s_same), P(sc), L, P(sb), P(soff), P(st)))),
    }, n, args.rounds)}
    shared.close()
    flag.close()

    # ---- sign, L = 10 ----
    n = int(262144 * args.scale)
    shared = A.BatchContext(SUITE, pkb, h, L)
    flag = A.BatchContext(SUITE, pkb, b"", L, per_item_headers=True)
    hdrs = [rng.bytes(64) for _ in range(n)]
    hb, hoff = A._pack_items(hdrs, n, "header")
    sc = scalars(rng, n * L)
    sigs = np.zeros(n * SUITE.signature_bytes, np.uint8)
    st = np.zeros(n, np.uint8)
    skp = P(np.frombuffer(skb, np.uint8))
    result["sign_L10"] = {"n": n, **run({
        "shared_header": (shared, lambda: ok(lib.bbs_core_sign_batch(shared.handle, skp, n, P(sc), L, P(sigs), None, P(st)))),
        "per_item_distinct": (flag, lambda: ok(lib.bbs_core_sign_batch_hdr(flag.handle, skp, n, P(sc), L, P(hb), P(hoff), P(sigs), None,
                                                                           P(st)))),
    }, n, args.rounds)}
    shared.close()
    flag.close()

    # ---- proof verify, L = 32, R = 16 ----
    n, L, R = int(262144 * args.scale), 32, 16
    dis = list(range(0, L, 2))
    U = L - R
    shared = A.BatchContext(SUITE, pkb, h, L)
    flag = A.BatchContext(SUITE, pkb, b"", L, per_item_headers=True)
    hdrs = [rng.bytes(64) for _ in range(n)]
    hb, hoff = A._pack_items(hdrs, n, "header")
    phs = [rng.bytes(32) for _ in range(n)]
    pb, poff = A._pack_items(phs, n, "ph")
    one_ph = np.frombuffer(b"one ph", np.uint8)
    ob, ooff = A._pack_items([b"one ph"] * n, n, "ph")
    sc = scalars(rng, n * L)
    dsc = np.ascontiguousarray(sc.reshape(n, L, 32)[:, dis]).reshape(-1)
    commit_off = np.arange(n + 1, dtype=np.uint64) * U
    dis_off = np.arange(n + 1, dtype=np.uint64) * R
    idx = np.tile(np.array(dis, np.uint32), n)
    rand_off = np.arange(n + 1, dtype=np.uint64) * (5 + U)

    def gen(ctx, gen_hdrs, ph_b, ph_off):
        """proofs from the GPU: _hdr sign, then _hdr proof gen (per-item or the context's header, per-item ph)"""
        ghb, ghoff = A._pack_items(gen_hdrs, n, "header") if gen_hdrs is not None else (None, None)
        sigs = np.zeros(n * SUITE.signature_bytes, np.uint8)
        g = np.zeros(n, np.uint8)
        sign_hb, sign_hoff = (ghb, ghoff) if gen_hdrs is not None else (sb_ctx, sboff_ctx)
        assert lib.bbs_core_sign_batch_hdr(flag.handle, skp, n, P(sc), L, P(sign_hb), P(sign_hoff), P(sigs), None, P(g)) == 0
        assert (g == 1).all()
        rand = scalars(rng, n * (5 + U))
        fixed = np.zeros(n * SUITE.proof_fixed_bytes, np.uint8)
        commit = np.zeros(int(commit_off[-1]) * 32, np.uint8)
        assert lib.bbs_core_proof_gen_batch_hdr(ctx.handle, n, P(sigs), P(sc), L, P(idx), P(dis_off), P(rand), P(rand_off),
                                                P(commit_off), P(ghb), P(ghoff), P(ph_b), P(ph_off), P(fixed), P(commit), P(g)) == 0
        assert (g == 1).all()
        return fixed, commit

    sb_ctx, sboff_ctx = A._pack_items([h] * n, n, "header")     # the shared context's header, for signing on `flag`
    f_sh, c_sh = gen(shared, None, ob, ooff)
    f_ph, c_ph = gen(shared, None, pb, poff)
    f_bo, c_bo = gen(flag, hdrs, pb, poff)
    st = np.zeros(n, np.uint8)
    result["proof_verify_L32_R16"] = {"n": n, **run({
        "shared_ph": (shared, lambda: ok(lib.bbs_core_proof_verify_batch(shared.handle, n, P(f_sh), P(c_sh), P(commit_off), P(idx), P(dsc),
                                                                         P(dis_off), P(one_ph), one_ph.size, P(st)))),
        "per_item_ph": (shared, lambda: ok(lib.bbs_core_proof_verify_batch_hdr(shared.handle, n, P(f_ph), P(c_ph), P(commit_off), P(idx),
                                                                               P(dsc), P(dis_off), None, None, P(pb), P(poff), P(st)))),
        "per_item_header_and_ph": (flag, lambda: ok(lib.bbs_core_proof_verify_batch_hdr(flag.handle, n, P(f_bo), P(c_bo), P(commit_off),
                                                                                        P(idx), P(dsc), P(dis_off), P(hb), P(hoff),
                                                                                        P(pb), P(poff), P(st)))),
    }, n, args.rounds)}
    shared.close()
    flag.close()
    for k in ("verify_L10", "sign_L10", "proof_verify_L32_R16"):
        r = result[k]
        base = r["shared_header"] if "shared_header" in r else r["shared_ph"]
        r["relative"] = {v: round(r[v]["items_per_s"] / base["items_per_s"], 4) for v in r if isinstance(r[v], dict) and "items_per_s" in r[v]}
    print(json.dumps(result))


if __name__ == "__main__":
    main()
