#!/usr/bin/env python3
"""bench.py -- BLS12-381 BBS batch verify / proof-verify throughput on B200 (BASELINE.json metric).

Headline (the JSON line's `value`): BASELINE configs[1] -- one pass of the hot path (msg_to_scalars -> core_verify G1
half -> two-pair pairing) over a batch of 65,536 synthetic signatures x L=10 messages of 32 bytes under one issuer
key, 1/16 of them corrupted; weak scaling (65,536 per GPU).  Signatures are produced by the library's own
`bbs_sign_batch` on the GPU (no oracle on the product path); the status vector of every run is checked against the
construction (valid -> 1, corrupted -> 0).

`extra` (same line): the rest of the metric, STRONG-scaled (the total is fixed, every GPU takes total / N):
  proof_l10  the metric's proof-verify leg at the headline's L: 524,288 proofs, L = 10, 5 disclosed (proof-verifies/s)
  proof  BASELINE configs[3]: 262,144 selective-disclosure proofs, L = 32, 16 disclosed   (proof-verifies/s)
  bn254  BASELINE configs[2]: 1,048,576 BN254 core_verify over 31 pre-hashed scalars       (verifies/s)
  sign   BASELINE configs[4], first leg: 4,194,304 signatures                              (signatures/s)
  rlc    BASELINE configs[4], second leg: ONE random-linear-combination verdict over 4,194,304 signatures

  python bench.py --gpus N --steps K --warmup W           our arm (torchrun for N > 1, one rank per GPU)
  python bench.py --workload proof|proof_l10|bn254|sign|rlc ...     one workload as the line itself (ad-hoc runs, profiling)
  python bench.py --impl reference ...                    CPU arm: the oracle port of the reference's path
  python bench.py ... --dump-outputs DIR                  also write what the timed steps returned (rank 0) as DIR/<name>.npy

Prints ONE JSON line (rank 0)."""
import argparse
import csv
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "bls12_381_bbs_verifies_per_sec_L10"
UNIT = "verifies/s"
N_DEFAULT = 65536
L_DEFAULT = 10
# IRTF draft key pair (test_vector.rs:140-160): sk little-endian, pk compressed
IRTF_SK = 0x60e55110f76883a13d030b2f6bd11883422d5abde717569fc0731f51237169fc
IRTF_PK = bytes.fromhex("a820f230f6ae38503b86c70dc50b61c58a77e45c39ab25c0652bbaa8fa136f2851bd4781c9dcde39fc9d1d52c9e60268"
                        "061e7d7632171d91aa8d460acee0e96f1e7c4cfb12d3ff9ab5d5dc91c277db75c845d649ef3c4f63aebc364cd55ded0c")
# counting model of SURVEY 8(d) / Appendix D: 32x32->64 products per item (BLS12-381 Fp: M = 300, S = 234; 8 limbs: 136, 108)
PRODUCTS_PER_VERIFY = 19509 * 300 + 3285 * 234              # 6.62e6   BLS12-381 verify, L = 10
PRODUCTS_PAIRING = (8116 + 7777) * 300 + (76 * 300 + 380 * 234)  # Miller + final exp + its one inversion
PRODUCTS_G1 = PRODUCTS_PER_VERIFY - PRODUCTS_PAIRING
PRODUCTS_PROOF = 27423 * 300 + 8521 * 234                   # 1.022e7  BLS12-381 proof_verify, L = 32, R = 16
PRODUCTS_BN254 = 26874 * 136 + 5846 * 108                   # 4.29e6   BN254 core_verify, L = 31
PRODUCTS_SIGN = 3616 * 300 + 3285 * 234                     # 1.85e6   BLS12-381 sign, L = 10
PRODUCTS_RLC = 74000                                        # 7.4e4    per signature of an RLC batch (+ 70 SHA-256 blocks)
TOTALS = {"proof": 262144, "proof_l10": 524288, "bn254": 1 << 20, "sign": 1 << 22, "rlc": 1 << 22}   # BASELINE configs[3], metric's
                                                                                   # proof leg at L = 10, configs[2], [4], [4]
SIG_BYTES = 80
MSG_BYTES = 32
PROOF_FIXED = 3 * 48 + 128
DUMP_VALUES = 1 << 20     # values kept per --dump-outputs array (4 MB of float32; 7 arrays at most in one run)


def ptr(a):
    return C.c_void_p(a.ctypes.data) if isinstance(a, np.ndarray) else C.c_void_p(a.data_ptr())


def verify_config(n, L):
    """`config` of the headline line; the CPU arm prints the same dict (it times bounded samples of this workload)."""
    return {"workload": f"BLS12-381-SHA-256 batch verify: {n} signatures x L={L} messages of 32 B, one issuer key, "
                        "1/16 corrupted (BASELINE configs[1])", "n_per_gpu": n, "L": L,
            "l2": "256 MB flush write between timed iterations", "sharding": "by signature index, no collective"}


def make_workload(ctx, lib, n, L, seed):
    """Synthetic batch: random 32-byte messages, signed on the GPU, 1/16 corrupted."""
    rng = np.random.default_rng(seed)
    msgs = rng.integers(0, 256, size=n * L * MSG_BYTES, dtype=np.uint8)
    offs = (np.arange(n * L + 1, dtype=np.uint64) * MSG_BYTES)
    sigs = np.zeros(n * SIG_BYTES, dtype=np.uint8)
    st = np.zeros(n, dtype=np.uint8)
    sk = np.frombuffer(IRTF_SK.to_bytes(32, "little"), dtype=np.uint8).copy()
    rc = lib.bbs_sign_batch(ctx.handle, ptr(sk), n, ptr(msgs), ptr(offs), L, ptr(sigs), None, ptr(st))
    if rc != 0 or not (st == 1).all():
        raise RuntimeError(f"bbs_sign_batch failed rc={rc}: {lib.bbs_last_error().decode()}")
    sigs = sigs.reshape(n, SIG_BYTES)
    expect = np.ones(n, dtype=np.uint8)
    bad = np.arange(3, n, 16)
    for k, i in enumerate(bad):
        kind = k % 4
        if kind == 0:      # flipped message byte
            msgs[(i * L + (k % L)) * MSG_BYTES + 7] ^= 0x40
        elif kind == 1:    # e ^ 1
            sigs[i, 48] ^= 1
        elif kind == 2:    # A = identity
            sigs[i, :48] = 0
            sigs[i, 0] = 0xC0
        else:              # A of the neighbouring signature
            sigs[i, :48] = sigs[i - 1, :48]
        expect[i] = 0
    return msgs, offs, np.ascontiguousarray(sigs.reshape(-1)), expect


PROOF_CORRUPTIONS = ("disclosed message byte", "e^ ^ 1", "Abar = identity", "challenge ^ 1", "commitments 0 <-> 1",
                     "Bbar of the neighbouring proof", "r3^ ^ 1")


def make_proof_workload(ctx, lib, n, seed, L=32, R=16):
    """n DISTINCT selective-disclosure proofs made on the GPU: bbs_sign_batch, then bbs_proof_gen_batch (byte-pinned to the
    oracle's proof_gen by tests/parity_cases.py case_proof_gen and the IRTF proof fixture) with the even indexes
    disclosed; every 16th proof is corrupted, cycling through the seven rejection classes of SURVEY 8d."""
    U = L - R
    rng = np.random.default_rng(seed)
    msgs = rng.integers(0, 256, size=n * L * MSG_BYTES, dtype=np.uint8)
    offs = (np.arange(n * L + 1, dtype=np.uint64) * MSG_BYTES)
    sigs = np.zeros(n * SIG_BYTES, dtype=np.uint8)
    st = np.zeros(n, dtype=np.uint8)
    sk = np.frombuffer(IRTF_SK.to_bytes(32, "little"), dtype=np.uint8).copy()
    if lib.bbs_sign_batch(ctx.handle, ptr(sk), n, ptr(msgs), ptr(offs), L, ptr(sigs), None, ptr(st)) != 0 or not (st == 1).all():
        raise RuntimeError(f"bbs_sign_batch failed: {lib.bbs_last_error().decode()}")
    dis = np.arange(0, L, 2, dtype=np.uint32)[:R]
    idx = np.tile(dis, n)
    dis_off = np.arange(n + 1, dtype=np.uint64) * R
    rand = rng.integers(0, 256, size=(n * (5 + U), 32), dtype=np.uint8)
    rand[:, 31] &= 0x3f                                  # < 2^254 < r: canonical scalars
    rand = np.ascontiguousarray(rand.reshape(-1))
    rand_off = np.arange(n + 1, dtype=np.uint64) * (5 + U)
    commit_off = np.arange(n + 1, dtype=np.uint64) * U
    fixed = np.zeros(n * PROOF_FIXED, dtype=np.uint8)
    commit = np.zeros(n * U * 32, dtype=np.uint8)
    st[:] = 0
    rc = lib.bbs_proof_gen_batch(ctx.handle, n, ptr(sigs), ptr(msgs), ptr(offs), L, ptr(idx), ptr(dis_off), ptr(rand),
                                 ptr(rand_off), ptr(commit_off), None, 0, ptr(fixed), ptr(commit), ptr(st))
    if rc != 0 or not (st == 1).all():
        raise RuntimeError(f"bbs_proof_gen_batch failed rc={rc}: {lib.bbs_last_error().decode()}")
    dmsg = np.ascontiguousarray(msgs.reshape(n, L, MSG_BYTES)[:, dis, :]).reshape(-1)
    moff = np.arange(n * R + 1, dtype=np.uint64) * MSG_BYTES
    fx = fixed.reshape(n, PROOF_FIXED)
    cm = commit.reshape(n, U * 32)
    dm = dmsg.reshape(n, R * MSG_BYTES)
    expect = np.ones(n, dtype=np.uint8)
    for k, i in enumerate(range(5, n, 16)):
        kind = k % 7
        if kind == 0:
            dm[i, (k % R) * MSG_BYTES + 3] ^= 0x10
        elif kind == 1:
            fx[i, 144] ^= 1
        elif kind == 2:
            fx[i, :48] = 0
            fx[i, 0] = 0xC0
        elif kind == 3:
            fx[i, 240] ^= 1
        elif kind == 4:
            t = cm[i, :32].copy()
            cm[i, :32] = cm[i, 32:64]
            cm[i, 32:64] = t
        elif kind == 5:
            fx[i, 48:96] = fx[i - 1, 48:96]
        else:
            fx[i, 208] ^= 1
        expect[i] = 0
    return {"fixed": fixed, "commit": commit, "commit_off": commit_off, "idx": idx, "dmsg": dmsg, "moff": moff,
            "dis_off": dis_off, "expect": expect, "sigs": sigs, "msgs": msgs, "rand": rand, "L": L, "R": R}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.dev, self.rows, self.proc = dev, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.dev)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 8 and r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        # under load = upper half of the samples
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class Env:
    """One process per GPU: torch only for device buffers, the launching stream, events and the NCCL plumbing."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from bbs_sign_b200 import api, _native
        self.torch, self.dist, self.api = torch, dist, api
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.lib = _native.load()
        self.stream = torch.cuda.current_stream()
        self.sp = C.c_void_p(self.stream.cuda_stream)
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)   # > 126 MB L2
        self.n_sm = torch.cuda.get_device_properties(self.local).multi_processor_count
        self.sm_max_mhz = 1965
        self._flush_k = 0
        self.outputs = {}

    def keep(self, name, a, width=1):
        """Records what the last timed step returned (rows of `width` values) for --dump-outputs, as float32.  An output
        of more than DUMP_VALUES values keeps a fixed, seeded sample of its rows (the same rows for the same size)."""
        a = np.asarray(a).reshape(-1, width)
        if a.size > DUMP_VALUES:
            a = a[np.sort(np.random.default_rng(0).choice(len(a), DUMP_VALUES // width, replace=False))]
        self.outputs[name] = a.astype(np.float32).squeeze(1) if width == 1 else a.astype(np.float32)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, seconds):
        t = self.torch.tensor([seconds], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def to_dev(self, a):
        return self.torch.from_numpy(_signed_view(a)).to(self.dev)

    def pin(self, a):
        return self.torch.from_numpy(_signed_view(a)).pin_memory()

    def peak_products(self):
        # IMAD.WIDE.U32 (one 32x32->64 product) issues at 8 lanes/clk/SMSP = 32 products/clk/SM on sm_100 (half the rate of
        # a 32-bit IMAD; ncu: 4 fmaheavy-pipe cycles per warp instruction; the in-run probe reaches ~92 % of this figure).
        # MEASURED_PEAKS.json has no integer entry, so the denominator is this nominal rate at the maximum SM clock.
        return self.n_sm * 32 * self.sm_max_mhz * 1e6

    def time_device(self, step, steps):
        """K steps on the launching stream, CUDA events around each, a 256 MB L2 flush write before each (outside the
        events); barrier + synchronize on both sides; seconds, max over ranks."""
        torch = self.torch
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.barrier()
        for k in range(steps):
            self._flush_k += 1
            self.flush.fill_(self._flush_k & 0xff)
            ev[k][0].record(self.stream)
            step()
            ev[k][1].record(self.stream)
            ev[k][1].synchronize()
        self.barrier()
        return self.max_over_ranks(sum(a.elapsed_time(b) for a, b in ev) * 1e-3)

    def time_host(self, step, steps):
        """K host-buffer calls (each copies in, computes, copies out and synchronises); wall clock between barriers, max
        over ranks."""
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        self.barrier()
        return self.max_over_ranks(time.perf_counter() - t0)

    def kernel_times(self, ctx, k):
        kt = (C.c_float * k)()
        self.lib.bbs_ctx_kernel_times(ctx.handle, kt, k)
        return [float(x) for x in kt]

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def _signed_view(a):
    if a.dtype == np.uint64:
        return a.view(np.int64)
    if a.dtype == np.uint32:
        return a.view(np.int32)
    return a


def _check(lib, rc):
    if rc != 0:
        raise RuntimeError(lib.bbs_last_error().decode())


def kernel_metrics(kernel):
    """DRAM traffic and multiplier-pipe utilisation of a kernel from the committed ncu summary profiles/kernel_metrics.csv
    (one row per kernel: the latest `ncu --set full` capture of the bench command); None when there is no capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "kernel_metrics.csv")) as f:
            rows = [r for r in csv.DictReader(l for l in f if not l.startswith("#")) if r["kernel"] == kernel]
    except OSError:
        return None
    return rows[-1] if rows else None


def imad_roofline(env, kernel, n_items, products_per_item, kernel_ms, traffic_key=None):
    peak = env.peak_products()
    achieved = n_items * products_per_item / (kernel_ms * 1e-3) if kernel_ms > 0 else 0.0
    out = {"kernel": kernel, "bound": "imad", "achieved": achieved / 1e12, "peak": peak / 1e12,
           "unit": "T(32x32->64 products)/s", "frac": achieved / peak, "algorithmic_products_per_item": int(products_per_item)}
    m = kernel_metrics(traffic_key) if traffic_key else None
    if m:
        scale = n_items / float(m["n"])
        out["traffic"] = int((float(m["dram_read_bytes"]) + float(m["dram_write_bytes"])) * scale)
        out["pipe_fmaheavy_pct"] = float(m["pipe_fmaheavy_pct"])
        out["traffic_source"] = f"profiles/kernel_metrics.csv ({m['source']}; ncu --set full at n = {m['n']}, scaled to n = {n_items})"
    else:
        out["traffic"] = None
    return out


# ---------------------------------------------------------------------------------------------------------------------
def bench_verify(env, args):
    """The headline: BASELINE configs[1], weak scaling."""
    torch, lib, api = env.torch, env.lib, env.api
    n, L = args.n, args.L
    ctx = api.BatchContext(api.BLS12_381, IRTF_PK, header=b"", n_messages=L, device=env.local)
    msgs, offs, sigs, expect = make_workload(ctx, lib, n, L, seed=1234 + env.rank)
    d_msgs, d_offs, d_sigs = env.to_dev(msgs), env.to_dev(offs), env.to_dev(sigs)
    d_status = torch.zeros(n, dtype=torch.uint8, device=env.dev)
    lib.bbs_ctx_set_profiling(ctx.handle, 1)
    ktimes = []

    def step():
        _check(lib, lib.bbs_verify_batch_dev(ctx.handle, n, ptr(d_sigs), ptr(d_msgs), ptr(d_offs), L, ptr(d_status), env.sp))

    def step_timed():
        step()
        torch.cuda.synchronize()
        ktimes.append(env.kernel_times(ctx, 3))

    for _ in range(args.warmup):
        step()
    env.barrier()
    got = d_status.cpu().numpy()
    if not np.array_equal(got, expect):
        raise RuntimeError(f"status vector mismatch: {int((got != expect).sum())} of {n} items")
    launches0 = ctx.launch_count()
    sampler = ClockSampler(env.local)
    sampler.start()
    try:
        t_max = env.time_device(step_timed, args.steps)
    finally:
        clocks = sampler.stop()       # never leave nvidia-smi running
    env.sm_max_mhz = clocks.get("sm_max_mhz") or env.sm_max_mhz
    launches = (ctx.launch_count() - launches0) // max(args.steps, 1)
    got = d_status.cpu().numpy()
    if not np.array_equal(got, expect):
        raise RuntimeError("status vector mismatch after the timed region")
    env.keep("verify_status", got)
    value = env.world * n * args.steps / t_max

    # ---- end-to-end arm: host (pinned) buffers through the reference-facing call, copies included ----
    lib.bbs_ctx_set_profiling(ctx.handle, 0)
    p_msgs, p_offs, p_sigs = env.pin(msgs), env.pin(offs), env.pin(sigs)
    p_status = torch.zeros(n, dtype=torch.uint8).pin_memory()

    def e2e_step():
        _check(lib, lib.bbs_verify_batch(ctx.handle, n, ptr(p_sigs), ptr(p_msgs), ptr(p_offs), L, ptr(p_status)))

    e2e_step()
    te = env.time_host(e2e_step, args.steps)
    if not np.array_equal(p_status.numpy(), expect):
        raise RuntimeError("e2e status vector mismatch")
    e2e_value = env.world * n * args.steps / te

    out = None
    if env.rank == 0:
        gprod, pk_ms = C.c_double(), C.c_float()
        peak_modes = {}
        for mode, name in ((0, "mad.lo+mad.hi"), (1, "mad.wide (IMAD.WIDE)")):
            lib.bbs_imad_peak(env.local, 2000, mode, C.byref(gprod), C.byref(pk_ms))
            peak_modes[name] = gprod.value * 1e9
        kmean = np.array(ktimes).mean(axis=0)
        pairing_s = float(kmean[2]) * 1e-3
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        alg_bytes = n * (6 * 12 * 4 + 4 + 1)        # pair record + flags in, status out
        peak = env.peak_products()
        roof = imad_roofline(env, "pairing_coop_kernel<Bls> (2-pair Miller loop + final exponentiation, 6 role-warps per 32 items)",
                             n, PRODUCTS_PAIRING, float(kmean[2]), traffic_key="pairing_coop_kernel<Bls>")
        roof.update({
            "peak_source": f"nominal IMAD.WIDE rate: {env.n_sm} SM x 32 products/clk x {env.sm_max_mhz} MHz (no integer entry in "
                           "MEASURED_PEAKS.json); in-run probe below",
            "peak_by_form_tprod_s": {k: v / 1e12 for k, v in peak_modes.items()},
            "whole_step_frac": value / env.world * PRODUCTS_PER_VERIFY / peak,
            "algorithmic_bytes_per_launch": int(alg_bytes),
            "hbm": {"achieved_gbs": alg_bytes / pairing_s / 1e9, "peak_gbs": hbm_peak,
                    "frac": alg_bytes / pairing_s / 1e9 / hbm_peak, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}})
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": env.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_max / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic", "checked": True,
            "config": verify_config(n, L),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(msgs.nbytes + offs.nbytes + sigs.nbytes),
                    "d2h_bytes_per_step": int(n)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "kernels_ms": {"msg_to_scalars": float(kmean[0]), "verify_g1": float(kmean[1]), "pairing": float(kmean[2])},
            "roofline": roof,
            "roofline_g1": imad_roofline(env, "verify_g1_split_kernel<Bls> + verify_g1_combine_kernel<Bls> (decompress + subgroup test of A and e*A | fixed-base MSM over the GLV tables, as two tasks per item; join: e*A - B to affine)",
                                         n, PRODUCTS_G1, float(kmean[1]), traffic_key="verify_g1_split_kernel<Bls>"),
        }
    ctx.close()
    return out


def bench_proof(env, n, steps, warmup, seed=77, L=32, R=16):
    """BASELINE configs[3] shape: BLS12-381 batch proof_verify, L = 32 with 16 disclosed messages, n DISTINCT proofs per GPU
    (make_proof_workload).  A step = msg_to_scalars of the disclosed messages + core_proof_verify (G1 half with the
    challenge hash, then the cooperative pairing kernel).  With L = 10, R = 5 it is the proof-verify leg of BASELINE.json's
    headline metric ("verifies/sec & proof-verifies/sec, L=10")."""
    torch, lib, api = env.torch, env.lib, env.api
    ctx = api.BatchContext(api.BLS12_381, IRTF_PK, header=b"", n_messages=L, device=env.local)
    w = make_proof_workload(ctx, lib, n, seed + env.rank, L, R)
    expect = w["expect"]
    keys = ("fixed", "commit", "commit_off", "idx", "dmsg", "moff", "dis_off")
    d = {k: env.to_dev(w[k]) for k in keys}
    d_scal = torch.zeros(n * R * 32, dtype=torch.uint8, device=env.dev)
    d_status = torch.zeros(n, dtype=torch.uint8, device=env.dev)
    lib.bbs_ctx_set_profiling(ctx.handle, 1)
    h2s_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))

    def step():
        h2s_ev[0].record(env.stream)
        _check(lib, lib.bbs_msg_to_scalars_dev(ctx.handle, n * R, ptr(d["dmsg"]), ptr(d["moff"]), ptr(d_scal), env.sp))
        h2s_ev[1].record(env.stream)
        _check(lib, lib.bbs_core_proof_verify_batch_dev(ctx.handle, n, ptr(d["fixed"]), ptr(d["commit"]), ptr(d["commit_off"]),
                                                        ptr(d["idx"]), ptr(d_scal), ptr(d["dis_off"]), None, 0, ptr(d_status), env.sp))

    for _ in range(warmup):
        step()
    env.barrier()
    got = d_status.cpu().numpy()
    if not np.array_equal(got, expect):
        raise RuntimeError(f"proof status vector mismatch: {int((got != expect).sum())} of {n}")
    launches0 = ctx.launch_count()
    t = env.time_device(step, steps)
    launches = (ctx.launch_count() - launches0) // max(steps, 1)
    env.keep(f"proof_L{L}_R{R}_status", d_status.cpu().numpy())
    kt = env.kernel_times(ctx, 3)
    kt[0] = h2s_ev[0].elapsed_time(h2s_ev[1])
    lib.bbs_ctx_set_profiling(ctx.handle, 0)
    value = env.world * n * steps / t
    p = {k: env.pin(w[k]) for k in keys}
    p_status = torch.zeros(n, dtype=torch.uint8).pin_memory()

    def e2e_step():
        _check(lib, lib.bbs_proof_verify_batch(ctx.handle, n, ptr(p["fixed"]), ptr(p["commit"]), ptr(p["commit_off"]), ptr(p["idx"]),
                                               ptr(p["dmsg"]), ptr(p["moff"]), ptr(p["dis_off"]), None, 0, ptr(p_status)))

    e2e_step()
    te = env.time_host(e2e_step, steps)
    if not np.array_equal(p_status.numpy(), expect):
        raise RuntimeError("e2e proof status vector mismatch")
    ctx.close()
    if env.rank != 0:
        return None
    step_ms = t / steps * 1e3
    config3 = (L, R) == (32, 16)
    # the counting model of SURVEY Appendix D covers configs[3]; other shapes report the pairing kernel against its own count
    products, g1_products = (PRODUCTS_PROOF, PRODUCTS_PROOF - PRODUCTS_PAIRING) if config3 else (None, None)
    return {"metric": f"bls12_381_bbs_proof_verifies_per_sec_L{L}_R{R}", "value": value, "unit": "proof-verifies/s",
            "n_gpus": env.world, "n_total": env.world * n, "n_per_gpu": n, "steps": steps, "warmup": warmup, "ms_per_step": step_ms,
            "checked": True,
            "config": {"workload": f"BLS12-381 batch proof_verify: {env.world * n} distinct proofs ({n} per GPU), L={L}, {R} disclosed "
                                   "32-B messages, one issuer key, made by bbs_sign_batch + bbs_proof_gen_batch, 1/16 corrupted over 7 "
                                   "rejection classes (" + ("BASELINE configs[3]" if config3 else "the proof-verify leg of BASELINE.json's "
                                   "metric at the headline's L") + ")",
                       "l2": "256 MB flush write between timed iterations", "sharding": "by proof index, no collective"},
            "e2e": {"value": env.world * n * steps / te, "unit": "proof-verifies/s",
                    "h2d_bytes_per_step": sum(int(w[k].nbytes) for k in keys), "d2h_bytes_per_step": int(n)},
            "gpu_launches": int(launches),
            "kernels_ms": {"msg_to_scalars": kt[0], "proof_g1": kt[1], "pairing": kt[2]},
            "roofline": dict(imad_roofline(env, "whole step: h2s_item + proof_g1_split_kernel<Bls> + proof_g1_join_kernel<Bls> + pairing_coop_kernel<Bls>", n, products,
                                           step_ms, traffic_key="proof_g1_split_kernel<Bls>") if config3 else
                             imad_roofline(env, "pairing_coop_kernel<Bls> (the dominant kernel of the step)", n, PRODUCTS_PAIRING, kt[2],
                                           traffic_key="pairing_coop_kernel<Bls>"),
                             g1_kernel_frac=n * g1_products / (kt[1] * 1e-3) / env.peak_products() if config3 and kt[1] > 0 else None,
                             pairing_kernel_frac=n * PRODUCTS_PAIRING / (kt[2] * 1e-3) / env.peak_products() if kt[2] > 0 else None)}


def bench_proof_l10(env, n, steps, warmup, seed=91):
    return bench_proof(env, n, steps, warmup, seed=seed, L=10, R=5)


def make_bn254_workload(ctx, lib, n, seed, L=31):
    key = np.load(os.path.join(ROOT, "tests", "golden", "bn254_bench_key.npz"))
    rng = np.random.default_rng(seed)
    sc = rng.integers(0, 256, size=(n * L, 32), dtype=np.uint8)
    sc[:, 31] &= 0x0f                                   # < 2^252 < r: canonical scalars
    sc = np.ascontiguousarray(sc.reshape(-1))
    sigs = np.zeros(n * 64, dtype=np.uint8)
    st = np.zeros(n, dtype=np.uint8)
    _check(lib, lib.bbs_core_sign_batch(ctx.handle, ptr(np.ascontiguousarray(key["sk"])), n, ptr(sc), L, ptr(sigs), None, ptr(st)))
    if not (st == 1).all():
        raise RuntimeError("bn254 sign status vector is not all ACCEPT")
    expect = np.ones(n, dtype=np.uint8)
    sg = sigs.reshape(n, 64)
    for k, i in enumerate(range(5, n, 16)):
        kind = k % 4
        if kind == 0:                                   # one message scalar changed
            sc[(i * L + (k % L)) * 32 + 2] ^= 0x04
        elif kind == 1:                                 # e ^ 1
            sg[i, 32] ^= 1
        elif kind == 2:                                 # A = identity (ark SW flags: infinity bit in the last byte)
            sg[i, :32] = 0
            sg[i, 31] = 0x40
        else:                                           # A of the neighbouring signature
            sg[i, :32] = sg[i - 1, :32]
        expect[i] = 0
    return sc, sigs, expect, key


def bench_bn254(env, n, steps, warmup, seed=5):
    """BASELINE configs[2] shape: BN254 core_verify over pre-hashed scalar messages (L = 31).  Key pair:
    tests/golden/bn254_bench_key.npz (made once with the oracle's key_gen / sk_to_pk); signatures are made on the GPU by
    bbs_core_sign_batch; 1/16 corrupted over the four signature rejection classes."""
    torch, lib, api = env.torch, env.lib, env.api
    L = 31
    key = np.load(os.path.join(ROOT, "tests", "golden", "bn254_bench_key.npz"))
    ctx = api.BatchContext(api.BN254, bytes(key["pk"]), header=b"", n_messages=L, device=env.local)
    sc, sigs, expect, _ = make_bn254_workload(ctx, lib, n, seed + env.rank, L)
    d_sigs, d_sc = env.to_dev(sigs), env.to_dev(sc)
    d_status = torch.zeros(n, dtype=torch.uint8, device=env.dev)

    def step():
        _check(lib, lib.bbs_core_verify_batch_dev(ctx.handle, n, ptr(d_sigs), ptr(d_sc), L, ptr(d_status), env.sp))

    lib.bbs_ctx_set_profiling(ctx.handle, 1)
    for _ in range(warmup):
        step()
    env.barrier()
    got = d_status.cpu().numpy()
    if not np.array_equal(got, expect):
        raise RuntimeError(f"bn254 status vector mismatch: {int((got != expect).sum())} of {n}")
    launches0 = ctx.launch_count()
    t = env.time_device(step, steps)
    launches = (ctx.launch_count() - launches0) // max(steps, 1)
    env.keep("bn254_status", d_status.cpu().numpy())
    kt = env.kernel_times(ctx, 3)
    lib.bbs_ctx_set_profiling(ctx.handle, 0)
    p_sigs, p_sc = env.pin(sigs), env.pin(sc)
    p_status = torch.zeros(n, dtype=torch.uint8).pin_memory()

    def e2e_step():
        _check(lib, lib.bbs_core_verify_batch(ctx.handle, n, ptr(p_sigs), ptr(p_sc), L, ptr(p_status)))

    e2e_step()
    te = env.time_host(e2e_step, steps)
    if not np.array_equal(p_status.numpy(), expect):
        raise RuntimeError("e2e bn254 status vector mismatch")
    ctx.close()
    if env.rank != 0:
        return None
    step_ms = t / steps * 1e3
    return {"metric": "bn254_bbs_core_verifies_per_sec_L31", "value": env.world * n * steps / t, "unit": "verifies/s",
            "n_gpus": env.world, "n_total": env.world * n, "n_per_gpu": n, "steps": steps, "warmup": warmup, "ms_per_step": step_ms,
            "checked": True,
            "config": {"workload": f"BN254 core_verify: {env.world * n} signatures ({n} per GPU) x L=31 pre-hashed scalar messages, one "
                                   "issuer key, 1/16 corrupted over 4 rejection classes (BASELINE configs[2])",
                       "l2": "256 MB flush write between timed iterations", "sharding": "by signature index, no collective"},
            "e2e": {"value": env.world * n * steps / te, "unit": "verifies/s",
                    "h2d_bytes_per_step": int(sigs.nbytes + sc.nbytes), "d2h_bytes_per_step": int(n)},
            "gpu_launches": int(launches),
            "kernels_ms": {"verify_g1": kt[1], "pairing": kt[2]},
            "roofline": dict(imad_roofline(env, "whole step: verify_g1_split_kernel<Bn> + verify_g1_combine_kernel<Bn> + pairing_coop_kernel<Bn>", n, PRODUCTS_BN254, step_ms,
                                           traffic_key="pairing_coop_kernel<Bn>"),
                             pairing_kernel_frac=n * 2530000 / (kt[2] * 1e-3) / env.peak_products() if kt[2] > 0 else None)}


def bench_sign(env, n, steps, warmup, L=10, seed=7):
    """BASELINE configs[4], first leg: batch signing (core_sign: B, e = H2S(sk || msgs || domain), A = B * 1/(sk + e)) of n
    message sets x L = 10.  `value`: device-resident messages (msg_to_scalars + sign_kernel); `e2e`: bbs_sign_batch with
    pinned host buffers.  The produced batch must pass the random-linear-combination verdict."""
    torch, lib, api = env.torch, env.lib, env.api
    ctx = api.BatchContext(api.BLS12_381, IRTF_PK, header=b"", n_messages=L, device=env.local)
    rng = np.random.default_rng(seed + env.rank)
    p_msgs = env.pin(rng.integers(0, 256, size=n * L * MSG_BYTES, dtype=np.uint8))
    p_offs = env.pin(np.arange(n * L + 1, dtype=np.uint64) * MSG_BYTES)
    p_sigs = env.pin(np.zeros(n * SIG_BYTES, dtype=np.uint8))
    p_st = env.pin(np.zeros(n, dtype=np.uint8))
    sk = np.frombuffer(IRTF_SK.to_bytes(32, "little"), dtype=np.uint8).copy()
    d_msgs, d_offs = p_msgs.to(env.dev), p_offs.to(env.dev)
    d_scal = torch.zeros(n * L * 32, dtype=torch.uint8, device=env.dev)
    d_sigs = torch.zeros(n * SIG_BYTES, dtype=torch.uint8, device=env.dev)
    d_st = torch.zeros(n, dtype=torch.uint8, device=env.dev)
    h2s_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))

    def step():
        h2s_ev[0].record(env.stream)
        _check(lib, lib.bbs_msg_to_scalars_dev(ctx.handle, n * L, ptr(d_msgs), ptr(d_offs), ptr(d_scal), env.sp))
        h2s_ev[1].record(env.stream)
        _check(lib, lib.bbs_core_sign_batch_dev(ctx.handle, ptr(sk), n, ptr(d_scal), L, ptr(d_sigs), None, ptr(d_st), env.sp))

    def e2e_step():
        _check(lib, lib.bbs_sign_batch(ctx.handle, ptr(sk), n, ptr(p_msgs), ptr(p_offs), L, ptr(p_sigs), None, ptr(p_st)))

    lib.bbs_ctx_set_profiling(ctx.handle, 1)
    for _ in range(warmup):
        step()
    env.barrier()
    launches0 = ctx.launch_count()
    t = env.time_device(step, steps)
    launches = (ctx.launch_count() - launches0) // max(steps, 1)
    sigs, st = d_sigs.cpu().numpy(), d_st.cpu().numpy()
    env.keep("sign_signatures", sigs, SIG_BYTES)
    env.keep("sign_status", st)
    kt = env.kernel_times(ctx, 2)
    kt[0] = h2s_ev[0].elapsed_time(h2s_ev[1])
    lib.bbs_ctx_set_profiling(ctx.handle, 0)
    e2e_step()
    te = env.time_host(e2e_step, steps)
    if not (p_st.numpy() == 1).all() or not (st == 1).all():
        raise RuntimeError("sign status vector is not all ACCEPT")
    if not np.array_equal(sigs, p_sigs.numpy()):
        raise RuntimeError("device-resident and host-buffer signing disagree")
    seed32 = np.frombuffer(os.urandom(32), dtype=np.uint8).copy()
    verdict = np.zeros(1, dtype=np.uint8)
    rc = lib.bbs_rlc_verify_batch(ctx.handle, n, ptr(p_sigs), ptr(p_msgs), ptr(p_offs), L, ptr(seed32), ptr(verdict))
    if rc != 0 or verdict[0] != 1:
        raise RuntimeError("the signed batch does not verify")
    ctx.close()
    if env.rank != 0:
        return None
    step_ms = t / steps * 1e3
    return {"metric": "bls12_381_bbs_signatures_per_sec_L10", "value": env.world * n * steps / t, "unit": "signatures/s",
            "n_gpus": env.world, "n_total": env.world * n, "n_per_gpu": n, "steps": steps, "warmup": warmup, "ms_per_step": step_ms,
            "checked": True,
            "config": {"workload": f"batch sign: {env.world * n} message sets ({n} per GPU) x L={L} of 32 B under one key (BASELINE "
                                   "configs[4], first leg); the batch is then accepted by the random-linear-combination check",
                       "l2": "256 MB flush write between timed iterations", "sharding": "by item index, no collective"},
            "e2e": {"value": env.world * n * steps / te, "unit": "signatures/s",
                    "h2d_bytes_per_step": int(p_msgs.numel() + p_offs.numel() * 8), "d2h_bytes_per_step": int(p_sigs.numel() + n)},
            "gpu_launches": int(launches),
            "kernels_ms": {"msg_to_scalars": kt[0], "sign_kernel": kt[1]},
            "roofline": dict(imad_roofline(env, "sign_kernel<Bls>", n, PRODUCTS_SIGN, kt[1], traffic_key="sign_kernel<Bls>"),
                             note="products per item are SURVEY 8d's model (8-bit fixed-base windows, 255-bit variable-base multiplication); "
                                  "the kernel needs fewer (GLV halves, 16-bit tables, one inversion per block), so the fraction can exceed 1")}


def bench_rlc(env, n, steps, warmup, L=10, seed=99):
    """BASELINE configs[4], second leg: ONE random-linear-combination verdict for world * n valid signatures under one
    issuer.  Every rank reduces its shard to two compressed G1 points through the host-buffer call (coefficients indexed
    globally, copies inside), the 96-byte partials are all-gathered (the path's only exchange), rank 0 adds them and does
    the single pairing.  There is no device-buffer entry point for this mode: `value` is the end-to-end number."""
    torch, lib, api, dist = env.torch, env.lib, env.api, env.dist
    world, rank = env.world, env.rank
    ctx = api.BatchContext(api.BLS12_381, IRTF_PK, header=b"", n_messages=L, device=env.local)
    rng = np.random.default_rng(seed + rank)
    p_msgs = env.pin(rng.integers(0, 256, size=n * L * MSG_BYTES, dtype=np.uint8))
    p_offs = env.pin(np.arange(n * L + 1, dtype=np.uint64) * MSG_BYTES)
    p_sigs = env.pin(np.zeros(n * SIG_BYTES, dtype=np.uint8))
    st = np.zeros(n, dtype=np.uint8)
    sk = np.frombuffer(IRTF_SK.to_bytes(32, "little"), dtype=np.uint8).copy()
    _check(lib, lib.bbs_sign_batch(ctx.handle, ptr(sk), n, ptr(p_msgs), ptr(p_offs), L, ptr(p_sigs), None, ptr(st)))
    # the seed is drawn after the batch is fixed, by rank 0, and shared; seeded, so that runs get the same inputs
    seed_t = torch.from_numpy(rng.integers(0, 256, size=32, dtype=np.uint8)).to(env.dev)
    if world > 1:
        dist.broadcast(seed_t, 0)
    seed32 = seed_t.cpu().numpy()
    verdict = np.zeros(1, dtype=np.uint8)
    parts = np.zeros(96, dtype=np.uint8)
    pst = np.zeros(1, dtype=np.uint8)
    d_parts = torch.zeros(96, dtype=torch.uint8, device=env.dev)
    d_all = torch.zeros(96 * world, dtype=torch.uint8, device=env.dev)

    def step(expect=1):
        if world == 1:
            _check(lib, lib.bbs_rlc_verify_batch(ctx.handle, n, ptr(p_sigs), ptr(p_msgs), ptr(p_offs), L, ptr(seed32), ptr(verdict)))
        else:
            rc = lib.bbs_rlc_partial(ctx.handle, n, ptr(p_sigs), ptr(p_msgs), ptr(p_offs), L, ptr(seed32), C.c_uint64(rank * n),
                                     ptr(parts), ptr(pst))
            if rc != 0 or pst[0] != 1:
                raise RuntimeError(lib.bbs_last_error().decode() or f"rlc partial status {pst[0]}")
            d_parts.copy_(torch.from_numpy(parts))
            dist.all_gather_into_tensor(d_all, d_parts)
            if rank == 0:
                allp = d_all.cpu().numpy()
                _check(lib, lib.bbs_rlc_combine(ctx.handle, world, ptr(allp), ptr(verdict)))
            else:
                verdict[0] = expect
        if verdict[0] != expect:
            raise RuntimeError(f"rlc verdict {verdict[0]}, expected {expect}")

    lib.bbs_ctx_set_profiling(ctx.handle, 1)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    kt = env.kernel_times(ctx, 7)
    lib.bbs_ctx_set_profiling(ctx.handle, 0)
    launches0 = ctx.launch_count()
    t = env.time_host(step, steps)
    launches = (ctx.launch_count() - launches0) // max(steps, 1)
    env.keep("rlc_verdict", verdict)
    # a corrupted batch must be rejected (one flipped bit of e in the last rank's shard)
    if rank == world - 1:
        p_sigs.numpy()[48] ^= 1
    step(expect=0)
    ctx.close()
    if rank != 0:
        return None
    v = world * n * steps / t
    names = ["first_chunk_upload_and_msg_to_scalars", "chunked_msg_to_scalars_and_rlc_prep_under_the_uploads", "msm_scan_scatter",
             "msm_bucket", "msm_reduce", "rlc_msm_finish", "pairing"]
    return {"metric": "bls12_381_bbs_rlc_batch_verified_signatures_per_sec_L10", "value": v, "unit": "signatures/s",
            "n_gpus": world, "n_total": world * n, "n_per_gpu": n, "steps": steps, "warmup": warmup, "ms_per_step": t / steps * 1e3,
            "checked": True, "value_is_e2e": True,
            "config": {"workload": f"random-linear-combination batch verify: ONE verdict for {world * n} valid signatures x L={L} "
                                   f"under one issuer ({n} per GPU; partial G1 sums of the shards combined on rank 0, then one pairing; "
                                   "BASELINE configs[4], second leg; pinned host buffers, copies inside the timed region); a batch with "
                                   "one flipped bit is rejected",
                       "l2": "inputs (1.7 GB per 4M signatures) stream from host memory every step", "sharding": "by item index; "
                       "96-byte partials all-gathered"},
            "e2e": {"value": v, "unit": "signatures/s", "h2d_bytes_per_step": int(p_msgs.numel() + p_offs.numel() * 8 + p_sigs.numel()),
                    "d2h_bytes_per_step": 2 * 48 + 1},
            "gpu_launches": int(launches),
            "kernels_ms": dict(zip(names, kt)),
            "roofline": imad_roofline(env, "whole step (bucket MSM pipeline; co-limited by 70 SHA-256 blocks per signature on the ALU pipe)",
                                      n, PRODUCTS_RLC, t / steps * 1e3, traffic_key="msm_bucket_kernel<Bls>")}


EXTRAS = {"proof": bench_proof, "proof_l10": bench_proof_l10, "bn254": bench_bn254, "sign": bench_sign, "rlc": bench_rlc}


def run_ours(args):
    env = Env()
    out = None
    try:
        if args.workload == "verify":
            out = bench_verify(env, args)
            extra = {}
            for name in args.extras:
                n = max(TOTALS[name] // env.world, 1) if args.extra_n is None else args.extra_n
                rec = EXTRAS[name](env, n, min(args.steps, args.extra_steps), 3)
                if rec is not None:
                    rec["scaling"] = "strong"
                    extra[name] = rec
            if out is not None and extra:
                out["extra"] = extra
        else:
            n = args.n if args.n is not None else max(TOTALS[args.workload] // env.world, 1)
            rec = EXTRAS[args.workload](env, n, args.steps, args.warmup)
            if rec is not None:
                rec.update({"higher_is_better": True, "scaling": "strong" if args.n is None else "weak", "vs_baseline": None,
                            "dtype": "u32", "data": "synthetic"})
            out = rec
        if out is not None and env.world == 1 and not args.no_cpu and args.workload == "verify":
            out["cpu_baseline"] = cpu_baseline(args, sample=args.cpu_sample)
        if args.dump_outputs and env.rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in env.outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    finally:
        env.close()
    return out


# one extra workload on its own (tests/test_gpu_fullsize.py)
def run_single(workload, n, steps=1, warmup=3):
    env = Env()
    try:
        return EXTRAS[workload](env, n, steps, warmup)
    finally:
        env.close()


def cpu_baseline(args, sample):
    """The oracle port of the reference's per-item path (msg_to_scalars + core_verify with two pairings) on
    the host.  Uses oracle/_ref/ (compiled C restatement, all cores) when present, else the big-int Python
    oracle on one core."""
    from oracle import cpu_ref
    return cpu_ref.time_verify(L=args.L, sample=sample)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    from oracle import cpu_ref
    vals = []
    for _ in range(args.warmup):
        cpu_ref.time_verify(L=args.L, sample=max(args.cpu_sample // 4, 1))
    last = None
    t_total = 0.0
    for _ in range(args.steps):
        last = cpu_ref.time_verify(L=args.L, sample=args.cpu_sample)
        vals.append(last["value"])
        t_total += last["seconds"]
    v = float(np.mean(vals))
    return {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_total / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        # the same workload as our arm; every step times a bounded sample of it (named in cpu_baseline.sample): CPU
        # throughput does not depend on the batch size
        "config": verify_config(N_DEFAULT if args.n is None else args.n, args.L),
        "cpu_baseline": {k: last[k] for k in ("value", "unit", "cores", "kind", "sample", "as_reference") if k in last},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=None, help="items per GPU (verify: 65,536; other workloads: BASELINE total / N)")
    ap.add_argument("--L", type=int, default=L_DEFAULT)
    ap.add_argument("--cpu-sample", type=int, default=0, help="signatures per CPU-baseline step (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--workload", default="verify", choices=["verify", "proof", "proof_l10", "rlc", "bn254", "sign"],
                    help="verify = BASELINE configs[1] (the headline) with the other configs under `extra`")
    ap.add_argument("--extras", default="proof_l10,proof,bn254,sign,rlc", help="comma list of extra workloads of the default run ('' = none)")
    ap.add_argument("--extra-steps", type=int, default=3, help="timed steps per extra workload (at most --steps)")
    ap.add_argument("--extra-n", type=int, default=None, help="items per GPU for every extra workload (default: BASELINE total / N)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="our arm: write what the last timed step of each workload returned (status vectors, signatures, the "
                         "RLC verdict) as DIR/<name>.npy in float32, at most 2^20 values each (a fixed seeded sample of "
                         "larger outputs); the inputs are seeded, so runs with the same arguments compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.extras = [x for x in args.extras.split(",") if x]
    if args.impl == "reference":
        out = run_reference(args)
    else:
        if args.workload == "verify" and args.n is None:
            args.n = N_DEFAULT
        out = run_ours(args)
    if out is not None:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
