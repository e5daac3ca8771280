#!/usr/bin/env python3
"""Generates bbs_sign_b200/csrc/gen_coop.cuh: the register-level primitives of the cooperative pairing
kernel (pairing_coop.cuh) as PTX carry chains that ptxas turns into full-rate IMAD.WIDE.U32[.X].

The cooperative kernel accumulates UNREDUCED double-width products (lazy reduction): an Fp2 coefficient of an
Fp12 product is  REDC( KP + sum_t +-x_t*y_t + beta*Z*R )  with one Montgomery reduction per Fp coefficient
instead of one per product.  Primitives (N = limbs of Fp: 12 for BLS12-381, 8 for BN254):

  coop_wmul_e<N>(w, a, b)   w[0..2N-1]  = sum_{i+j even} a_j b_i 2^(32(i+j))      (fresh, even-aligned pairs)
  coop_wmul_o<N>(v, a, b)   v[0..2N-2]  = sum_{i+j odd } a_j b_i 2^(32(i+j-1))    (fresh, value sits at word 1)
  coop_merge<N>(w, v)       w += v << 32: the full 2N-word product
  coop_acc_{add,sub}_e<N>(acc, w)       acc[0..2N] +-= w, two's complement
  coop_acc_{add,sub}_hi<N>(acc, z)      acc[N..2N] +-= z[0..N-1]                  (adds z*R before REDC)
  coop_redc_<curve>(r, acc)             r[0..N-1] = (acc + M p) / R,  needs 0 <= acc < (2^(32N) - p) R
  coop_sub_kp_<curve><K>(d, r)          d = r - K p, returns the borrow mask      (canonicalisation steps)
  coop_add_p_<curve>(r)                 r += p  ... etc.

Every row of a product is ONE asm statement whose (lo, hi) destination pairs keep a fixed register-pair
alignment (products at even word positions live in `w`, products at odd positions in `v`), which is the
condition for the mad.lo.cc / madc.hi.cc -> IMAD.WIDE fusion (see tools/gen_mont_mul.py).  The generator
EXECUTES every program on random big integers with an emulated carry flag before printing it.
"""
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gen_mont_mul import Prog as BaseProg, MASK  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "bbs_sign_b200", "csrc", "gen_coop.cuh")

X_BLS = -0xD201000000010000
R_BLS = X_BLS ** 4 - X_BLS ** 2 + 1
P_BLS = (X_BLS - 1) ** 2 * R_BLS // 3 + X_BLS
T_BN = 4965661367192848881
P_BN = 36 * T_BN ** 4 + 36 * T_BN ** 3 + 24 * T_BN ** 2 + 6 * T_BN + 1
CURVES = {"bls": (12, P_BLS), "bn": (8, P_BN)}


class Prog(BaseProg):
    """BaseProg + subtraction with borrow + hex immediates."""

    def run(self, env):
        for ops in self.stmts:
            cc = 0
            for op in ops:
                name, d, srcs = op[0], op[1], op[2:]
                v = [env[s] if isinstance(s, str) else s for s in srcs]
                base = name.replace(".cc", "")
                if name in ("mul.lo", "mul.hi"):
                    pr = v[0] * v[1]
                    env[d] = (pr & MASK) if name == "mul.lo" else (pr >> 32)
                    continue
                if base in ("sub", "subc"):
                    bin_ = cc if base == "subc" else 0
                    t = v[0] - v[1] - bin_
                    env[d] = t & MASK
                    if name.endswith(".cc"):
                        cc = 1 if t < 0 else 0
                    continue
                cin = cc if base.startswith(("madc", "addc")) else 0
                if base in ("mad.lo", "madc.lo"):
                    t = ((v[0] * v[1]) & MASK) + v[2] + cin
                elif base in ("mad.hi", "madc.hi"):
                    t = ((v[0] * v[1]) >> 32) + v[2] + cin
                elif base in ("add", "addc"):
                    t = v[0] + v[1] + cin
                else:
                    raise ValueError(name)
                env[d] = t & MASK
                if name.endswith(".cc"):
                    cc = t >> 32
                elif d not in getattr(self, "wrap_ok", ()):
                    assert t >> 32 == 0, ("carry lost", op)
        return env

    def emit(self, arrays):
        out = []
        for ops in self.stmts:
            outs, ins = [], []
            for op in ops:
                if op[1] not in outs:
                    outs.append(op[1])
            rw, seen_w = {}, set()
            for op in ops:
                for s in op[2:]:
                    if isinstance(s, str) and s in outs and s not in seen_w:
                        rw[s] = "+"
                seen_w.add(op[1])
            for op in ops:
                for s in op[2:]:
                    if isinstance(s, str) and s not in outs and s not in ins:
                        ins.append(s)
            assert len(outs) + len(ins) <= 30, ("too many asm operands", len(outs) + len(ins))
            idx = {v: i for i, v in enumerate(outs + ins)}
            lines = []
            for op in ops:
                name, d, srcs = op[0], op[1], op[2:]
                args = ", ".join(("%%%d" % idx[s]) if isinstance(s, str) else ("0x%x" % s) for s in (d,) + tuple(srcs))
                lines.append(f"{name}.u32 {args};")
            o = ", ".join(f'"{rw.get(v, "=")}&r"({arrays(v)})' if rw.get(v) != "+" else f'"+r"({arrays(v)})' for v in outs)
            i = ", ".join(f'"r"({arrays(v)})' for v in ins)
            out.append(f'    asm("{" ".join(lines)}" : {o} : {i});')
        return "\n".join(out)


def limbs(x, n):
    return [(x >> (32 * i)) & MASK for i in range(n)]


def from_limbs(env, name, n):
    return sum(env[f"{name}{i}"] << (32 * i) for i in range(n))


# ---- fresh half products ------------------------------------------------------------------------------
def wmul_prog(n, odd, rows_per_stmt=2):
    """even part: w_k at word k; odd part: v_k at word k+1.  Rows alternate between the multiplicand's even and
    odd limbs so that every product lands on a fixed (2k, 2k+1) pair of the output array.

    `rows_per_stmt` consecutive rows share one asm statement and ONE carry chain: a row always ends with the carry
    flag clear (its last instruction cannot overflow), so the next row may start with madc.  That makes ptxas keep
    the rows of a block in order; without it the scheduler walks the rows x columns grid column-wise and has to
    spill up to 12 live carry predicates through P2R / ISETP (seen in the SASS of the first version)."""
    P = Prog()
    W = lambda k: f"w{k}"
    half = n // 2
    cur = []
    for i in range(n):
        # limbs j of a with (i + j) of the wanted parity
        js = [j for j in range(n) if (i + j) % 2 == (1 if odd else 0)]
        pos0 = i + js[0] - (1 if odd else 0)          # array index of the first pair (even)
        assert pos0 % 2 == 0
        if i == 0:
            ops = []
            for k, j in enumerate(js):
                ops.append(("mul.lo", W(pos0 + 2 * k), f"a{j}", "b0"))
                ops.append(("mul.hi", W(pos0 + 2 * k + 1), f"a{j}", "b0"))
            P.stmt(ops)
            top = pos0 + 2 * half          # first index never written so far
            continue
        ops = []
        chained = len(cur) > 0
        for k, j in enumerate(js):
            lo, hi = pos0 + 2 * k, pos0 + 2 * k + 1
            first = k == 0 and not chained
            if lo < top:
                ops.append(("mad.lo.cc" if first else "madc.lo.cc", W(lo), f"a{j}", f"b{i}", W(lo)))
            else:
                ops.append(("mad.lo.cc" if first else "madc.lo.cc", W(lo), f"a{j}", f"b{i}", 0))
            last = k == half - 1
            if hi < top:
                ops.append(("madc.hi.cc", W(hi), f"a{j}", f"b{i}", W(hi)))
                if last:
                    ops.append(("addc.cc", W(hi + 1), 0, 0))      # carry into a fresh word; leaves CF = 0
                    newtop = hi + 2
            else:
                assert last
                ops.append(("madc.hi.cc", W(hi), f"a{j}", f"b{i}", 0))   # hi + carry never overflows: CF = 0
                newtop = hi + 1
        top = newtop
        cur += ops
        if (i % rows_per_stmt) == 0 or i == n - 1:
            P.stmt(cur)
            cur = []
    assert not cur
    return P, top


def check_wmul(n, trials=300, operands=None):
    """operands: (a, b) pairs of n-word values to run instead of the edge and random ones"""
    rnd = random.Random(100 + n)
    pe, te = wmul_prog(n, False)
    po, to = wmul_prog(n, True)
    assert te == 2 * n and to == 2 * n - 1, (te, to)
    if operands is None:
        operands = [([0, (1 << (32 * n)) - 1, 1][t], [(1 << (32 * n)) - 1, (1 << (32 * n)) - 1, 0][t]) if t < 3 else
                    (rnd.getrandbits(32 * n), rnd.getrandbits(32 * n)) for t in range(trials)]
    for t, (a, b) in enumerate(operands):
        env = {}
        for i in range(n):
            env[f"a{i}"], env[f"b{i}"] = limbs(a, n)[i], limbs(b, n)[i]
        e1 = pe.run(dict(env))
        e2 = po.run(dict(env))
        E = from_limbs(e1, "w", te)
        O = from_limbs(e2, "w", to)
        assert E + (O << 32) == a * b, (n, t)


# ---- chunked add / sub chains ----------------------------------------------------------------------------
def addsub_prog(dst, src, sub, chunk=13, final_wrap=True):
    """dst[k] +-= src[k] over len(src) words, then the carry / borrow is propagated through the rest of dst.
    src entries may be ints (immediates).  Two's-complement wrap at the top of dst is allowed."""
    P = Prog()
    P.wrap_ok = set()
    n = len(dst)
    srcs = list(src) + [0] * (n - len(src))
    k = 0
    first_chunk = True
    while k < n:
        m = min(chunk, n - k)
        ops = []
        for q in range(m):
            idx = k + q
            lastword = idx == n - 1
            if q == 0 and first_chunk:
                name = ("sub" if sub else "add") + ("" if lastword else ".cc")
            elif q == 0:
                # re-inject the carry / borrow saved by the previous chunk
                ops.append(("sub.cc", "cy", 0, "cy") if sub else ("add.cc", "cy", "cy", MASK))
                name = ("subc" if sub else "addc") + ("" if lastword else ".cc")
            else:
                name = ("subc" if sub else "addc") + ("" if lastword else ".cc")
            ops.append((name, dst[idx], dst[idx], srcs[idx]))
            if lastword:
                P.wrap_ok.add(dst[idx])
        if k + m < n:
            ops.append(("subc", "cy", 0, 0) if sub else ("addc", "cy", 0, 0))
            P.wrap_ok.add("cy")
        P.stmt(ops)
        k += m
        first_chunk = False
    return P


def merge_prog(n):
    """w[1 + k] += v[k], k = 0..2n-2: the two half products of coop_wmul_{e,o} -> the full 2n-word product in w."""
    dst = [f"w{k + 1}" for k in range(2 * n - 1)]
    src = [f"v{k}" for k in range(2 * n - 1)]
    P = addsub_prog(dst, src, False)
    P.wrap_ok = {"cy"}          # the product fits 2n words: a lost carry at the top is an error
    return P


def check_merge(n, trials=200, operands=None):
    """operands: (a, b) pairs of n-word values to run instead of the edge and random ones"""
    rnd = random.Random(300 + n)
    pe, _ = wmul_prog(n, False)
    po, _ = wmul_prog(n, True)
    pm = merge_prog(n)
    if operands is None:
        top = (1 << (32 * n)) - 1
        operands = [(top, top)] + [(rnd.getrandbits(32 * n), rnd.getrandbits(32 * n)) for _ in range(trials - 1)]
    for a, b in operands:
        env = {}
        for i in range(n):
            env[f"a{i}"], env[f"b{i}"] = limbs(a, n)[i], limbs(b, n)[i]
        e1 = pe.run(dict(env))
        e2 = po.run(dict(env))
        env2 = {"cy": 0}
        for k in range(2 * n):
            env2[f"w{k}"] = e1[f"w{k}"]
        for k in range(2 * n - 1):
            env2[f"v{k}"] = e2[f"w{k}"]
        pm.run(env2)
        assert from_limbs(env2, "w", 2 * n) == a * b


def check_addsub():
    rnd = random.Random(7)
    for n, ns in ((25, 24), (25, 23), (17, 16), (17, 17), (13, 12), (9, 8)):
        for sub in (False, True):
            dst = [f"d{i}" for i in range(n)]
            src = [f"s{i}" for i in range(ns)]
            P = addsub_prog(dst, src, sub)
            for t in range(200):
                d = rnd.getrandbits(32 * n) if t > 2 else [0, (1 << (32 * n)) - 1, 1][t]
                s = rnd.getrandbits(32 * ns) if t > 2 else [(1 << (32 * ns)) - 1, (1 << (32 * ns)) - 1, 0][t]
                env = {"cy": 0}
                for i in range(n):
                    env[f"d{i}"] = limbs(d, n)[i]
                for i in range(ns):
                    env[f"s{i}"] = limbs(s, ns)[i]
                # the emulator asserts on lost carries except for wrap_ok destinations
                P.run(env)
                want = (d - s if sub else d + s) % (1 << (32 * n))
                assert from_limbs(env, "d", n) == want, (n, ns, sub, t)


# ---- Montgomery reduction of a double-width value ----------------------------------------------------------
def redc_prog(n, p):
    """r = (T + M p) / R for T = t0..t_{2n-1} (t_{2n} must be zero): "multiply by one" CIOS on the low half with the
    running value split as E + O*2^32 (gen_mont_mul.py), then + the high half.  p and -p^-1 are immediates."""
    inv = (-pow(p, -1, 1 << 32)) % (1 << 32)
    pl = limbs(p, n)
    P = Prog()
    half = n // 2
    E = [f"t{j}" for j in range(n)] + ["x0"]    # low half of the input, modified in place; x0 = extra top word
    O = [f"o{j}" for j in range(n)]
    p_even = [pl[2 * k] for k in range(half)]
    p_odd = [pl[2 * k + 1] for k in range(half)]

    def echain(Ev, first_fold=None):
        ops = []
        for k in range(half):
            lo, hi = Ev[2 * k], Ev[2 * k + 1]
            ops.append(("mad.lo.cc" if k == 0 else "madc.lo.cc", lo, "m", p_even[k], lo))
            ops.append(("madc.hi.cc", hi, "m", p_even[k], hi))
        ops.append(("addc", Ev[n], Ev[n], 0))
        return ops

    for i in range(n):
        if i == 0:
            P.stmt([("add", "x0", 0, 0)])
            P.stmt([("mul.lo", "m", E[0], inv)])
            ops = []
            for k in range(half):
                ops.append(("mul.lo", O[2 * k], "m", p_odd[k]))
                ops.append(("mul.hi", O[2 * k + 1], "m", p_odd[k]))
            P.stmt(ops)
            P.stmt(echain(E))
        else:
            oldE, oldO = E, O
            E = oldO + [oldE[0]]                  # oldE[0] == 0 after the previous row
            O = oldE[2:] + [oldE[1]]              # top word is fresh (oldE[1] is consumed by the fold)
            ops = [("add.cc", E[0], E[0], oldE[1]), ("mul.lo", "m", E[0], inv)]
            for k in range(half):
                lo, hi = O[2 * k], O[2 * k + 1]
                ops.append(("madc.lo.cc", lo, "m", p_odd[k], lo))
                if k == half - 1:
                    ops.append(("madc.hi", hi, "m", p_odd[k], 0))
                else:
                    ops.append(("madc.hi.cc", hi, "m", p_odd[k], hi))
            P.stmt(ops)
            P.stmt(echain(E))
    # result = O + (E >> 32) + T_hi     (E[0] == 0), accumulated in place in O
    P.wrap_ok = set()
    ops = []
    for j in range(n):
        ops.append(("add.cc" if j == 0 else ("addc.cc" if j < n - 1 else "addc"), O[j], O[j], E[j + 1]))
    P.stmt(ops)
    ops = []
    for j in range(n):
        ops.append(("add.cc" if j == 0 else ("addc.cc" if j < n - 1 else "addc"), O[j], O[j], f"t{n + j}"))
    P.stmt(ops)
    P.result = list(O)
    return P


def redc_wide_prog(n, p):
    """redc_prog for accumulators that use the top word t_{2n}: the result has n + 1 words, r < T / R + p."""
    P = redc_prog(n, p)
    # drop the two final n-word additions and redo them with a carry word
    final2 = P.stmts[-2:]
    P.stmts = P.stmts[:-2]
    O = P.result
    Esrc = [op[3] for op in final2[0]]
    ops = [("add.cc" if j == 0 else "addc.cc", O[j], O[j], Esrc[j]) for j in range(n)]
    ops.append(("addc", "x1", 0, 0))
    P.stmt(ops)
    ops = [("add.cc" if j == 0 else "addc.cc", O[j], O[j], f"t{n + j}") for j in range(n)]
    ops.append(("addc", "x1", "x1", f"t{2 * n}"))
    P.stmt(ops)
    P.result = list(O) + ["x1"]
    return P


def check_redc_wide(n, p, limit_p2, trials=300, operands=None):
    """operands: accumulators 0 <= T < limit_p2 p^2 to run instead of the edge and random ones"""
    R = 1 << (32 * n)
    rnd = random.Random(900 + n)
    P = redc_wide_prog(n, p)
    lim = limit_p2 * p * p
    assert lim < 1 << (32 * (2 * n + 1))
    if operands is None:
        operands = [0, lim - 1, R - 1, p * p * 12] + [rnd.randrange(lim) for _ in range(trials - 4)]
    for t, T in enumerate(operands):
        assert 0 <= T < lim
        env = {"m": 0}
        for i in range(2 * n + 1):
            env[f"t{i}"] = limbs(T, 2 * n + 1)[i]
        P.run(env)
        r = sum(env[v] << (32 * j) for j, v in enumerate(P.result))
        assert (r * R - T) % p == 0 and r < T // R + p + 1, (n, t)


def check_canon_q(p, trials=200000, operands=None):
    """pairing_coop.cuh Coop<Bn>::canon_q: the quotient estimate from the top 29 bits is q or q - 1 for every w < 128 p.
    operands: values w to run instead of the edge and random ones"""
    M = (1 << 32) // ((p >> 232) + 1)
    assert M == 1354
    rnd = random.Random(77)
    cases = operands
    if cases is None:
        cases = [k * p + d for k in range(128) for d in (-1, 0, 1, 1 << 200, -(1 << 200)) if 0 <= k * p + d < 128 * p]
        cases += [rnd.randrange(128 * p) for _ in range(trials)]
    for w in cases:
        assert 0 <= w < 128 * p
        v = ((w >> 256) << 24) | (((w >> 224) & MASK) >> 8)
        assert v < 1 << 32
        q = (v * M) >> 32
        assert q in (w // p, w // p - 1), (w, q)


def check_canon_q_bls(p, trials=200000, operands=None):
    """pairing_coop.cuh Coop<Bls>::canon_q: for every 12-word w the estimate q^ = (w[11] * M) >> 56,
    M = floor(2^56 / ((p >> 352) + 1)), is q or q - 1 with q = floor(w / p) < 10.
    operands: values w to run instead of the edge and random ones"""
    M = (1 << 56) // ((p >> 352) + 1)
    assert M == 165164498 and M < 1 << 32
    R = 1 << 384
    assert 9 * p < R < 10 * p
    rnd = random.Random(78)
    cases = operands
    if cases is None:
        cases = [k * p + d for k in range(11) for d in (-1, 0, 1, 1 << 352, -(1 << 352), (1 << 352) - 1) if 0 <= k * p + d < R]
        cases += [R - 1, 0] + [rnd.randrange(R) for _ in range(trials)]
        cases += [(v << 352) + d for v in (rnd.randrange(1 << 32) for _ in range(20000)) for d in (0, (1 << 352) - 1)]
    for w in cases:
        assert 0 <= w < R
        q = ((w >> 352) * M) >> 56
        assert q in (w // p, w // p - 1) and q < 10, (w, q)


def check_redc(n, p, trials=300, operands=None):
    """operands: accumulators 0 <= T < (R - p) R to run instead of the edge and random ones"""
    R = 1 << (32 * n)
    rnd = random.Random(200 + n)
    P = redc_prog(n, p)
    lim = (R - p) * R
    if operands is None:
        operands = [0, lim - 1, R - 1, p * p * 12] + [rnd.randrange(lim) for _ in range(trials - 4)]
    for t, T in enumerate(operands):
        assert 0 <= T < lim
        env = {"m": 0}
        for i in range(2 * n):
            env[f"t{i}"] = limbs(T, 2 * n)[i]
        P.run(env)
        r = sum(env[v] << (32 * j) for j, v in enumerate(P.result))
        assert (r * R - T) % p == 0 and r < T // R + p + 1, (n, t)


# ---- emission -------------------------------------------------------------------------------------------
def arr(mapping):
    def f(v):
        for prefix, expr in mapping:
            if v.startswith(prefix) and v[len(prefix):].isdigit():
                return expr % int(v[len(prefix):])
        if v in ("m", "cy", "cz", "x0", "x1", "ext"):
            return v
        raise KeyError(v)
    return f


def emit_all():
    s = ["// GENERATED by tools/gen_coop.py (every program self-verified by emulation before emission) -- do not edit.",
         "#pragma once", "#include <stdint.h>", "#ifdef __CUDACC__", ""]
    for n in (8, 12):
        for odd in (False, True):
            prog, top = wmul_prog(n, odd, int(os.environ.get('COOP_ROWS_PER_STMT_%d' % n, 3)))
            nm = "o" if odd else "e"
            s.append(f"// {'odd' if odd else 'even'}-aligned half of the {n}x{n}-limb product, fresh ({top} words)")
            s.append(f"__device__ __forceinline__ void coop_wmul_{nm}{n}(uint32_t* w, const uint32_t* a, const uint32_t* b) {{")
            s.append(prog.emit(arr([("w", "w[%d]"), ("a", "a[%d]"), ("b", "b[%d]")])))
            s.append("}\n")
        # accumulate: acc has 2n+1 words
        for nm, ns, off in (("e", 2 * n, 0), ("hi", n, n)):
            for sub in (False, True):
                dst = [f"d{i}" for i in range(off, 2 * n + 1)]
                src = [f"s{i}" for i in range(ns)]
                prog = addsub_prog(dst, src, sub)
                op = "sub" if sub else "add"
                s.append(f"// acc[{off}..{2 * n}] {'-' if sub else '+'}= w[0..{ns - 1}] (two's complement, wraps at the top)")
                s.append(f"__device__ __forceinline__ void coop_acc_{op}_{nm}{n}(uint32_t* acc, const uint32_t* w) {{")
                s.append("    uint32_t cy = 0; (void)cy;")
                s.append(prog.emit(arr([("d", "acc[%d]"), ("s", "w[%d]")])))
                s.append("}\n")
        prog = merge_prog(n)
        s.append(f"// w[1..{2 * n - 1}] += v[0..{2 * n - 2}]: even + odd half products -> full product in w")
        s.append(f"__device__ __forceinline__ void coop_merge{n}(uint32_t* w, const uint32_t* v) {{")
        s.append("    uint32_t cy = 0; (void)cy;")
        s.append(prog.emit(arr([("w", "w[%d]"), ("v", "v[%d]")])))
        s.append("}\n")
        # plain n-word add / sub (operand forms), returning nothing (no overflow by construction)
        for sub in (False, True):
            dst = [f"d{i}" for i in range(n)]
            src = [f"s{i}" for i in range(n)]
            prog = addsub_prog(dst, src, sub)
            op = "sub" if sub else "add"
            s.append(f"__device__ __forceinline__ void coop_{op}n{n}(uint32_t* d, const uint32_t* w) {{")
            s.append(prog.emit(arr([("d", "d[%d]"), ("s", "w[%d]")])))
            s.append("}\n")
    for cname, (n, p) in CURVES.items():
        prog = redc_prog(n, p)
        s.append(f"// r[0..{n - 1}] = (t + M p) / 2^{32 * n}; t[0..{2 * n - 1}] is destroyed, t[{2 * n}] must be zero; needs t < (2^{32 * n} - p) 2^{32 * n}")
        s.append(f"__device__ __forceinline__ void coop_redc_{cname}(uint32_t* r, uint32_t* t) {{")
        s.append(f"    uint32_t o[{n}], m, x0;")
        amap = arr([("t", "t[%d]"), ("o", "o[%d]")])
        s.append(prog.emit(amap))
        s.append("    " + " ".join(f"r[{j}] = {amap(v)};" for j, v in enumerate(prog.result)))
        s.append("}\n")
        # d = r - K p with borrow mask, for canonicalisation; and r += p, r = K p - r helpers
        R = 1 << (32 * n)
        for K in (1, 2, 4, 8):
            if K * p >= R:
                continue
            kp = limbs(K * p, n)
            P = Prog()
            P.wrap_ok = {"cy"}
            ops = []
            for j in range(n):
                ops.append(("sub.cc" if j == 0 else "subc.cc", f"d{j}", f"r{j}", kp[j]))
            ops.append(("subc", "cy", 0, 0))
            P.stmt(ops)
            # emulate
            rnd = random.Random(K)
            for t in range(100):
                r = rnd.randrange(R)
                env = {"cy": 0}
                for j in range(n):
                    env[f"r{j}"] = limbs(r, n)[j]
                P.run(env)
                assert from_limbs(env, "d", n) == (r - K * p) % R and env["cy"] == (MASK if r < K * p else 0)
            s.append(f"// d = r - {K}p; returns 0xffffffff when r < {K}p (borrow)")
            s.append(f"__device__ __forceinline__ uint32_t coop_sub_{K}p_{cname}(uint32_t* d, const uint32_t* r) {{")
            s.append("    uint32_t cy = 0; (void)cy;")
            s.append(P.emit(arr([("d", "d[%d]"), ("r", "r[%d]")])))
            s.append("    return cy;")
            s.append("}\n")
        if cname == "bn":
            # wide variant: accumulators use all 2n+1 words (xi = 9 + u is applied to them), the reduction returns n+1 words
            prog = redc_wide_prog(n, p)
            s.append(f"// r[0..{n}] = (t + M p) / 2^{32 * n} for t[0..{2 * n}] (destroyed): r < t / 2^{32 * n} + p")
            s.append(f"__device__ __forceinline__ void coop_redc_wide_{cname}(uint32_t* r, uint32_t* t) {{")
            s.append(f"    uint32_t o[{n}], m, x0, x1;")
            amap = arr([("t", "t[%d]"), ("o", "o[%d]")])
            s.append(prog.emit(amap))
            s.append("    " + " ".join(f"r[{j}] = {amap(v)};" for j, v in enumerate(prog.result)))
            s.append("}\n")
            for K in (1, 2, 4, 8, 16, 32, 64):
                kp = limbs(K * p, n + 1)
                P = Prog()
                P.wrap_ok = {"cy"}
                ops = [("sub.cc" if j == 0 else "subc.cc", f"d{j}", f"r{j}", kp[j]) for j in range(n + 1)]
                ops.append(("subc", "cy", 0, 0))
                P.stmt(ops)
                rnd = random.Random(K + 50)
                R9 = 1 << (32 * (n + 1))
                for t in range(100):
                    r = rnd.randrange(128 * p)
                    env = {"cy": 0}
                    for j in range(n + 1):
                        env[f"r{j}"] = limbs(r, n + 1)[j]
                    P.run(env)
                    assert from_limbs(env, "d", n + 1) == (r - K * p) % R9 and env["cy"] == (MASK if r < K * p else 0)
                s.append(f"// d = r - {K}p on {n + 1} words; returns 0xffffffff when r < {K}p (borrow)")
                s.append(f"__device__ __forceinline__ uint32_t coop_sub_{K}p_{cname}{n + 1}(uint32_t* d, const uint32_t* r) {{")
                s.append("    uint32_t cy = 0; (void)cy;")
                s.append(P.emit(arr([("d", "d[%d]"), ("r", "r[%d]")])))
                s.append("    return cy;")
                s.append("}\n")
            for sub in (False, True):
                dst = [f"d{i}" for i in range(2 * n + 1)]
                src = [f"s{i}" for i in range(2 * n + 1)]
                prog = addsub_prog(dst, src, sub)
                op = "sub" if sub else "add"
                s.append(f"// acc[0..{2 * n}] {'-' if sub else '+'}= w[0..{2 * n}] (two's complement, wraps at the top)")
                s.append(f"__device__ __forceinline__ void coop_acc_{op}_f{n}(uint32_t* acc, const uint32_t* w) {{")
                s.append("    uint32_t cy = 0; (void)cy;")
                s.append(prog.emit(arr([("d", "acc[%d]"), ("s", "w[%d]")])))
                s.append("}\n")
        # r += p (for the difference form c0 - c1 + p)
        P = Prog()
        pl = limbs(p, n)
        ops = []
        for j in range(n):
            ops.append(("add.cc" if j == 0 else ("addc.cc" if j < n - 1 else "addc"), f"r{j}", f"r{j}", pl[j]))
        P.stmt(ops)
        s.append(f"__device__ __forceinline__ void coop_add_p_{cname}(uint32_t* r) {{")
        s.append(P.emit(arr([("r", "r[%d]")])))
        s.append("}\n")
    s.append("#endif  // __CUDACC__")
    return "\n".join(s) + "\n"


def main():
    for n in (8, 12):
        check_wmul(n)
    check_addsub()
    for n in (8, 12):
        check_merge(n)
    for cname, (n, p) in CURVES.items():
        check_redc(n, p)
    check_redc_wide(8, P_BN, 127 * (1 << 256) // P_BN)
    check_canon_q(P_BN)
    check_canon_q_bls(P_BLS)
    txt = emit_all()
    with open(OUT, "w") as f:
        f.write(txt)
    print("verified and wrote", os.path.normpath(OUT), len(txt), "bytes")


if __name__ == "__main__":
    main()
