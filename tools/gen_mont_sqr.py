#!/usr/bin/env python3
"""Generates bbs_sign_b200/csrc/gen_mont_sqr.cuh: dedicated Montgomery SQUARINGS for the two base fields
(BLS12-381 Fp: 12 limbs, BN254 Fp: 8 limbs) -- n(n+1)/2 + n^2 + n products instead of the 2n^2 + n of a
multiplication (234 vs 300, 108 vs 136: the S of SURVEY 8d's counting model).

    a^2 = sum_i a_i 2^(64 i) * ( a_i + 2 * (a >> 32(i+1)) * 2^32 )

Row i multiplies a_i by the limbs  m_0 = a_i,  m_1 = a_{i+1} << 1,  m_k = (a_{i+k} << 1) | (a_{i+k-1} >> 31)  (k >= 2) of the
doubled upper part, so the cross products are never doubled afterwards (the doubled limbs are shared by all rows; both
moduli leave the top bit of the top limb free, so the doubled value still has n limbs).  Products at even word positions
accumulate in E, products at odd positions in O (value O * 2^32): every (lo, hi) destination is a fixed aligned register
pair, the condition for ptxas to fuse mad.lo.cc / madc.hi.cc into IMAD.WIDE.U32.X (tools/gen_mont_mul.py).  Then
T = E + (O << 32) and one Montgomery reduction with the modulus as immediates (tools/gen_coop.py redc_prog).

Like the other generators this one EXECUTES every program on integers (emulated carry flag, lost-carry assertions) against
a*a*R^-1 mod p before it prints anything."""
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gen_coop import Prog, redc_prog, addsub_prog, limbs, P_BLS, P_BN, arr, MASK  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "bbs_sign_b200", "csrc", "gen_mont_sqr.cuh")


def sqr_wide_prog(n):
    """t0..t_{2n-1} = a^2 from a_i, s_k = a_k << 1 (k = 1..n-1), d_k = funnel(a_{k-1}, a_k) (k = 2..n-1).
    E lives in t*, O in o* (value at word + 1)."""
    P = Prog()
    tops = {"t": 0, "o": 0}

    def limb(i, k):
        if k == 0:
            return f"a{i}"
        if k == 1:
            return f"s{i + 1}"
        return f"d{i + k}"

    def chain(arr_name, pairs, size):
        """pairs: [(index of lo word, x, y)] with consecutive even indexes; one statement, carry threaded to the end"""
        top = tops[arr_name]
        W = lambda j: f"{arr_name}{j}"
        ops = []
        for t, (idx, x, y) in enumerate(pairs):
            lo, hi = idx, idx + 1
            ops.append(("mad.lo.cc" if t == 0 else "madc.lo.cc", W(lo), x, y, W(lo) if lo < top else 0))
            ops.append(("madc.hi.cc", W(hi), x, y, W(hi) if hi < top else 0))
        j = pairs[-1][0] + 2
        newtop = max(top, j)
        while j < size:
            if j >= top:
                ops.append(("addc", W(j), 0, 0))            # fresh word takes the carry: cannot overflow
                newtop = max(newtop, j + 1)
                break
            last = j == size - 1
            ops.append(("addc" if last else "addc.cc", W(j), W(j), 0))
            j += 1
        else:
            # the chain ended at the top of the array: the flag must be clear (checked by the emulator through a dummy op)
            ops.append(("addc", "cz", 0, 0))
        tops[arr_name] = newtop
        P.stmt(ops)

    for i in range(n):
        ks = list(range(0, n - i))
        ev = [(2 * i + k, limb(i, k), f"a{i}") for k in ks if k % 2 == 0]
        od = [(2 * i + k - 1, limb(i, k), f"a{i}") for k in ks if k % 2 == 1]
        if ev:
            chain("t", ev, 2 * n)
        if od:
            chain("o", od, 2 * n - 1)
    # zero the words never written; T = E + (O << 32) is a second program (merge_prog)
    for name, size in (("t", 2 * n), ("o", 2 * n - 1)):
        for j in range(tops[name], size):
            P.stmt([("add", f"{name}{j}", 0, 0)])
    return P


def merge_prog(n):
    M = addsub_prog([f"t{j}" for j in range(1, 2 * n)], [f"o{j}" for j in range(2 * n - 1)], False)
    M.wrap_ok = {"cy"}          # a^2 fits 2n words: a lost carry at the top is an error
    return M


def env_for(a, n):
    env = {"m": 0, "cy": 0, "cz": 0}
    al = limbs(a, n)
    for i in range(n):
        env[f"a{i}"] = al[i]
    for k in range(1, n):
        env[f"s{k}"] = (al[k] << 1) & MASK
        env[f"d{k}"] = ((al[k] << 1) | (al[k - 1] >> 31)) & MASK
    return env


def check(n, p, trials=400, operands=None):
    """operands: values a < 2^(32n - 1) to run instead of the edge and random ones"""
    assert p < 1 << (32 * n - 1), "the doubled operand must fit in n limbs"
    R = 1 << (32 * n)
    rnd = random.Random(300 + n)
    W = sqr_wide_prog(n)
    M = merge_prog(n)
    Rd = redc_prog(n, p)
    if operands is None:
        edge = [0, 1, p - 1, p - 2, R % p, (1 << (32 * n - 1)) - 1, int("5" * (8 * n), 16) % p, int("a" * (8 * n), 16) >> 1,
                (1 << (32 * n - 1)) - (1 << 31), sum(0xffffffff << (64 * k) for k in range(n // 2)) >> 1]
        operands = edge + [rnd.randrange(p) for _ in range(trials - len(edge))]
    for t, a in enumerate(operands):
        assert 0 <= a < 1 << (32 * n - 1)
        env = env_for(a, n)
        W.run(env)
        M.run(env)
        T = sum(env[f"t{j}"] << (32 * j) for j in range(2 * n))
        assert T == a * a, (n, t, hex(a))
        assert env["cz"] == 0
        Rd.run(env)
        r = sum(env[v] << (32 * j) for j, v in enumerate(Rd.result))
        if a < p:
            assert r < 2 * p and (r * R - a * a) % p == 0, (n, t)
    return W, M, Rd


def emit(n, p, name):
    W, M, Rd = check(n, p)
    mp = arr([("t", "t[%d]"), ("o", "o[%d]"), ("a", "A[%d]"), ("s", "s[%d]"), ("d", "d[%d]")])    # m, cy, x0: scalars
    res = ", ".join(mp(v) for v in Rd.result)
    products = n * (n + 1) // 2 + n * n + n
    return "\n".join([
        f"// r[0..{n - 1}] = A*A*R^-1 mod-ish (< 2p) for {name}; {products} products; caller does the final conditional subtraction",
        f"__device__ __forceinline__ void bbs_mont_sqr_{name}(uint32_t* r, const uint32_t* A) {{",
        f"    uint32_t t[{2 * n}], o[{2 * n}], s[{n}], d[{n}], m, x0, cy, cz = 0;",
        f"#pragma unroll",
        f"    for (int k = 1; k < {n}; k++) {{ s[k] = A[k] << 1; d[k] = __funnelshift_l(A[k - 1], A[k], 1); }}",
        W.emit(mp),
        M.emit(mp),
        Rd.emit(mp),
        f"    const uint32_t res[{n}] = {{{res}}};",
        f"#pragma unroll",
        f"    for (int k = 0; k < {n}; k++) r[k] = res[k];",
        f"    (void)cy; (void)cz;",
        "}", ""])


def main():
    s = ["// GENERATED by tools/gen_mont_sqr.py (self-verified by emulation before emission) -- do not edit.",
         "#pragma once", "#include <stdint.h>", "#ifdef __CUDA_ARCH__", "",
         emit(12, P_BLS, "bls_fp"), emit(8, P_BN, "bn_fp"), "#endif  // __CUDA_ARCH__"]
    with open(OUT, "w") as f:
        f.write("\n".join(s) + "\n")
    print("verified and wrote", os.path.normpath(OUT))


if __name__ == "__main__":
    main()
