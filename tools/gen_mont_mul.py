#!/usr/bin/env python3
"""Generates bbs_sign_b200/csrc/gen_mont_mul.cuh: fully unrolled Montgomery products for N = 8 and 12
32-bit limbs as PTX carry chains whose (lo, hi) register pairs never change parity.

Why: ptxas fuses `mad.lo.cc d0,a,b,c0; madc.hi.cc d1,a,b,c1` into one full-rate IMAD.WIDE.U32.X only when
(d0,d1) and (c0,c1) are aligned register pairs.  With a single accumulator array the even-limb chain pairs
(t0,t1),(t2,t3).. and the odd-limb chain pairs (t1,t2),(t3,t4).., so every word changes pair parity between
chains and ptxas inserts one IMAD.MOV per product (seen in the round-1 SASS).  Here the running value is kept
as T = E + O * 2^32 in TWO arrays: products of even limbs of the multiplicand go to E, products of odd limbs
go to O, each with fixed pairs.  Dividing by 2^32 after a reduction row swaps the roles of the two arrays
(E' = O + E[1], O' = E[2..]) which is pure index bookkeeping, done here at generation time.

The generator builds an abstract instruction list, EXECUTES it on random big integers (with an emulated
carry flag) to prove it computes a*b*R^-1 mod p (and the squaring / wide-product variants), and only then
prints it as inline asm.  Every chain is ONE asm statement.
"""
import os
import random

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "bbs_sign_b200", "csrc", "gen_mont_mul.cuh")
MASK = 0xFFFFFFFF


class Prog:
    """A list of statements; a statement is a list of PTX-like ops sharing one carry flag."""

    def __init__(self):
        self.stmts = []

    def stmt(self, ops):
        self.stmts.append(ops)

    # ---- emulation -----------------------------------------------------------------------------
    def run(self, env):
        for ops in self.stmts:
            cc = 0
            for op in ops:
                name, d, srcs = op[0], op[1], op[2:]
                v = [env[s] if isinstance(s, str) else s for s in srcs]
                if name in ("mul.lo", "mul.hi"):
                    pr = v[0] * v[1]
                    env[d] = (pr & MASK) if name == "mul.lo" else (pr >> 32)
                    continue
                base = name.replace(".cc", "")
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
                else:
                    assert t >> 32 == 0, ("carry lost", op)
        return env

    # ---- emission ------------------------------------------------------------------------------
    def emit(self, arrays):
        """arrays: name -> C expression prefix, e.g. 'a' -> 'a[%d]'.  Variables are like 'a3', 'e5', 'm'."""
        out = []
        for ops in self.stmts:
            outs, ins = [], []   # ordered operand lists
            written = set()
            for op in ops:
                d = op[1]
                if d not in outs:
                    outs.append(d)
            # an output that is read before/without being written first is "+", else "="
            rw = {}
            seen_w = set()
            for op in ops:
                for s in op[2:]:
                    if isinstance(s, str) and s in outs and s not in seen_w:
                        rw[s] = "+"
                seen_w.add(op[1])
            for op in ops:
                for s in op[2:]:
                    if isinstance(s, str) and s not in outs and s not in ins:
                        ins.append(s)
            idx = {v: i for i, v in enumerate(outs + ins)}
            lines = []
            for op in ops:
                name, d, srcs = op[0], op[1], op[2:]
                args = ", ".join(("%%%d" % idx[s]) if isinstance(s, str) else str(s) for s in (d,) + tuple(srcs))
                lines.append(f"{name}.u32 {args};")
            cexpr = lambda v: arrays(v)
            o = ", ".join(f'"{rw.get(v, "=")}&r"({cexpr(v)})' for v in outs)
            i = ", ".join(f'"r"({cexpr(v)})' for v in ins)
            body = " ".join(lines)
            out.append(f'    asm("{body}" : {o} : {i});')
        return "\n".join(out)


def mont_mul_prog(n, square=False):
    """T = E + O*2^32; returns (prog, result variable names r0..r{n-1} before the final conditional subtraction)."""
    P = Prog()
    bname = (lambda i: f"a{i}") if square else (lambda i: f"b{i}")
    E = [f"e{j}" for j in range(n + 1)]   # logical E[j] -> variable
    O = [f"o{j}" for j in range(n)]
    half = n // 2

    def chain_inplace(arr, limbs, mult, first_op_carry_in=False, top=None):
        ops = []
        for k in range(half):
            lo, hi = arr[2 * k], arr[2 * k + 1]
            ops.append(("mad.lo.cc" if (k == 0 and not first_op_carry_in) else "madc.lo.cc", lo, limbs[k], mult, lo))
            last = (k == half - 1) and top is None
            ops.append(("madc.hi" if last else "madc.hi.cc", hi, limbs[k], mult, hi))
        if top is not None:
            ops.append(("addc", top, top, 0))
        return ops

    a_even = [f"a{2 * k}" for k in range(half)]
    a_odd = [f"a{2 * k + 1}" for k in range(half)]
    p_even = [f"p{2 * k}" for k in range(half)]
    p_odd = [f"p{2 * k + 1}" for k in range(half)]

    for i in range(n):
        bi = bname(i)
        if i == 0:
            ops = []
            for k in range(half):
                ops.append(("mul.lo", E[2 * k], a_even[k], bi))
                ops.append(("mul.hi", E[2 * k + 1], a_even[k], bi))
            P.stmt(ops)
            ops = []
            for k in range(half):
                ops.append(("mul.lo", O[2 * k], a_odd[k], bi))
                ops.append(("mul.hi", O[2 * k + 1], a_odd[k], bi))
            P.stmt(ops)
            P.stmt([("add", E[n], 0, 0)])
        else:
            # role swap after the division by 2^32:  E' = O + E[1],  O' = E[2..n] ++ [fresh],  E'[n] = old E[0] (== 0)
            oldE, oldO = E, O
            E = oldO + [oldE[0]]
            O = oldE[2:] + [oldE[1]]
            ops = [("add.cc", E[0], E[0], oldE[1])]
            for k in range(half):
                lo, hi = O[2 * k], O[2 * k + 1]
                ops.append(("madc.lo.cc", lo, a_odd[k], bi, lo))
                if k == half - 1:
                    ops.append(("madc.hi", hi, a_odd[k], bi, 0))       # fresh top word (old E[1] is dead here)
                else:
                    ops.append(("madc.hi.cc", hi, a_odd[k], bi, hi))
            P.stmt(ops)
            P.stmt(chain_inplace(E, a_even, bi, top=E[n]))
        P.stmt([("mul.lo", "m", E[0], "inv")])
        P.stmt(chain_inplace(O, p_odd, "m"))
        P.stmt(chain_inplace(E, p_even, "m", top=E[n]))
    # result = O + (E >> 32)  (E[0] == 0)
    ops = []
    for j in range(n):
        ops.append(("add.cc" if j == 0 else ("addc.cc" if j < n - 1 else "addc"), f"r{j}", O[j], E[j + 1]))
    P.stmt(ops)
    return P


def check(n, p, trials=200, operands=None):
    """operands: (a, b) pairs with a, b < p to run instead of the edge and random ones (the squaring takes each a once)"""
    R = 1 << (32 * n)
    inv = (-pow(p, -1, 1 << 32)) % (1 << 32)
    rnd = random.Random(n)
    if operands is None:
        operands = [([0, 1, p - 1, R % p][t], [p - 1, 0, p - 1, R % p][t]) if t < 4 else (rnd.randrange(p), rnd.randrange(p))
                    for t in range(trials)]
    for square in (False, True):
        prog = mont_mul_prog(n, square)
        for t, (a, b) in enumerate(sorted({(a, a) for a, _ in operands}) if square else operands):
            env = {"inv": inv, "m": 0}
            for i in range(n):
                env[f"a{i}"] = (a >> (32 * i)) & MASK
                env[f"b{i}"] = (b >> (32 * i)) & MASK
                env[f"p{i}"] = (p >> (32 * i)) & MASK
            prog.run(env)
            r = sum(env[f"r{j}"] << (32 * j) for j in range(n))
            assert r < 2 * p and (r - a * b * pow(R, -1, p)) % p == 0, (n, square, t)
    return True


def emit_func(n, square):
    prog = mont_mul_prog(n, square)

    def arrays(v):
        if v in ("m", "inv"):
            return v
        name, idx = v[0], int(v[1:])
        return {"a": "A[%d]", "b": "B[%d]", "p": "M[%d]", "e": "e[%d]", "o": "o[%d]", "r": "t[%d]"}[name] % idx

    fname = f"bbs_mont_sqr{n}" if square else f"bbs_mont_mul{n}"
    sig = f"uint32_t* t, const uint32_t* A, const uint32_t* M, uint32_t inv" if square else \
          f"uint32_t* t, const uint32_t* A, const uint32_t* B, const uint32_t* M, uint32_t inv"
    return (f"// t[0..{n - 1}] = A*{'A' if square else 'B'}*R^-1 mod-ish (< 2p); caller does the final conditional subtraction\n"
            f"__device__ __forceinline__ void {fname}({sig}) {{\n"
            f"    uint32_t e[{n + 1}], o[{n}], m;\n{prog.emit(arrays)}\n}}\n")


def main():
    x = -0xD201000000010000
    r_bls = x ** 4 - x ** 2 + 1
    p_bls = (x - 1) ** 2 * r_bls // 3 + x
    t = 4965661367192848881
    p_bn = 36 * t ** 4 + 36 * t ** 3 + 24 * t ** 2 + 6 * t + 1
    r_bn = 36 * t ** 4 + 36 * t ** 3 + 18 * t ** 2 + 6 * t + 1
    for n, p in ((12, p_bls), (8, r_bls), (8, p_bn), (8, r_bn)):
        check(n, p)
    s = ["// GENERATED by tools/gen_mont_mul.py (self-verified by emulation before emission) -- do not edit.",
         "#pragma once", "#include <stdint.h>", "#ifdef __CUDA_ARCH__", ""]
    for n in (8, 12):
        s.append(emit_func(n, False))
    s.append("template <int N> __device__ __forceinline__ void bbs_mont_mul(uint32_t* t, const uint32_t* A, const uint32_t* B, const uint32_t* M, uint32_t inv);")
    for n in (8, 12):
        s.append(f"template <> __device__ __forceinline__ void bbs_mont_mul<{n}>(uint32_t* t, const uint32_t* A, const uint32_t* B, const uint32_t* M, uint32_t inv) {{ bbs_mont_mul{n}(t, A, B, M, inv); }}")
    s.append("#endif  // __CUDA_ARCH__")
    with open(OUT, "w") as f:
        f.write("\n".join(s) + "\n")
    print("verified and wrote", os.path.normpath(OUT))


if __name__ == "__main__":
    main()
