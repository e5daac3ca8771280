"""Field arithmetic of the four prime fields (BLS12-381 Fp / Fr, BN254 Fp / Fr) at structured operands, through
bbs_selftest_field, compared with Python integers.

Production values live in the Montgomery domain, so the operands are also fed as Montgomery words (op | 0x100): a
chosen limb pattern such as a run of 0xffffffff, p - 1 or R - 1 mod p then reaches the mad.lo.cc / madc.hi.cc chains of
gen_mont_mul.cuh and gen_mont_sqr.cuh as it is.  Without the flag the library multiplies each operand by R first,
which turns every edge value but 0 into an effectively random one.  The canonical-I/O mode is run on the same set too.

Every binary operation runs on all pairs of the structured set and on 4,096 random pairs; every unary one on the
set and the random values.  The host simulation (`-m "not gpu"`) checks the expectations and the plumbing; the GPU
tests run the compiled sm_100a kernels, including the dedicated squaring (op 9)."""
import os
import random
import sys

import numpy as np
import pytest

import hostsim
import parity_cases as P
from bbs_sign_b200 import _native

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import coop_consts as CC  # noqa: E402
import gen_coop  # noqa: E402
import gen_mont_mul  # noqa: E402
import gen_mont_sqr  # noqa: E402

MONT = 0x100
# op codes per field kind (include/bbs_b200.h); sqrt and the dedicated squaring exist on the base fields only
FP_OPS = {"mul": 0, "add": 1, "sub": 2, "inv": 3, "sqrt": 4, "inv_vt": 7, "sqr": 9, "neg": 10}
FR_OPS = {"mul": 5, "add": 11, "sub": 12, "inv": 6, "inv_vt": 8, "neg": 13}
BINARY = ("mul", "add", "sub")


def field_params(curve, kind):
    ocs = P.SUITES[curve][1]
    m = ocs.p if kind == "Fp" else ocs.r
    width = ocs.fp_bytes if kind == "Fp" else 32
    return m, width, (FP_OPS if kind == "Fp" else FR_OPS)


def structured_set(m, nlimbs):
    """Edge operands below m: small values and their negatives, halves, powers of the Montgomery radix, 2^k and
    2^k +- 1 and m - 2^k at every limb boundary, the largest value below m whose lower limbs are all 0xffffffff, and
    alternating / repeated limb patterns (each reduced below m)."""
    R = 1 << (32 * nlimbs)
    s = [0, 1, 2, 3, m - 1, m - 2, m - 3, (m - 1) // 2, (m + 1) // 2,
         R % m, R * R % m, pow(R, -1, m), -R % m, (R - 1) % m]
    for j in range(1, nlimbs + 1):
        for k in (32 * j - 1, 32 * j, 32 * j + 1):
            s += [(1 << k) % m, ((1 << k) - 1) % m, ((1 << k) + 1) % m, (m - (1 << k)) % m]
    s += limb_patterns(m, nlimbs)
    assert all(0 <= x < m for x in s)
    return sorted(set(s))


def limb_patterns(m, nlimbs):
    """the largest value below m whose lower limbs are all 0xffffffff, and repeated limb patterns reduced below m"""
    lower = 32 * (nlimbs - 1)

    def limbs(f):
        return sum(f(i) << (32 * i) for i in range(nlimbs)) % m

    return [(((m >> lower) - 1) << lower) | ((1 << lower) - 1),
            limbs(lambda i: 0xffffffff if i % 2 == 0 else 0), limbs(lambda i: 0 if i % 2 == 0 else 0xffffffff),
            limbs(lambda i: 0xaaaaaaaa if i % 2 == 0 else 0x55555555),
            limbs(lambda i: 0x55555555 if i % 2 == 0 else 0xaaaaaaaa), limbs(lambda i: 0x80000000),
            limbs(lambda i: 0xffffffff)]


def partners(m, nlimbs):
    """second operands for the emulator checks, which are too slow for every pair of the structured set: the ends of
    the range, R^k mod m, every run of 0xffffffff limbs from the bottom (2^(32j) - 1) and the limb patterns"""
    R = 1 << (32 * nlimbs)
    return sorted({0, 1, 2, m - 1, m - 2, (m - 1) // 2, (m + 1) // 2, R % m, (R - 1) % m, R * R % m}
                  | {((1 << (32 * j)) - 1) % m for j in range(1, nlimbs + 1)} | set(limb_patterns(m, nlimbs)))


def expected(name, x, y, m, mont, nlimbs):
    """op on the values the operands stand for, returned in the same representation as the operands"""
    R = 1 << (32 * nlimbs)
    if mont:
        ri = pow(R, -1, m)
        x, y = x * ri % m, y * ri % m
    if name == "mul":
        v = x * y % m
    elif name == "sqr":
        v = x * x % m
    elif name == "add":
        v = (x + y) % m
    elif name == "sub":
        v = (x - y) % m
    elif name == "neg":
        v = -x % m
    elif name in ("inv", "inv_vt"):
        v = pow(x, m - 2, m)
    else:                                    # sqrt: the kernel returns x^((p+1)/4) when that is a root, else 0
        s = pow(x, (m + 1) // 4, m)
        v = s if s * s % m == x else 0
    return v * R % m if mont else v


def run_op(lib, curve_id, op, xs, ys, width):
    n = len(xs)
    a = np.frombuffer(b"".join(x.to_bytes(width, "little") for x in xs), dtype=np.uint8)
    b = np.frombuffer(b"".join(y.to_bytes(width, "little") for y in ys), dtype=np.uint8)
    out = np.zeros(n * width, dtype=np.uint8)
    rc = lib.bbs_selftest_field(curve_id, 0, op, n, P.ptr(a), P.ptr(b), P.ptr(out))
    assert rc == 0, lib.bbs_last_error()
    raw = out.tobytes()
    return [int.from_bytes(raw[i * width:(i + 1) * width], "little") for i in range(n)]


def check_field(lib, curve, kind, mont, n_random=4096):
    suite = P.SUITES[curve][0]
    m, width, ops = field_params(curve, kind)
    nlimbs = width // 4
    S = structured_set(m, nlimbs)
    rnd = random.Random(f"{curve}/{kind}/{mont}")
    rx = [rnd.randrange(m) for _ in range(n_random)]
    ry = [rnd.randrange(m) for _ in range(n_random)]
    for name, op in ops.items():
        if name in BINARY:
            xs = [x for x in S for _ in S] + rx
            ys = [y for _ in S for y in S] + ry
        else:
            xs = S + rx
            if name == "sqrt":       # half of the random values are squares (of the represented value)
                R = 1 << (32 * nlimbs)
                xs = S + [x * x * (R if mont else 1) % m for x in rx[: n_random // 2]] + rx[n_random // 2:]
            ys = list(reversed(xs))
        got = run_op(lib, suite.curve_id, op | (MONT if mont else 0), xs, ys, width)
        bad = [(hex(x), hex(y), hex(g)) for x, y, g in zip(xs, ys, got)
               if g != expected(name, x, y, m, mont, nlimbs)]
        assert not bad, (curve, kind, name, "mont" if mont else "canonical", len(bad), bad[:4])


def test_structured_set_covers_the_edges():
    m, width, _ = field_params("BLS12_381", "Fp")
    S = structured_set(m, width // 4)
    R = 1 << (32 * 12)
    for v in (0, m - 1, (m + 1) // 2, R % m, (R - 1) % m, (1 << 383) % m, ((1 << 352) + 1) % m):
        assert v in S
    # every 32-bit boundary of the 12-limb field appears, and a value with all eleven lower limbs 0xffffffff
    assert all((1 << (32 * j)) % m in S for j in range(1, 13))
    assert any(x & ((1 << 352) - 1) == (1 << 352) - 1 and x < m and (x >> 352) == (m >> 352) - 1 for x in S)


def test_expectations_in_montgomery_form():
    """the expected values of the Montgomery mode are mont(op(A R^-1, B R^-1)): spot-check against plain algebra"""
    m, width, _ = field_params("BN254", "Fp")
    R = 1 << 256
    x, y = 12345, m - 7
    X, Y = x * R % m, y * R % m
    assert expected("mul", X, Y, m, True, 8) == x * y * R % m
    assert expected("inv", X, 0, m, True, 8) == pow(x, -1, m) * R % m
    assert expected("sqr", R % m, 0, m, True, 8) == R % m           # mont(1)^2 = mont(1)
    assert expected("sqrt", 4 * R % m, 0, m, True, 8) in (2 * R % m, (m - 2) * R % m)


@pytest.fixture(scope="module")
def hostsim_lib():
    path = hostsim.build()
    return _native.load(path, allow_host_simulation=True)   # tests only: the product loader refuses non-CUDA builds


@pytest.mark.parametrize("mont", [True, False], ids=["mont", "canonical"])
@pytest.mark.parametrize("kind", ["Fp", "Fr"])
@pytest.mark.parametrize("curve", ["BLS12_381", "BN254"])
def test_field_edges_host_simulation(hostsim_lib, curve, kind, mont):
    check_field(hostsim_lib, curve, kind, mont)


def test_field_rejects_unknown_ops(hostsim_lib):
    a = np.zeros(48, dtype=np.uint8)
    out = np.zeros(48, dtype=np.uint8)
    for op in (14, 0x100 | 14, 0x200, -1):
        assert hostsim_lib.bbs_selftest_field(P.SUITES["BLS12_381"][0].curve_id, 0, op, 1, P.ptr(a), P.ptr(a),
                                              P.ptr(out)) != 0


@pytest.mark.gpu
@pytest.mark.parametrize("mont", [True, False], ids=["mont", "canonical"])
@pytest.mark.parametrize("kind", ["Fp", "Fr"])
@pytest.mark.parametrize("curve", ["BLS12_381", "BN254"])
def test_field_edges_gpu(curve, kind, mont):
    check_field(_native.load(), curve, kind, mont)


# ---- the generators' own emulators (tools/gen_mont_mul.py, gen_mont_sqr.py, gen_coop.py) at the same edges -----------
# Each generator executes its PTX carry chains on Python integers (emulated carry flag, lost-carry assertions) before it
# prints them; by default on a few fixed and many random operands.  Here the chains run on the structured set and on the
# ends of the ranges the kernels feed them: the largest square operand, the cooperative operand forms c0 + c1,
# c0 - c1 + p and their left shifts, and accumulators up to the REDC bound of the cooperative program.
def _moduli():
    out = {}
    for curve in ("BLS12_381", "BN254"):
        for kind in ("Fp", "Fr"):
            m, width, _ = field_params(curve, kind)
            out[f"{curve}/{kind}"] = (width // 4, m)
    return out


def operand_forms(n, p):
    """the largest values of the cooperative kernel's operand forms that fit n words: c0 + c1 <= 2p - 2,
    c0 - c1 + p <= 2p - 1, each shifted left by 0..2 (coop_prog.py encodes shifts up to 2)"""
    R = 1 << (32 * n)
    return [v for base in (p - 1, 2 * p - 2, 2 * p - 1) for s in range(3) for v in (base << s,) if v < R] + [R - 1]


@pytest.mark.parametrize("field", ["BLS12_381/Fp", "BLS12_381/Fr", "BN254/Fp", "BN254/Fr"])
def test_mont_mul_generator_at_edges(field):
    n, m = _moduli()[field]
    S = structured_set(m, n)
    gen_mont_mul.check(n, m, operands=[(a, b) for a in S for b in partners(m, n)])


@pytest.mark.parametrize("field", ["BLS12_381/Fp", "BN254/Fp"])
def test_mont_sqr_generator_at_edges(field):
    n, p = _moduli()[field]
    top = 1 << (32 * n - 1)      # the doubled operand must fit n words
    gen_mont_sqr.check(n, p, operands=structured_set(p, n) + [top - 1, top - 2, top - (1 << 31), 2 * p - 1, 2 * p - 2])


@pytest.mark.parametrize("curve", ["BLS12_381", "BN254"])
def test_coop_products_at_edges(curve):
    n, p = _moduli()[f"{curve}/Fp"]
    X = structured_set(p, n) + operand_forms(n, p)
    gen_coop.check_wmul(n, operands=[(a, b) for a in X for b in partners(p, n) + operand_forms(n, p)])
    # the merge's carry chain is longest where both half products are large
    gen_coop.check_merge(n, operands=[(a, b) for a in operand_forms(n, p) for b in X])


def accumulator_edges(n, p, lim):
    """REDC inputs: the ends of [0, lim), multiples of p^2 and of p R around every whole multiple below lim, and values
    whose low and high halves are structured"""
    R = 1 << (32 * n)
    S = structured_set(p, n)
    T = [0, 1, lim - 1, lim - 2, lim - p, R - 1, R, R + 1, p * p - 1, p * p, p * p + 1]
    T += [k * p * p + d for k in range(1, lim // (p * p) + 1) for d in (-1, 0, 1)]
    T += [k * p * R + d for k in range(1, lim // (p * R) + 1) for d in (-1, 0, 1)]
    T += [hi * R + lo for hi in S[:: max(1, len(S) // 24)] for lo in S + [R - 1]]
    return sorted({t for t in T if 0 <= t < lim})


def test_coop_redc_at_edges():
    n, p = _moduli()["BLS12_381/Fp"]
    R = 1 << (32 * n)
    lim = (R - p) * R
    assert CC.BLS.acc_limit * p * p == lim          # the program's accumulator bound is the reduction's input bound
    gen_coop.check_redc(n, p, operands=accumulator_edges(n, p, lim))
    n, p = _moduli()["BN254/Fp"]
    R = 1 << (32 * n)
    gen_coop.check_redc(n, p, operands=accumulator_edges(n, p, (R - p) * R))


def test_coop_redc_wide_at_edges():
    n, p = _moduli()["BN254/Fp"]
    limit_p2 = CC.BN.acc_limit                     # exact Fraction: (2^7 - 1) R / p
    lim = int(limit_p2 * p * p)
    assert lim == limit_p2 * p * p
    gen_coop.check_redc_wide(n, p, limit_p2, operands=accumulator_edges(n, p, lim))


def test_canon_q_at_every_multiple():
    p = gen_coop.P_BLS
    R = 1 << 384
    gen_coop.check_canon_q_bls(p, operands=[w for k in range(10) for d in (-1, 0, 1) for w in (k * p + d,) if 0 <= w < R]
                               + [R - 1, R - 2])
    p = gen_coop.P_BN
    gen_coop.check_canon_q(p, operands=[w for k in range(128) for d in (-1, 0, 1) for w in (k * p + d,)
                                        if 0 <= w < 128 * p] + [128 * p - 1])


def test_generated_headers_are_the_committed_ones(tmp_path, monkeypatch):
    """the operand lists change only the checks: regenerating prints the same .cuh files word for word"""
    csrc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bbs_sign_b200", "csrc")
    for mod, name in ((gen_mont_mul, "gen_mont_mul.cuh"), (gen_mont_sqr, "gen_mont_sqr.cuh"), (gen_coop, "gen_coop.cuh")):
        out = tmp_path / name
        monkeypatch.setattr(mod, "OUT", str(out))
        if mod is gen_coop:
            out.write_text(gen_coop.emit_all())          # main() would rerun the 200k-value canon_q checks
        else:
            mod.main()
        assert out.read_text() == open(os.path.join(csrc, name)).read(), name
