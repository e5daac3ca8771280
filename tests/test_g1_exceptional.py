"""The G1 group law at its exceptional cases: P + P, P + (-P) and the identity, inside the addition formulas, the Straus
products, the proof paths and the bucket MSMs of the random-linear-combination mode.

g1_add and g1_add_mixed (csrc/g1.cuh) are complete only through their rare-case branches: H == 0 doubles when rr == 0
and gives the identity otherwise.  Random inputs almost never reach those branches, so every case here is built to:
  1. bbs_selftest_g1 on Jacobian operands, one affine point under several Z = l (l = 1, p - 1, R^-1 mod p whose
     Montgomery word is 1, ...), and the Straus products g1_msm_scalar<C, 2 / 3> on scalars chosen so that the
     accumulator meets a table entry (equal points, opposite points, P and 32 P with digits one window apart, phi(P));
  2. proofs whose random scalars make Abar = D, Abar = -D and T1 = O, through generation and every verify path;
  3. (GPU) bucket MSMs over batches that draw their signatures from {P, -P, 2P, phi(P), Q}, at sizes up to one past the
     upload chunk, at forced window counts, with coefficient indexes crossing 2^32, S1 = O and a zero fixed-base scalar.
Every expectation comes from the oracle's exact integers (oracle/bbs_oracle.py); every comparison is on bytes."""
import hashlib
import random

import numpy as np
import pytest

import hostsim
import parity_cases as P
from bbs_sign_b200 import _native
from bbs_sign_b200 import api as A
from oracle import bbs_oracle as O

CURVES = ["BLS12_381", "BN254"]
ADD, ADD_MIXED, DBL, MSM2, MSM3 = range(5)
BLS_X = -0xd201000000010000
BN_T = 4965661367192848881


@pytest.fixture(scope="module")
def hs_lib():
    return _native.load(hostsim.build(), allow_host_simulation=True)


# ---- a model of g1_msm_win4 on discrete logarithms (which additions meet equal or opposite points) ---------------------
class Curve:
    """per-curve constants: the GLV eigenvalue lam with phi(x, y) = (beta x, y) = lam P, and the split of g1.cuh"""

    def __init__(self, name):
        self.name = name
        self.suite, self.ocs = P.SUITES[name]
        ocs = self.ocs
        self.F, self.p, self.r = ocs.F1, ocs.p, ocs.r
        self.n = ocs.fp_bytes // 4
        if name == "BLS12_381":
            self.lam = BLS_X * BLS_X - 1
        else:
            self.a, self.b = 6 * BN_T * BN_T + 2 * BN_T, 2 * BN_T + 1
            self.lam = self.a * pow(self.b, -1, self.r) % self.r
        # the cube root of unity in Fp that acts as lam on G1
        g = 2
        while pow(g, (self.p - 1) // 3, self.p) == 1:
            g += 1
        w = pow(g, (self.p - 1) // 3, self.p)
        lp = O.ec_mul(self.F, ocs.BP1, self.lam)
        self.beta = next(bt for bt in (w, w * w % self.p) if (bt * ocs.BP1[0] % self.p, ocs.BP1[1]) == lp)

    def phi(self, pt):
        return None if pt is None else (self.beta * pt[0] % self.p, pt[1])

    def split(self, k):
        if self.name == "BLS12_381":
            return k % self.lam, k // self.lam
        a, b, r = self.a, self.b, self.r
        kp = k + r
        c1 = ((a + b) * kp + 2 * b * b) * ((1 << 384) // r) >> 384      # the quotients by reciprocal, as bn_glv_split
        c2 = (b * kp - 2 * a * b) * ((1 << 320) // r) >> 320
        return kp - c1 * a - c2 * b, c1 * b - c2 * (a + b)

    def straus_events(self, logs, ks, solve=None):
        """the additions g1_msm_win4 makes for points logs[j] * G (None = identity) and scalars ks[j]: a list of
        'copy' (accumulator at O), 'dbl' (equal operands), 'cancel' (opposite operands) or 'add', and the result's log.
        solve = (j, 'dbl' | 'cancel'): logs[j] is chosen at point j's first addition so that it meets the accumulator
        (returned as a third value; None if the accumulator is O there)."""
        r = self.r
        logs = list(logs)
        C_ = sum(16 << (5 * w) for w in range(26))
        halves = []
        for k in ks:
            k1, k2 = self.split(k)
            assert (k1 + k2 * self.lam - k) % r == 0 and 0 <= k1 < 1 << 128 and 0 <= k2 < 1 << 128
            halves.append((k1 + C_, k2 + C_))
        acc, ev = 0, []

        def add(e):
            nonlocal acc
            ev.append("copy" if acc == 0 else "dbl" if acc == e else "cancel" if (acc + e) % r == 0 else "add")
            acc = (acc + e) % r

        for w in range(25, -1, -1):
            acc = acc * 32 % r
            for j, (u1, u2) in enumerate(halves):
                if logs[j] is None:
                    continue
                for u, mult in ((u1, 1), (u2, self.lam)):
                    d = ((u >> (5 * w)) & 31) - 16
                    if d and solve and solve[0] == j and logs[j] == "?":
                        if acc == 0:
                            return ev, None, None
                        logs[j] = (1 if solve[1] == "dbl" else -1) * acc * pow(d * mult, -1, r) % r
                    if d:
                        add(d * mult * logs[j] % r)
        return (ev, acc, logs) if solve else (ev, acc)


CURVE = {}


def curve(name):
    if name not in CURVE:
        CURVE[name] = Curve(name)
    return CURVE[name]


# ---- bbs_selftest_g1 ----------------------------------------------------------------------------------------------------
def jac(cv, pt, lam):
    """(l^2 x, l^3 y, l) as three canonical LE field elements; the identity is (l^2, l^3, 0)"""
    p, w = cv.p, cv.ocs.fp_bytes
    x, y, z = (1, 1, 0) if pt is None else (pt[0], pt[1], 1)
    vals = (x * lam * lam % p, y * pow(lam, 3, p) % p, z * lam % p)
    return b"".join(v.to_bytes(w, "little") for v in vals)


def run_g1(lib, cv, op, ps, qs=None, ks=None):
    """one bbs_selftest_g1 call: ps[i] (and qs[i]) operand bytes, ks[i] a list of scalars; the compressed results"""
    n = len(ps)
    buf = lambda b: np.frombuffer(b or b"\0", dtype=np.uint8).copy()
    p = buf(b"".join(ps))
    q = buf(b"".join(qs)) if qs is not None else None
    s = buf(b"".join(k.to_bytes(32, "little") for row in ks for k in row)) if ks is not None else None
    out = np.zeros(max(n, 1) * cv.suite.g1_bytes, dtype=np.uint8)
    rc = lib.bbs_selftest_g1(cv.suite.curve_id, 0, op, n, P.ptr(p), None if q is None else P.ptr(q),
                             None if s is None else P.ptr(s), P.ptr(out))
    assert rc == 0, lib.bbs_last_error()
    g = cv.suite.g1_bytes
    return [out[i * g:(i + 1) * g].tobytes() for i in range(n)]


def lambdas(cv):
    R = 1 << (32 * cv.n)
    return [1, cv.p - 1, pow(R, -1, cv.p), 2, random.Random(cv.name).randrange(2, cv.p)]


def pair_cases(cv):
    """(op, p bytes, q bytes, expected point, label) for the additions and the doubling"""
    F, rnd = cv.F, random.Random(3)
    Pt = O.ec_mul(F, cv.ocs.BP1, rnd.randrange(1, cv.r))
    nP, P2 = O.ec_neg(F, Pt), O.ec_add(F, Pt, Pt)
    lams = lambdas(cv)
    out = []
    for la in lams:
        for lb in lams:
            for name, a, b in (("P+P", Pt, Pt), ("P+(-P)", Pt, nP), ("P+2P", Pt, P2), ("2P+(-P)", P2, nP)):
                out.append((ADD, jac(cv, a, la), jac(cv, b, lb), O.ec_add(F, a, b), f"{name} l={la:#x},{lb:#x}"))
        for name, a, b in (("O+P", None, Pt), ("P+O", Pt, None), ("O+O", None, None)):
            out.append((ADD, jac(cv, a, la), jac(cv, b, lams[(lams.index(la) + 1) % len(lams)]), O.ec_add(F, a, b), name))
        for name, a, b in (("P+P", Pt, Pt), ("P+(-P)", Pt, nP), ("P+2P", Pt, P2), ("2P+(-P)", P2, nP), ("O+P", None, Pt)):
            out.append((ADD_MIXED, jac(cv, a, la), jac(cv, b, 1), O.ec_add(F, a, b), f"mixed {name} l={la:#x}"))
        for name, a in (("2P", Pt), ("2(-P)", nP), ("2O", None)):
            out.append((DBL, jac(cv, a, la), None, O.ec_add(F, a, a), f"dbl {name} l={la:#x}"))
    return out


def check_pairs(lib, cv):
    cases = pair_cases(cv)
    for op in (ADD, ADD_MIXED, DBL):
        sel = [c for c in cases if c[0] == op]
        got = run_g1(lib, cv, op, [c[1] for c in sel], [c[2] for c in sel] if op != DBL else None)
        for c, g in zip(sel, got):
            assert g == cv.ocs.g1_compress(c[3]), (cv.name, c[4])


def search(cv, logs, make, want, tries=2000):
    """scalars make(rnd) for which the modelled Straus loop makes a `want` addition"""
    rnd = random.Random(want + str(logs))
    for _ in range(tries):
        ks = make(rnd)
        ev, _ = cv.straus_events(logs, ks)
        if want in ev:
            return ks
    raise AssertionError(f"no scalars found for {want} at {logs}")


def straus_cases(cv):
    """(logs, scalars, label): points logs[j] * G (G a fixed random point), each case reaching the wanted branch"""
    r, lam, rnd = cv.r, cv.lam, random.Random(5)
    # scalars are built from their GLV halves (h1 + h2 lam) in ranges the split returns as they are (the model checks),
    # with the first half of the equal-scalar cases below the second: they meet at the second half's top windows
    H = lambda h1, h2: (h1 + h2 * lam) % r
    lo = lambda g: g.randrange(1 << 120, 1 << 122)
    hi = lambda g: g.randrange(1 << 124, 1 << 125)
    k = H(lo(rnd), hi(rnd))
    cases = [
        ([1, 1], [k, k], "dbl", "(P, P), equal scalars"),
        ([1, r - 1], [k, k], "cancel", "(P, -P), equal scalars"),
        ([1, 1, 1], [k, k, k], "dbl", "(P, P, P), equal scalars"),
        ([1, r - 1, 1], [k, k, k], "cancel", "(P, -P, P), equal scalars"),
        ([1, r - 1, 2], [k, k, k], "cancel", "(P, -P, 2P), equal scalars"),
    ]
    make = []
    if cv.name == "BLS12_381":
        # k = k1 + k2 lam with k1 < lam.  P's phi half against phi(P)'s own half: both tables hold d phi(P), under
        # different Z.  And m below 2^123 has 32 m's digits one window above its own, so the accumulator after P's digits
        # equals a table entry of 32P.  (BN254's lattice split returns neither a second half below the first nor halves
        # that small: there the solved points below take these roles.)
        phi2 = lambda g: (lambda x: [H(lo(g), x), H(x, lo(g))])(hi(g))
        phi3 = lambda g: (lambda x: [H(x, lo(g)), H(lo(g), x), H(lo(g), lo(g))])(hi(g))
        mid = lambda g: H(g.randrange(1 << 105, 1 << 115), g.randrange(1 << 90, 1 << 100))
        shifted = lambda g: (lambda m: [32 * m % r, m])(mid(g))
        shifted3 = lambda g: (lambda m: [1024 * m % r, 32 * m % r, m])(mid(g))
        make += [(phi2, [1, lam], "dbl", "(P, phi(P))"), (phi2, [1, r - lam], "cancel", "(P, -phi(P))"),
                 (phi3, [lam, 1, 32], "dbl", "(phi(P), P, 32P)"),
                 (shifted, [1, 32], "dbl", "(P, 32P), digits one window apart"),
                 (shifted, [1, r - 32], "cancel", "(P, -32P), digits one window apart"),
                 (shifted3, [1, 32, 1024], "dbl", "(P, 32P, 1024P), digits one window apart")]
    for mk, logs, what, label in make:
        cases.append((logs, search(cv, logs, mk, what), what, label))
    # on either curve: the point Q that equals (or cancels) the accumulator at Q's first addition, which then meets a
    # table entry held under another Z (the situation of P and 32P above)
    for logs, what in (([1, "?"], "dbl"), ([1, "?"], "cancel"), ([1, 2, "?"], "dbl"), ([1, "?", 3], "cancel"),
                       ([lam, "?"], "dbl"), ([1, lam, "?"], "cancel")):
        for t in range(50):
            g = random.Random(f"{what}{logs}{t}")
            ks = [H(hi(g), lo(g)) for _ in logs]
            _, _, solved = cv.straus_events(logs, ks, solve=(logs.index("?"), what))
            if solved is not None:
                break
        label = "(" + ", ".join("Q" if x == "?" else "phi(P)" if x == lam else f"{x}P" for x in logs) + f"), Q meets the accumulator: {what}"
        cases.append((solved, ks, what, label))
    # an identity slot, and the identity as the result
    cases.append(([1, None], [k, 7], "copy", "(P, O)"))
    cases.append(([None, 1, None], [3, k, 5], "copy", "(O, P, O)"))
    out = []
    for logs, ks, what, label in cases:
        ev, res = cv.straus_events(logs, ks)
        assert what in ev, (cv.name, label, ev)
        want = sum(((s or 0) * kk for s, kk in zip(logs, ks))) % r
        assert res == want
        out.append((logs, ks, label))
    return out


def check_straus(lib, cv):
    F = cv.F
    G = O.ec_mul(F, cv.ocs.BP1, random.Random(9).randrange(1, cv.r))
    cases = straus_cases(cv)
    for op, npts in ((MSM2, 2), (MSM3, 3)):
        sel = [c for c in cases if len(c[0]) == npts]
        ps, ks, want = [], [], []
        for logs, sc, label in sel:
            pts = [None if s is None else O.ec_mul(F, G, s) for s in logs]
            ps.append(b"".join(jac(cv, pt, 1) for pt in pts))
            ks.append(sc)
            acc = None
            for pt, kk in zip(pts, sc):
                acc = O.ec_add(F, acc, O.ec_mul(F, pt, kk))
            want.append(cv.ocs.g1_compress(acc))
        got = run_g1(lib, cv, op, ps, ks=ks)
        for (logs, sc, label), g, w in zip(sel, got, want):
            assert g == w, (cv.name, label)
    # phi(P) given as its affine point (beta x, y), checked against lam P
    assert cv.phi(G) == O.ec_mul(F, G, cv.lam)


def check_refusals(lib, cv):
    one = np.zeros(64 * 3 * 3, dtype=np.uint8)
    out = np.zeros(64, dtype=np.uint8)
    for op in (-1, 5, 0x100):
        assert lib.bbs_selftest_g1(cv.suite.curve_id, 0, op, 1, P.ptr(one), P.ptr(one), P.ptr(one), P.ptr(out)) != 0
    assert lib.bbs_selftest_g1(cv.suite.curve_id, 0, ADD, 1, P.ptr(one), None, None, P.ptr(out)) != 0
    assert lib.bbs_selftest_g1(cv.suite.curve_id, 0, MSM2, 1, P.ptr(one), None, None, P.ptr(out)) != 0
    assert lib.bbs_selftest_g1(99, 0, DBL, 1, P.ptr(one), None, None, P.ptr(out)) != 0


# ---- proofs with related points -----------------------------------------------------------------------------------------
PROOF_KINDS = ["plain", "Abar=D", "Abar=D, e~=r1~", "T1=O", "r1-negated"]


def related_proofs(ocs, curve_name, L, dis, kinds=PROOF_KINDS, header=b"g1x", ph=b"ph-g1x"):
    """(signature bytes, messages, random scalars, oracle proof) per kind.  With r1 = sk + e, Abar = A r1 r2 = B r2 = D;
    with e~ = r1~ as well, proof gen's T1 = Abar e~ + D r1~ is a Straus product of equal points and scalars; with
    r1 = -(sk + e), Abar = -D and T1 = O; negating r1 negates Abar and Bbar."""
    r = ocs.r
    sk, pk = P.keypair(ocs, 1)
    U = L - len(set(dis))
    out = []
    for i, kind in enumerate(kinds):
        msgs = [P.rng_bytes(f"g1x{curve_name}{L}{i}.{j}", 32) for j in range(L)]
        a, e = O.sign(ocs, sk, msgs, header)
        rs = O.seeded_random_scalars(ocs, f"g1x{i}".encode(), b"rs-dst", 5 + U)
        if kind in ("Abar=D", "Abar=D, e~=r1~"):
            rs[0] = (sk + e) % r
        elif kind == "T1=O":
            rs[0] = (-(sk + e)) % r
        elif kind == "r1-negated":
            rs[0] = (-rs[0]) % r
        if kind in ("Abar=D, e~=r1~", "T1=O"):
            rs[2] = rs[3]
        pr = O.proof_gen(ocs, pk, (a, e), header, ph, msgs, dis, random_scalars=rs)
        if kind.startswith("Abar=D"):
            assert pr.a_bar == pr.d
        if kind == "T1=O":
            assert pr.a_bar == O.ec_neg(ocs.F1, pr.d)
        out.append((O.signature_to_bytes(ocs, (a, e)), msgs, rs, pr))
    return sk, pk, out


def check_related_proofs(lib_path, curve_name, L, dis, rlc=False):
    suite, ocs = P.SUITES[curve_name]
    header, ph = b"g1x", b"ph-g1x"
    sk, pk, items = related_proofs(ocs, curve_name, L, dis)
    ctx, _ = P.make_ctx(lib_path, suite, ocs, pk, header, L)
    got, st = ctx.proof_gen_batch([it[0] for it in items], [it[1] for it in items], [list(dis)] * len(items),
                                  [[ocs.scalar_le(x) for x in it[2]] for it in items], ph)
    assert st.tolist() == [A.ST_ACCEPT] * len(items)
    for (_, _, _, pr), g, kind in zip(items, got, PROOF_KINDS):
        want = A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, pr))
        assert (g.fixed, g.commitments) == (want.fixed, want.commitments), (curve_name, L, kind)
    # T1 = O: the challenge hashed the identity encoding
    pr = items[PROOF_KINDS.index("T1=O")][3]
    gens = O.create_generators_cached(ocs, L + 1, ocs.api_id)
    ms = O.msg_to_scalars(ocs, items[PROOF_KINDS.index("T1=O")][1], ocs.api_id)
    pts, dom = O.proof_verify_init(ocs, pk, pr, gens, header, [ms[j] for j in dis], dis, ocs.api_id)
    assert pts[3] is None
    dm = [[it[1][j] for j in dis] for it in items]
    proofs = [A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, it[3])) for it in items]
    for it, d in zip(items, dm):
        assert O.proof_verify(ocs, pk, it[3], header, ph, d, dis, trapdoor_sk=sk)
    n = len(items)
    for split in (None, 0):                      # the default two-task G1 path, then the one-thread path
        if split is not None:
            ctx.set_g1_split(split)
        assert ctx.proof_verify_batch(proofs, ph, dm, [list(dis)] * n).tolist() == [A.ST_ACCEPT] * n, (curve_name, L, split)
        if rlc:
            st, comb = ctx.rlc_proof_verify_batch(proofs, ph, dm, [list(dis)] * n, seed=b"\x07" * 32)
            assert st.tolist() == [A.ST_ACCEPT] * n and comb == A.ST_ACCEPT, (curve_name, L, split)
    ctx.close()


PROOF_SHAPES = [(0, []), (3, [1]), (4, [0, 3])]


# ---- CPU: host simulation -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve_name", CURVES)
def test_exceptional_pairs_hostsim(hs_lib, curve_name):
    check_pairs(hs_lib, curve(curve_name))


@pytest.mark.parametrize("curve_name", CURVES)
def test_straus_collisions_hostsim(hs_lib, curve_name):
    check_straus(hs_lib, curve(curve_name))


@pytest.mark.parametrize("curve_name", CURVES)
def test_unknown_ops_refused_hostsim(hs_lib, curve_name):
    check_refusals(hs_lib, curve(curve_name))


@pytest.mark.parametrize("curve_name", CURVES)
@pytest.mark.parametrize("L,dis", PROOF_SHAPES)
def test_related_point_proofs_hostsim(curve_name, L, dis):
    check_related_proofs(hostsim.build(), curve_name, L, dis)


# ---- GPU: the sm_100a kernels -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("curve_name", CURVES)
def test_exceptional_pairs_gpu(curve_name):
    check_pairs(_native.load(), curve(curve_name))


@pytest.mark.gpu
@pytest.mark.parametrize("curve_name", CURVES)
def test_straus_collisions_gpu(curve_name):
    check_straus(_native.load(), curve(curve_name))


@pytest.mark.gpu
@pytest.mark.parametrize("curve_name", CURVES)
def test_unknown_ops_refused_gpu(curve_name):
    check_refusals(_native.load(), curve(curve_name))


@pytest.mark.gpu
@pytest.mark.parametrize("curve_name", CURVES)
@pytest.mark.parametrize("L,dis", PROOF_SHAPES)
def test_related_point_proofs_gpu(curve_name, L, dis):
    check_related_proofs(None, curve_name, L, dis, rlc=True)


# ---- GPU: bucket MSMs on structured batches -----------------------------------------------------------------------------
RLC_L = 2
RLC_SEED = hashlib.sha256(b"test_g1_exceptional rlc").digest()
# one past the first upload chunk of bbs_rlc_partial on a 148-SM B200: two waves of 4 x 148 blocks of 128 items
PAST_CHUNK = 2 * 4 * 148 * 128 + 4097


class RlcBatch:
    """n signatures (A_i, e_i) with A_i from a small set of multiples of one point G and B_i from a few message classes;
    the expected partial sums need one scalar multiplication per distinct point"""

    def __init__(self, cv, n, seed, index_base, solve_s1=False, zero_column=False):
        self.cv, self.n, self.index_base = cv, n, index_base
        ocs, F, r = cv.ocs, cv.F, cv.r
        rnd = random.Random(seed)
        self.sk, self.pk = P.keypair(ocs, 1)
        self.gens = O.create_generators_cached(ocs, RLC_L + 1, ocs.api_id)
        self.dom = O.calculate_domain(ocs, self.pk, self.gens[0], self.gens[1:], b"rlcx", ocs.api_id)
        self.G = O.ec_mul(F, ocs.BP1, rnd.randrange(1, r))
        logs = [1, r - 1, 2, cv.lam, rnd.randrange(1, r)]          # P, -P, 2P, phi(P), Q
        self.coeff = [P.rlc_coeff(RLC_SEED, index_base + i) for i in range(n)]
        # runs of one point (buckets holding many copies of it, and of its negation) with a random tail
        self.cls = [(i // 7) % 5 if i % 3 else rnd.randrange(5) for i in range(n)]
        self.alog = [logs[c] for c in self.cls]
        self.e = [rnd.randrange(r) for _ in range(n)]
        classes = [[rnd.randrange(r) for _ in range(RLC_L)] for _ in range(3)]
        self.rows = [classes[i % 3 if i % 5 else 0] for i in range(n)]
        if solve_s1 and n > 1:                  # sum r_i A_i = O
            t = sum(c * a for c, a in zip(self.coeff[:-1], self.alog[:-1])) % r
            self.alog[-1] = (-t * pow(self.coeff[-1], -1, r)) % r
        if zero_column and n > 1:               # sum_i r_i m_i0 = 0: a zero scalar reaches the fixed-base term
            last = list(self.rows[-1])
            t = sum(c * m[0] for c, m in zip(self.coeff[:-1], self.rows[:-1])) % r
            last[0] = (-t * pow(self.coeff[-1], -1, r)) % r
            self.rows[-1] = last

    def signatures(self):
        cv = self.cv
        enc = {}
        out = []
        for a, e in zip(self.alog, self.e):
            if a not in enc:
                enc[a] = cv.ocs.g1_compress(O.ec_mul(cv.F, self.G, a))
            out.append(enc[a] + e.to_bytes(32, "little"))
        return b"".join(out)

    def expected(self):
        cv, r, F = self.cv, self.cv.r, self.cv.F
        s1, s2 = {}, {}
        for c, a, e in zip(self.coeff, self.alog, self.e):
            s1[a] = (s1.get(a, 0) + c) % r
            s2[a] = (s2.get(a, 0) + c * e) % r
        S1 = sum((a * k for a, k in s1.items())) % r
        S2a = sum((a * k for a, k in s2.items())) % r
        bsum = {}
        for c, row in zip(self.coeff, self.rows):
            bsum[tuple(row)] = (bsum.get(tuple(row), 0) + c) % r
        S2 = O.ec_mul(F, self.G, S2a)
        for row, k in bsum.items():
            B = O.compute_B(cv.ocs, self.gens, self.dom, list(row))
            S2 = O.ec_add(F, S2, O.ec_neg(F, O.ec_mul(F, B, k)))
        return cv.ocs.g1_compress(O.ec_mul(F, self.G, S1)) + cv.ocs.g1_compress(S2), S1 == 0

    def partial(self, ctx):
        """bbs_rlc_partial_core: the message scalars as given"""
        lib, g = ctx.lib, self.cv.suite.g1_bytes
        sigs = np.frombuffer(self.signatures(), dtype=np.uint8)
        sc = np.frombuffer(b"".join(m.to_bytes(32, "little") for row in self.rows for m in row), dtype=np.uint8)
        seed = np.frombuffer(RLC_SEED, dtype=np.uint8)
        parts = np.zeros(2 * g, dtype=np.uint8)
        st = np.full(1, 255, dtype=np.uint8)
        rc = lib.bbs_rlc_partial_core(ctx.handle, self.n, P.ptr(sigs), P.ptr(sc), RLC_L, P.ptr(seed), self.index_base,
                                      P.ptr(parts), P.ptr(st))
        assert rc == 0, lib.bbs_last_error()
        return parts.tobytes(), int(st[0])


@pytest.fixture(scope="module", params=CURVES)
def rlc_ctx(request):
    cv = curve(request.param)
    sk, pk = P.keypair(cv.ocs, 1)
    gens = O.create_generators_cached(cv.ocs, RLC_L + 1, cv.ocs.api_id)
    ctx = A.BatchContext(cv.suite, cv.ocs.g2_compress(pk), b"rlcx", generators=P.gens_bytes(cv.ocs, gens))
    yield cv, ctx
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 33, 4096, 65536, PAST_CHUNK])
def test_bucket_msm_structured_batches(rlc_ctx, n):
    cv, ctx = rlc_ctx
    base = (1 << 32) - n // 2
    variants = [RlcBatch(cv, n, f"plain{n}", base)]
    if n >= 2:
        variants.append(RlcBatch(cv, n, f"s1zero{n}", base, solve_s1=True, zero_column=True))
    expected = [v.expected() for v in variants]
    if n >= 2:
        assert expected[1][1], "S1 = O by construction"
    try:
        for windows in (0, 8, 13, 32):
            ctx.set_rlc_windows(windows)
            for v, (want, _) in zip(variants, expected):
                parts, st = v.partial(ctx)
                assert st == A.ST_ACCEPT
                assert parts[:len(want) // 2] == want[:len(want) // 2], (cv.name, n, windows, "S1")
                assert parts == want, (cv.name, n, windows, "S2")
    finally:
        ctx.set_rlc_windows(0)


@pytest.mark.gpu
@pytest.mark.parametrize("curve_name", CURVES)
@pytest.mark.parametrize("n", [64, 4096])
def test_rlc_proofs_of_one_point(curve_name, n):
    """n copies of one proof, and the same proof alternating with its r1-negated twin: every bucket holds many copies of
    one point (or of it and its negation); the combined check must hold without the per-item fallback"""
    suite, ocs = P.SUITES[curve_name]
    L, dis, header, ph = 3, [1], b"g1x", b"ph-g1x"
    sk, pk, items = related_proofs(ocs, curve_name, L, dis, kinds=["plain"], header=header, ph=ph)
    _, msgs, rs, pr = items[0]
    twin_rs = [(-rs[0]) % ocs.r] + rs[1:]
    twin = O.proof_gen(ocs, pk, O.sign(ocs, sk, msgs, header), header, ph, msgs, dis, random_scalars=twin_rs)
    assert twin.a_bar == O.ec_neg(ocs.F1, pr.a_bar) and twin.b_bar == O.ec_neg(ocs.F1, pr.b_bar)
    one = A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, pr))
    neg = A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, twin))
    ctx, _ = P.make_ctx(None, suite, ocs, pk, header, L)
    dm = [[msgs[j] for j in dis]] * n
    try:
        for windows in (0, 32):
            ctx.set_rlc_windows(windows)
            for proofs in ([one] * n, [one if i % 2 == 0 else neg for i in range(n)]):
                st, comb = ctx.rlc_proof_verify_batch(proofs, ph, dm, [dis] * n, seed=RLC_SEED)
                assert st.tolist() == [A.ST_ACCEPT] * n, (curve_name, n, windows)
                assert comb == A.ST_ACCEPT, (curve_name, n, windows)
    finally:
        ctx.close()
