"""Proof verification with the pairing half by one random linear combination (bbs_rlc_*proof_verify_batch*): per-item
statuses equal to those of the per-item pairing calls and of the oracle, the `combined` verdict (ACCEPT exactly when no
proof that reaches the pairing fails it), the documented coefficients, launch counts, and the Python / sharding layers."""
import hashlib

import numpy as np
import pytest

import hostsim
import parity_cases as P
from bbs_sign_b200 import _native
from bbs_sign_b200 import api as A
from oracle import bbs_oracle as O

CURVES = ["BLS12_381", "BN254"]
SEED = hashlib.sha256(b"test_rlc_proof").digest()


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_host_simulation_stubs_return_cuda_error():
    lib = _native.load(hostsim.build(), allow_host_simulation=True)
    one = np.zeros(64, dtype=np.uint8)
    off = np.zeros(2, dtype=np.uint64)
    st = np.zeros(1, dtype=np.uint8)
    p = P.ptr
    calls = [
        ("bbs_rlc_core_proof_verify_batch", (None, 1, p(one), p(one), p(off), p(one), p(one), p(off), None, 0, None, p(st), p(st))),
        ("bbs_rlc_proof_verify_batch", (None, 1, p(one), p(one), p(off), p(one), p(one), p(off), p(off), None, 0, None, p(st), p(st))),
        ("bbs_rlc_core_proof_verify_batch_hdr", (None, 1, p(one), p(one), p(off), p(one), p(one), p(off), None, None, p(one), p(off),
                                                 None, p(st), p(st))),
        ("bbs_rlc_proof_verify_batch_hdr", (None, 1, p(one), p(one), p(off), p(one), p(one), p(off), p(off), None, None, p(one),
                                            p(off), None, p(st), p(st))),
    ]
    for name, args in calls:
        assert getattr(lib, name)(*args) == -2, name          # BBS_E_CUDA
        assert lib.bbs_last_error().decode()


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"the library was called ({name})")


@pytest.mark.parametrize("core", [False, True])
def test_wrapper_answers_length_mismatches_without_the_library(core):
    ctx = object.__new__(A.BatchContext)
    ctx.suite, ctx.lib, ctx._h = A.BLS12_381, _NoLibrary(), None
    pf = A.ProofBytes(bytes(A.BLS12_381.proof_fixed_bytes), bytes(64))
    proofs = [pf, pf]
    idxs = [[0, 1], [0, 7]]
    disclosed = [[b"x" * 32], [b"y" * 32]]                 # one message for two indexes
    fn = ctx.rlc_core_proof_verify_batch if core else ctx.rlc_proof_verify_batch
    st, combined = fn(proofs, [b"a", b"b"], disclosed, idxs, seed=SEED)
    assert st.tolist() == [A.ST_ERR_IDX_MSG_LEN, A.ST_ERR_DISCLOSED_INDEX]
    assert combined == A.ST_ACCEPT
    st, combined = fn([], b"", [], [])
    assert st.tolist() == [] and combined == A.ST_ACCEPT


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _proof(ocs, pk, sig, header, ph, msgs, dis, seed, rs0=None):
    rs = O.seeded_random_scalars(ocs, seed.encode(), b"rs-dst", 5 + len(msgs) - len(set(dis)))
    if rs0 is not None:
        rs[0] = rs0
    return O.proof_gen(ocs, pk, sig, header, ph, msgs, dis, random_scalars=rs)


def _pairing_fails(ocs, pk, p, header, ph, dm, dis, sk):
    """the proof passes every check before the pairing (challenge included) and fails the pairing (trapdoor: pk = sk BP2)"""
    try:
        ms = O.msg_to_scalars(ocs, dm, ocs.api_id)
        gens = O.create_generators_cached(ocs, len(p.commitments) + len(dis) + 1, ocs.api_id)
        pts, dom = O.proof_verify_init(ocs, pk, p, gens, header, ms, dis, ocs.api_id)
        if O.proof_challenge_calculate(ocs, pts, dom, ms, dis, ph, ocs.api_id) != p.challenge % ocs.r:
            return False
    except Exception:
        return False
    return O.ec_mul(ocs.F1, p.a_bar, sk % ocs.r) != p.b_bar


def _both(ctx, proofs, ph, dm, didx, headers=None, core_ocs=None, seed=SEED):
    """(per-item statuses, rlc statuses, combined) of the byte-message calls, or of the core_ calls with core_ocs"""
    if core_ocs is not None:
        dsc = [[core_ocs.scalar_le(x) for x in O.msg_to_scalars(core_ocs, d, core_ocs.api_id)] for d in dm]
        ref = ctx.core_proof_verify_batch(proofs, ph, dsc, didx, headers=headers)
        got, comb = ctx.rlc_core_proof_verify_batch(proofs, ph, dsc, didx, headers=headers, seed=seed)
    else:
        ref = ctx.proof_verify_batch(proofs, ph, dm, didx, headers=headers)
        got, comb = ctx.rlc_proof_verify_batch(proofs, ph, dm, didx, headers=headers, seed=seed)
    return ref.tolist(), got.tolist(), comb


KINDS = ["ok", "challenge+1", "pairing-only", "wrong-msg", "ok", "Bbar-mutated", "e_cap+1"]


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
@pytest.mark.parametrize("L,disclosed", [(0, []), (1, [0]), (1, []), (4, [0, 2]), (4, [1, 2, 3]), (8, [0, 3, 7]), (8, [])])
def test_statuses_match_per_item_calls_and_oracle(curve, L, disclosed):
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    header, ph = b"h", b"ph"
    ctx, _ = P.make_ctx(None, suite, ocs, pk, header, L)
    dis = sorted(set(disclosed))
    proofs, dmsgs, didx, exp, fails = [], [], [], [], []
    for i, kind in enumerate(KINDS):
        msgs = [P.rng_bytes(f"rp{curve}{L}{i}.{j}", 32) for j in range(L)]
        a, e = O.sign(ocs, sk, msgs, header)
        if kind == "pairing-only":
            e ^= 1
        p = _proof(ocs, pk, (a, e), header, ph, msgs, dis, f"rp{curve}{L}{i}")
        dm = [msgs[j] for j in dis]
        if kind == "challenge+1":
            p.challenge = (p.challenge + 1) % ocs.r
        elif kind == "wrong-msg" and dm:
            dm[0] = dm[0] + b"!"
        elif kind == "Bbar-mutated":
            p.b_bar = O.ec_add(ocs.F1, p.b_bar, ocs.BP1)
        elif kind == "e_cap+1":
            p.e_cap = (p.e_cap + 1) % ocs.r
        proofs.append(A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, p)))
        dmsgs.append(dm)
        didx.append(dis)
        exp.append(int(O.proof_verify(ocs, pk, p, header, ph, dm, dis, trapdoor_sk=None if i == 2 else sk)))
        fails.append(_pairing_fails(ocs, pk, p, header, ph, dm, dis, sk))
    assert fails[2] and exp[2] == 0
    for core in (None, ocs):
        ref, got, comb = _both(ctx, proofs, ph, dmsgs, didx, core_ocs=core)
        assert ref == exp and got == exp, (ref, got, exp)
        assert comb == A.ST_REJECT
        keep = [i for i in range(len(KINDS)) if not fails[i]]
        ref, got, comb = _both(ctx, [proofs[i] for i in keep], ph, [dmsgs[i] for i in keep], [didx[i] for i in keep], core_ocs=core)
        assert ref == got == [exp[i] for i in keep]
        assert comb == A.ST_ACCEPT
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_err_and_malformed_items(curve):
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, dis = 4, [0, 2]
    ctx, _ = P.make_ctx(None, suite, ocs, pk, b"", L)
    (pr, msgs), = P.make_proofs(ocs, sk, pk, b"", b"", L, dis, 1)
    pb = A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, pr))
    dm = [msgs[0], msgs[2]]
    zero = A.ProofBytes(bytes(suite.g1_bytes * 3 + 128), bytes(64))
    forged = A.ProofBytes(ocs.g1_compress(None) * 3 + bytes(128), bytes(64))
    p0 = O.Proof(None, None, None, 0, 0, 0, [0, 0], 0)
    forged_want = int(O.proof_verify(ocs, pk, p0, b"", b"", dm, [0, 2]))
    proofs = [pb, pb, pb, pb, pb, zero, forged]
    m = [dm, dm, [msgs[0]], dm + [b"x"], [msgs[0], msgs[0]], dm, dm]
    idx = [[0, 2], [0, 9], [0, 2], [0, 2, 3], [0, 0], [0, 2], [0, 2]]
    want = [1, A.ST_ERR_DISCLOSED_INDEX, A.ST_ERR_IDX_MSG_LEN, A.ST_ERR_MSG_GEN_LEN, A.ST_ERR_MALFORMED, None, forged_want]
    ref, got, comb = _both(ctx, proofs, b"", m, idx)
    assert got == ref
    assert [g for g, w in zip(got, want) if w is not None] == [w for w in want if w is not None]
    assert comb == A.ST_ACCEPT
    ctx.close()


@pytest.mark.gpu
def test_golden_l32_fixture():
    import os
    fx = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "proofs_bls_L32_R16.npz"))
    ctx = A.BatchContext(A.BLS12_381, bytes(fx["pk"]), header=b"", n_messages=32)
    n = fx["fixed"].shape[0]
    proofs = [A.ProofBytes(bytes(fx["fixed"][i]), bytes(fx["commitments"][i])) for i in range(n)]
    dis = [int(x) for x in fx["disclosed_idx"]]
    msgs = [[bytes(fx["disclosed_msgs"][i][32 * k: 32 * k + 32]) for k in range(len(dis))] for i in range(n)]
    st, comb = ctx.rlc_proof_verify_batch(proofs, b"", msgs, [dis] * n)
    assert st.tolist() == fx["expect"].tolist() == ctx.proof_verify_batch(proofs, b"", msgs, [dis] * n).tolist()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_identity_points(curve):
    """identity Abar alone (fails only at the pairing), identity Abar and Bbar (accepted, as by the reference), and a
    context whose public key is the identity"""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, dis, header = 3, [1], b"id"
    msgs = [[P.rng_bytes(f"id{curve}{i}.{j}", 32) for j in range(L)] for i in range(3)]
    for key_sk, key_pk in ((sk, pk), (0, None)):
        ctx, _ = P.make_ctx(None, suite, ocs, key_pk, header, L)
        ps = []
        a0, e0 = O.sign(ocs, sk, msgs[0], header)
        ps.append(_proof(ocs, key_pk, (a0, e0), header, b"", msgs[0], dis, "id0"))               # valid under pk only
        ps.append(_proof(ocs, key_pk, (None, e0), header, b"", msgs[1], dis, "id1"))             # Abar = identity
        ps.append(_proof(ocs, key_pk, (a0, e0), header, b"", msgs[2], dis, "id2", rs0=0))        # Abar = Bbar = identity
        proofs = [A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, p)) for p in ps]
        dm = [[m[j] for j in dis] for m in msgs]
        exp = [int(O.proof_verify(ocs, key_pk, p, header, b"", d, dis, trapdoor_sk=key_sk)) for p, d in zip(ps, dm)]
        assert ps[1].a_bar is None and ps[2].a_bar is None and ps[2].b_bar is None and exp[2] == 1
        fails = [_pairing_fails(ocs, key_pk, p, header, b"", d, dis, key_sk) for p, d in zip(ps, dm)]
        assert fails[1]
        ref, got, comb = _both(ctx, proofs, b"", dm, [dis] * 3)
        assert ref == got == exp
        assert comb == A.ST_REJECT
        keep = [i for i in range(3) if not fails[i]]
        ref, got, comb = _both(ctx, [proofs[i] for i in keep], b"", [dm[i] for i in keep], [dis] * len(keep))
        assert ref == got == [exp[i] for i in keep]
        assert comb == A.ST_ACCEPT
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_per_item_ph_and_headers(curve):
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, dis, hdr0 = 3, [0, 2], b"ctx-header"
    gens = O.create_generators_cached(ocs, L + 1, ocs.api_id)
    ctx = A.BatchContext(suite, ocs.g2_compress(pk), hdr0, generators=P.gens_bytes(ocs, gens), per_item_headers=True)
    n = 5
    headers = [hdr0, b"", b"other", b"x" * 70, hdr0]
    phs = [b"nonce-%d" % i for i in range(n)]
    for hdrs in (None, headers):
        proofs, dm, exp, fails = [], [], [], []
        for i in range(n):
            h = hdr0 if hdrs is None else hdrs[i]
            msgs = [P.rng_bytes(f"ph{curve}{i}.{j}", 32) for j in range(L)]
            a, e = O.sign(ocs, sk, msgs, h)
            p = _proof(ocs, pk, (a, e ^ (i == 3)), h, phs[i], msgs, dis, f"ph{i}")
            proofs.append(A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, p)))
            dm.append([msgs[j] for j in dis])
            exp.append(int(O.proof_verify(ocs, pk, p, h, phs[i], dm[-1], dis, trapdoor_sk=sk)))
            fails.append(_pairing_fails(ocs, pk, p, h, phs[i], dm[-1], dis, sk))
        assert exp == [1, 1, 1, 0, 1] and fails[3]
        for core in (None, ocs):
            ref, got, comb = _both(ctx, proofs, phs, dm, [dis] * n, headers=hdrs, core_ocs=core)
            assert ref == got == exp and comb == A.ST_REJECT
            k = [0, 1, 2, 4]
            ref, got, comb = _both(ctx, [proofs[i] for i in k], [phs[i] for i in k], [dm[i] for i in k], [dis] * 4,
                                   headers=None if hdrs is None else [hdrs[i] for i in k], core_ocs=core)
            assert ref == got == [1, 1, 1, 1] and comb == A.ST_ACCEPT
        # swapped phs fail at the challenge: statuses exact, combined ACCEPT
        ref, got, comb = _both(ctx, proofs[:2], phs[1::-1], dm[:2], [dis] * 2, headers=None if hdrs is None else hdrs[:2])
        assert ref == got == [0, 0] and comb == A.ST_ACCEPT
    ctx.close()


# ---- device-made batches (bench.make_proof_workload: every 16th proof corrupted, failing at the challenge) -----------
@pytest.fixture(scope="module")
def workload():
    import bench
    lib = _native.load()
    ctx = A.BatchContext(A.BLS12_381, bench.IRTF_PK, header=b"", n_messages=4)
    w = bench.make_proof_workload(ctx, lib, 4096, 5, L=4, R=2)
    yield ctx, lib, w
    ctx.close()


def _raw(lib, ctx, w, n, fixed=None, rlc=True, seed=SEED, commit=None):
    """the first n proofs of the workload through bbs_[rlc_]proof_verify_batch: (status, combined, launches)"""
    import bench
    ptr = bench.ptr
    fixed = w["fixed"] if fixed is None else fixed
    commit = w["commit"] if commit is None else commit
    st = np.full(max(n, 1), 255, dtype=np.uint8)
    comb = np.full(1, 255, dtype=np.uint8)
    l0 = ctx.launch_count()
    args = (ctx.handle, n, ptr(fixed), ptr(commit), ptr(w["commit_off"]), ptr(w["idx"]), ptr(w["dmsg"]), ptr(w["moff"]),
            ptr(w["dis_off"]), None, 0)
    if rlc:
        sd = None if seed is None else np.frombuffer(seed, np.uint8).copy()
        rc = lib.bbs_rlc_proof_verify_batch(*args, None if sd is None else ptr(sd), ptr(st), ptr(comb))
    else:
        rc = lib.bbs_proof_verify_batch(*args, ptr(st))
    assert rc == 0, lib.bbs_last_error().decode()
    return st[:n], int(comb[0]), ctx.launch_count() - l0


def _pairing_only(ctx, lib, w):
    """copies of the workload's proofs and commitments in which proof 2048 is made from a signature with e flipped in bit 0:
    it fails only at its pairing.  (fixed, commit, expect)"""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import bench_rlc_proof as T
    n = len(w["expect"])
    return T.pairing_only_variant(ctx, lib, w, every=n)


def _dead(w):
    """the workload's proofs with every challenge wrong (bit 0 of its second byte: the workload's own corruptions flip the
    first byte, and flipping that back would repair them)"""
    dead = w["fixed"].copy().reshape(len(w["expect"]), -1)
    dead[:, 241] ^= 1
    return dead.reshape(-1)


def _poison(lib, ctx, w, n):
    """a per-item call in which every proof fails its challenge: the context's status scratch then holds REJECT for items
    [0, n), so a later call that left a status unwritten would show it"""
    assert _raw(lib, ctx, w, n, fixed=_dead(w), rlc=False)[0].tolist() == [0] * n


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 129, 4096])
def test_batch_sizes(workload, n):
    ctx, lib, w = workload
    ref, _, _ = _raw(lib, ctx, w, n, rlc=False)
    _poison(lib, ctx, w, n)
    st, comb, _ = _raw(lib, ctx, w, n)
    assert st.tolist() == ref.tolist() == w["expect"][:n].tolist()
    assert comb == A.ST_ACCEPT


@pytest.mark.gpu
def test_pairing_only_failure_takes_the_fallback(workload):
    ctx, lib, w = workload
    fixed, commit, expect = _pairing_only(ctx, lib, w)  # item 2048 fails only at its pairing
    assert expect[2048] == 0
    for n in (2049, 4096):
        assert _raw(lib, ctx, w, n)[0][2048] == A.ST_ACCEPT      # the original proof 2048 is valid
        st, comb, _ = _raw(lib, ctx, w, n, fixed=fixed, commit=commit)
        ref, _, _ = _raw(lib, ctx, w, n, fixed=fixed, commit=commit, rlc=False)
        assert st.tolist() == ref.tolist() == expect[:n].tolist()
        assert comb == A.ST_REJECT
    _poison(lib, ctx, w, 2048)
    st, comb, _ = _raw(lib, ctx, w, 2048, fixed=fixed, commit=commit)      # the bad proof is not in the call
    assert comb == A.ST_ACCEPT and st.tolist() == expect[:2048].tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("windows", [0, 8, 9, 13, 16, 32])
def test_forced_window_geometries(workload, windows):
    """a wrong MSM sum shows up as combined == REJECT (the fallback would still keep the statuses right)"""
    ctx, lib, w = workload
    ctx.set_rlc_windows(windows)
    try:
        for n in (33, 4096):
            _poison(lib, ctx, w, n)
            st, comb, _ = _raw(lib, ctx, w, n)
            assert comb == A.ST_ACCEPT, (windows, n)
            assert st.tolist() == w["expect"][:n].tolist()
    finally:
        ctx.set_rlc_windows(0)


@pytest.mark.gpu
def test_launch_counts(workload):
    """byte messages: hashing, the two G1 kernels, prep, scan, scatter, buckets, reduction, finish, the combined pairing,
    then the acceptance kernel (fast path) or the per-item pairing (fallback); a batch that no proof survives to the
    pairing stops after the prep kernel"""
    ctx, lib, w = workload
    assert _raw(lib, ctx, w, 4096, rlc=False)[2] == 4
    assert _raw(lib, ctx, w, 4096)[2] == 11
    fixed, commit, _ = _pairing_only(ctx, lib, w)
    st, comb, launches = _raw(lib, ctx, w, 4096, fixed=fixed, commit=commit)
    assert comb == A.ST_REJECT and launches == 11
    st, comb, launches = _raw(lib, ctx, w, 64, fixed=_dead(w))
    assert st.tolist() == [0] * 64 and comb == A.ST_ACCEPT and launches == 4
    assert _raw(lib, ctx, w, 0)[2] == 0


@pytest.mark.gpu
def test_sharded_matches_one_context(workload):
    import bench
    from bbs_sign_b200.sharding import ShardedVerifier
    ctx, lib, w = workload
    n, R, pf = 300, 2, A.BLS12_381.proof_fixed_bytes
    fixed, commit, expect = _pairing_only(ctx, lib, w)
    for fx, cm, want_comb in ((w["fixed"], w["commit"], A.ST_ACCEPT), (fixed, commit, A.ST_REJECT)):
        m = 4096 if want_comb == A.ST_REJECT else n
        proofs = [A.ProofBytes(bytes(fx[i * pf:(i + 1) * pf]), bytes(cm[i * 64:(i + 1) * 64])) for i in range(m)]
        dm = [[bytes(w["dmsg"][(i * R + k) * 32:(i * R + k + 1) * 32]) for k in range(R)] for i in range(m)]
        didx = [[0, 2]] * m
        one, c1 = ctx.rlc_proof_verify_batch(proofs, b"", dm, didx)
        sv = ShardedVerifier(A.BLS12_381, bench.IRTF_PK, b"", 4, devices=[0, 0])
        two, c2 = sv.rlc_proof_verify_batch(proofs, b"", dm, didx)
        sv.close()
        assert two.tolist() == one.tolist() == ctx.proof_verify_batch(proofs, b"", dm, didx).tolist()
        assert one.tolist() == (expect[:m] if want_comb == A.ST_REJECT else w["expect"][:m]).tolist()
        assert c1 == c2 == want_comb


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_coefficients_are_the_documented_ones(curve):
    """Two proofs of forged signatures A_k = (B_k + X_k) / (sk + e_k) fail their pairings with Bbar_k - sk Abar_k =
    -s_k X_k (s_k = r0_k r1_k, the prover's random scalars).  With X_2 = -(c_1 s_1 / (c_2 s_2)) X_1 for the coefficients c_k
    of a chosen seed, the two failures cancel in the combined check under THAT seed -- the documented caveat of a
    predictable seed -- and only under it."""
    suite, ocs = P.SUITES[curve]
    F, r = ocs.F1, ocs.r
    sk, pk = P.keypair(ocs, 1)
    L, dis, header = 2, [0], b"coef"
    gens = O.create_generators_cached(ocs, L + 1, ocs.api_id)
    ctx, _ = P.make_ctx(None, suite, ocs, pk, header, L)
    domain = O.calculate_domain(ocs, pk, gens[0], gens[1:], header, ocs.api_id)
    c = [P.rlc_coeff(SEED, 0), P.rlc_coeff(SEED, 1)]
    X1 = O.ec_mul(F, ocs.BP1, 12345)
    proofs, dm = [], []
    rss = [O.seeded_random_scalars(ocs, b"coef%d" % k, b"rs-dst", 5 + L - 1) for k in range(2)]
    s = [rs[0] * rs[1] % r for rs in rss]
    X = [X1, O.ec_mul(F, X1, (-c[0] * s[0] * pow(c[1] * s[1], -1, r)) % r)]
    for k in range(2):
        msgs = [P.rng_bytes(f"coef{curve}{k}.{j}", 32) for j in range(L)]
        ms = O.msg_to_scalars(ocs, msgs, ocs.api_id)
        e = int.from_bytes(hashlib.sha256(b"e%d" % k).digest(), "big") % r
        B = O.compute_B(ocs, gens, domain, ms)
        Ak = O.ec_mul(F, O.ec_add(F, B, X[k]), pow((sk + e) % r, -1, r))
        p = O.core_proof_gen(ocs, pk, (Ak, e), header, gens, b"", ms, dis, ocs.api_id, random_scalars=rss[k])
        assert O.ec_add(F, p.b_bar, O.ec_neg(F, O.ec_mul(F, p.a_bar, sk))) == O.ec_neg(F, O.ec_mul(F, X[k], s[k]))
        proofs.append(A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, p)))
        dm.append([msgs[0]])
    st, comb = ctx.rlc_proof_verify_batch(proofs, b"", dm, [dis] * 2, seed=SEED)
    assert st.tolist() == [1, 1] and comb == A.ST_ACCEPT
    for other in (None, hashlib.sha256(b"another seed").digest()):
        st, comb = ctx.rlc_proof_verify_batch(proofs, b"", dm, [dis] * 2, seed=other)
        assert st.tolist() == [0, 0] and comb == A.ST_REJECT
    assert ctx.proof_verify_batch(proofs, b"", dm, [dis] * 2).tolist() == [0, 0]
    ctx.close()
