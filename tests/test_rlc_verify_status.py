"""Signature verification with per-item statuses by one random linear combination (bbs_rlc_*verify_batch_status*):
statuses equal to those of the per-item calls and of the oracle, the `combined` verdict (ACCEPT exactly when the one
combined check held or no item reached it), malformed items kept out of the sums, the documented coefficients, per-item
headers, launch counts, and the Python / sharding layers."""
import hashlib

import numpy as np
import pytest

import hostsim
import parity_cases as P
from bbs_sign_b200 import _native
from bbs_sign_b200 import api as A
from oracle import bbs_oracle as O

CURVES = ["BLS12_381", "BN254"]
SEED = hashlib.sha256(b"test_rlc_verify_status").digest()


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_host_simulation_stubs_return_cuda_error():
    lib = _native.load(hostsim.build(), allow_host_simulation=True)
    one = np.zeros(96, dtype=np.uint8)
    off = np.zeros(2, dtype=np.uint64)
    st = np.zeros(1, dtype=np.uint8)
    p = P.ptr
    calls = [
        ("bbs_rlc_core_verify_batch_status", (None, 1, p(one), p(one), 1, None, p(st), p(st))),
        ("bbs_rlc_verify_batch_status", (None, 1, p(one), p(one), p(off), 1, None, p(st), p(st))),
        ("bbs_rlc_core_verify_batch_status_hdr", (None, 1, p(one), p(one), 1, p(one), p(off), None, p(st), p(st))),
        ("bbs_rlc_verify_batch_status_hdr", (None, 1, p(one), p(one), p(off), 1, p(one), p(off), None, p(st), p(st))),
    ]
    for name, args in calls:
        assert getattr(lib, name)(*args) == -2, name          # BBS_E_CUDA
        assert lib.bbs_last_error().decode()


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"the library was called ({name})")


def test_wrapper_answers_empty_batches_and_length_mismatches_without_the_library():
    ctx = object.__new__(A.BatchContext)
    ctx.suite, ctx.lib, ctx._h, ctx.L = A.BLS12_381, _NoLibrary(), None, 2
    sig = bytes(A.BLS12_381.signature_bytes)
    st, comb = ctx.rlc_verify_batch_status([sig, sig], [[b"a"], [b"a", b"b", b"c"]], seed=SEED)
    assert st.tolist() == [A.ST_ERR_MSG_GEN_LEN] * 2 and comb == A.ST_ACCEPT
    st, comb = ctx.rlc_verify_batch_status([sig], [[b"a"]], headers=[b"h"])
    assert st.tolist() == [A.ST_ERR_MSG_GEN_LEN] and comb == A.ST_ACCEPT
    st, comb = ctx.rlc_core_verify_batch_status(sig * 3, bytes(3 * 32), 1, seed=SEED)
    assert st.tolist() == [A.ST_ERR_MSG_GEN_LEN] * 3 and comb == A.ST_ACCEPT
    for fn, args in ((ctx.rlc_verify_batch_status, (b"", [])), (ctx.rlc_core_verify_batch_status, (b"", b"", 2))):
        st, comb = fn(*args)
        assert st.tolist() == [] and comb == A.ST_ACCEPT
    with pytest.raises(A.BbsError):
        ctx.rlc_verify_batch_status([sig], [])


# ---- GPU ------------------------------------------------------------------------------------------------------------
KINDS = ["ok", "msg-flip", "e^1", "A=identity", "A-neighbour", "other-key", "bad-flags", "x>=p", "off-subgroup", "e>=r",
         "m>=r", "ok"]


def _mix(curve, sk, header_of, L, tag, core, kinds=KINDS):
    """signature bytes, messages and LE32 scalar rows per item of `kinds` (kinds that do not apply to the curve, L or
    message form are left out); item i is signed under header_of(i)"""
    suite, ocs = P.SUITES[curve]
    g = suite.g1_bytes
    sk2, _ = P.keypair(ocs, 2)
    sigs, msgs, rows, used = [], [], [], []
    prev = None
    for kind in kinds:
        if (kind == "msg-flip" and not L) or (kind == "m>=r" and (not L or not core)) or (kind == "off-subgroup" and curve != "BLS12_381"):
            continue
        i = len(sigs)
        m = [P.rng_bytes(f"{tag}{i}.{j}", 32) for j in range(L)]
        s = O.signature_to_bytes(ocs, O.sign(ocs, sk2 if kind == "other-key" else sk, m, header_of(i)))
        b = bytearray(s)
        if kind == "msg-flip":
            m[L - 1] = m[L - 1] + b"!"
        sc = [ocs.scalar_le(x) for x in O.msg_to_scalars(ocs, m, ocs.api_id)]
        if kind == "e^1":
            b[g] ^= 1
        elif kind == "A=identity":
            b[:g] = ocs.g1_compress(None)
        elif kind == "A-neighbour":
            b[:g] = prev[:g]
        elif kind == "bad-flags":                 # BLS12-381: compression flag cleared; BN254: both flag bits set
            if curve == "BLS12_381":
                b[0] ^= 0x80
            else:
                b[g - 1] |= 0xC0
        elif kind == "x>=p":
            b[:g] = bytes([0x9f]) + b"\xff" * (g - 1) if curve == "BLS12_381" else b"\xff" * (g - 1) + bytes([0x3f])
        elif kind == "off-subgroup":
            b[:g] = ocs.g1_compress(P.off_subgroup_g1(ocs))
        elif kind == "e>=r":
            b[g:] = (ocs.r + 3).to_bytes(32, "little")
        elif kind == "m>=r":
            sc[0] = (ocs.r + 1).to_bytes(32, "little")
        prev = s
        sigs.append(bytes(b))
        msgs.append(m)
        rows.append(sc)
        used.append(kind)
    return sigs, msgs, rows, used


def _oracle(curve, pk, sk, header, sig, row, L):
    """the reference's result for one item: ERR_MALFORMED for undecodable input, else the verification (trapdoor form)"""
    suite, ocs = P.SUITES[curve]
    g = suite.g1_bytes
    try:
        a = ocs.g1_decompress(sig[:g])
    except ValueError:
        return A.ST_ERR_MALFORMED
    e = int.from_bytes(sig[g:], "little")
    ms = [int.from_bytes(x, "little") for x in row]
    if e >= ocs.r or any(x >= ocs.r for x in ms):
        return A.ST_ERR_MALFORMED
    gens = O.create_generators_cached(ocs, L + 1, ocs.api_id)
    return int(O.core_verify(ocs, pk, (a, e), gens, header, ms, ocs.api_id, trapdoor_sk=sk))


def _both(ctx, sigs, msgs, rows, L, core, headers=None, seed=SEED):
    """(per-item statuses, rlc statuses, combined); the rlc call runs first, on whatever the status scratch held"""
    blob = np.frombuffer(b"".join(sigs), dtype=np.uint8)
    if core:
        sc = np.frombuffer(b"".join(x for r in rows for x in r) or b"\0", dtype=np.uint8)[: len(sigs) * L * 32]
        got, comb = ctx.rlc_core_verify_batch_status(blob, sc, L, headers=headers, seed=seed)
        ref = ctx.core_verify_batch(blob, sc, L, headers=headers)
    else:
        got, comb = ctx.rlc_verify_batch_status(blob, msgs, headers=headers, seed=seed)
        ref = ctx.verify_batch(blob, msgs, headers=headers)
    return ref.tolist(), got.tolist(), comb


def _poison(ctx, n, L):
    """a per-item call over n items of the wrong message count: the context's status scratch then holds ERR_MSG_GEN_LEN
    for items [0, n), so a later call that left a status unwritten would show it"""
    st = ctx.core_verify_batch(np.zeros(n * ctx.suite.signature_bytes, np.uint8), np.zeros(n * (L + 1) * 32, np.uint8), L + 1)
    assert st.tolist() == [A.ST_ERR_MSG_GEN_LEN] * n


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
@pytest.mark.parametrize("L", [0, 1, 4, 10])
def test_statuses_match_per_item_calls_and_oracle(curve, L):
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    header = b"rvs"
    ctx, _ = P.make_ctx(None, suite, ocs, pk, header, L)
    for core in (False, True):
        sigs, msgs, rows, kinds = _mix(curve, sk, lambda i: header, L, f"st{curve}{L}", core)
        exp = [_oracle(curve, pk, sk, header, s, r, L) for s, r in zip(sigs, rows)]
        assert exp[0] == exp[-1] == 1 and exp[kinds.index("e^1")] == 0
        _poison(ctx, len(sigs), L)
        ref, got, comb = _both(ctx, sigs, msgs, rows, L, core)
        assert ref == got == exp, (core, kinds, ref, got, exp)
        assert comb == A.ST_REJECT
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_malformed_items_stay_out_of_the_combined_check(curve):
    """valid and malformed items: exact statuses, combined ACCEPT, and no per-item kernel (the launch delta of an
    all-valid batch of the same size)"""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, header = 3, b"mal"
    ctx, _ = P.make_ctx(None, suite, ocs, pk, header, L)
    kinds = ["ok", "bad-flags", "ok", "x>=p", "off-subgroup", "e>=r", "m>=r", "ok"]
    for core in (False, True):
        sigs, msgs, rows, used = _mix(curve, sk, lambda i: header, L, f"mal{curve}", core, kinds)
        exp = [1 if k == "ok" else A.ST_ERR_MALFORMED for k in used]
        assert exp == [_oracle(curve, pk, sk, header, s, r, L) for s, r in zip(sigs, rows)]
        _poison(ctx, len(sigs), L)
        ref, got, comb = _both(ctx, sigs, msgs, rows, L, core)
        assert ref == got == exp and comb == A.ST_ACCEPT
        valid = [i for i, k in enumerate(used) if k == "ok"]
        allv = [valid[i % len(valid)] for i in range(len(used))]
        deltas = []
        for items in (list(range(len(used))), allv):
            l0 = ctx.launch_count()
            st, comb = _rlc_only(ctx, [sigs[i] for i in items], [msgs[i] for i in items], [rows[i] for i in items], L, core)
            deltas.append(ctx.launch_count() - l0)
            assert comb == A.ST_ACCEPT and st == [exp[i] for i in items]
        # hashing (byte messages), prep, scan, scatter, buckets, reduction, finish, combined pairing, acceptance
        assert deltas == [8 + (0 if core else 1)] * 2
    ctx.close()


def _rlc_only(ctx, sigs, msgs, rows, L, core, headers=None, seed=SEED):
    blob = np.frombuffer(b"".join(sigs), dtype=np.uint8)
    if core:
        sc = np.frombuffer(b"".join(x for r in rows for x in r) or b"\0", dtype=np.uint8)[: len(sigs) * L * 32]
        st, comb = ctx.rlc_core_verify_batch_status(blob, sc, L, headers=headers, seed=seed)
    else:
        st, comb = ctx.rlc_verify_batch_status(blob, msgs, headers=headers, seed=seed)
    return st.tolist(), comb


def _raw(ctx, n, sigs, sc, n_msgs, combined=True):
    """bbs_rlc_core_verify_batch_status on raw buffers: (rc, status, combined or None, launches)"""
    st = np.full(max(n, 1), 255, np.uint8)
    comb = np.full(1, 255, np.uint8)
    sd = np.frombuffer(SEED, np.uint8).copy()
    l0 = ctx.launch_count()
    rc = ctx.lib.bbs_rlc_core_verify_batch_status(ctx.handle, n, P.ptr(sigs), P.ptr(sc), n_msgs, P.ptr(sd), P.ptr(st),
                                                  P.ptr(comb) if combined else None)
    return rc, st[:n].tolist(), int(comb[0]) if combined else None, ctx.launch_count() - l0


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_no_item_reaches_the_combined_check(curve):
    """all items malformed: statuses from the prep kernel alone (one launch, plus hashing); n_msgs != L and n = 0:
    nothing is launched.  `combined` is ACCEPT in every case, and may be NULL."""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, header = 2, b"none"
    ctx, _ = P.make_ctx(None, suite, ocs, pk, header, L)
    kinds = ["bad-flags", "x>=p", "e>=r", "m>=r", "e>=r"]
    for core in (False, True):
        sigs, msgs, rows, used = _mix(curve, sk, lambda i: header, L, f"none{curve}", core, kinds)
        _poison(ctx, len(sigs), L)
        l0 = ctx.launch_count()
        st, comb = _rlc_only(ctx, sigs, msgs, rows, L, core)
        assert st == [A.ST_ERR_MALFORMED] * len(sigs) and comb == A.ST_ACCEPT
        assert ctx.launch_count() - l0 == (1 if core else 2)
    n = 4
    sigs = np.zeros(n * suite.signature_bytes, np.uint8)
    sc = np.zeros(n * (L + 1) * 32, np.uint8)
    assert _raw(ctx, n, sigs, sc, L + 1) == (0, [A.ST_ERR_MSG_GEN_LEN] * n, A.ST_ACCEPT, 0)
    assert _raw(ctx, n, sigs, sc, L + 1, combined=False) == (0, [A.ST_ERR_MSG_GEN_LEN] * n, None, 0)
    assert _raw(ctx, 0, sigs, sc, L) == (0, [], A.ST_ACCEPT, 0)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("windows", [8, 13, 32])
def test_forced_window_geometries(windows):
    curve = "BLS12_381"
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, header = 4, b"win"
    ctx, _ = P.make_ctx(None, suite, ocs, pk, header, L)
    sigs, msgs, rows, kinds = _mix(curve, sk, lambda i: header, L, "win", True)
    ref0, got0, _ = _both(ctx, sigs, msgs, rows, L, True)
    ctx.set_rlc_windows(windows)
    ref, got, comb = _both(ctx, sigs, msgs, rows, L, True)
    assert got == ref == ref0 == got0 and comb == A.ST_REJECT
    good = [i for i, s in enumerate(ref) if s != 0]               # without the items that fail at the pairing
    st, comb = _rlc_only(ctx, [sigs[i] for i in good], None, [rows[i] for i in good], L, True)
    assert st == [ref[i] for i in good] and comb == A.ST_ACCEPT, windows
    ctx.close()


@pytest.mark.gpu
def test_large_batch_over_several_prep_and_fallback_chunks():
    """300,077 items signed on the GPU (two prep chunks of 2 x 4 x 148 x 128 items on a B200; two G1 chunks in the
    fallback), with bench.py's 1/16 corruptions plus scattered malformed items: statuses equal bbs_verify_batch's, and
    without the items that fail at the pairing the combined check holds"""
    import bench
    lib = _native.load()
    n, L = 300077, 2
    ctx = A.BatchContext(A.BLS12_381, bench.IRTF_PK, header=b"", n_messages=L)
    msgs, offs, sigs, expect = bench.make_workload(ctx, lib, n, L, seed=17)
    sb = bench.SIG_BYTES
    s2 = sigs.reshape(n, sb)
    mal = np.arange(5, n, 997)
    s2[mal[0::2], 48:] = 0xff                                    # e >= r
    s2[mal[1::2], 0] &= 0x7f                                     # compression flag cleared
    expect[mal] = A.ST_ERR_MALFORMED

    def both(sig_arr):
        ref = np.full(n, 255, np.uint8)
        got = np.full(n, 255, np.uint8)
        comb = np.full(1, 255, np.uint8)
        assert lib.bbs_verify_batch(ctx.handle, n, bench.ptr(sig_arr), bench.ptr(msgs), bench.ptr(offs), L, bench.ptr(ref)) == 0
        sd = np.frombuffer(SEED, np.uint8).copy()
        assert lib.bbs_rlc_verify_batch_status(ctx.handle, n, bench.ptr(sig_arr), bench.ptr(msgs), bench.ptr(offs), L,
                                               bench.ptr(sd), bench.ptr(got), bench.ptr(comb)) == 0
        return ref, got, int(comb[0])

    ref, got, comb = both(sigs)
    assert np.array_equal(ref, expect) and np.array_equal(got, expect) and comb == A.ST_REJECT
    fixed = s2.copy()
    fail = np.where(expect == 0)[0]
    fixed[fail] = s2[fail - 1]                                   # replace the failing items with their valid neighbours...
    m2 = msgs.reshape(n, L * bench.MSG_BYTES)
    m2[fail] = m2[fail - 1]                                      # ...and their messages
    exp2 = expect.copy()
    exp2[fail] = expect[fail - 1]
    ref, got, comb = both(np.ascontiguousarray(fixed.reshape(-1)))
    assert np.array_equal(ref, exp2) and np.array_equal(got, exp2) and comb == A.ST_ACCEPT
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_coefficients_are_the_documented_ones(curve):
    """Two valid signatures whose first message scalars are shifted by +r_1 and -r_0 (r_i = the documented coefficient of
    position i under SEED) fail one by one, but cancel in the combined check under THAT seed -- the documented caveat of a
    predictable seed -- and only under it."""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, header = 2, b"coef"
    ctx, _ = P.make_ctx(None, suite, ocs, pk, header, L)
    sigs, msgs, rows, _ = _mix(curve, sk, lambda i: header, L, f"coef{curve}", True, ["ok", "ok"])
    c = [P.rlc_coeff(SEED, 0), P.rlc_coeff(SEED, 1)]
    for k, delta in ((0, c[1]), (1, -c[0])):
        rows[k][0] = ((int.from_bytes(rows[k][0], "little") + delta) % ocs.r).to_bytes(32, "little")
    st, comb = _rlc_only(ctx, sigs, None, rows, L, True, seed=SEED)
    assert st == [1, 1] and comb == A.ST_ACCEPT
    for other in (None, hashlib.sha256(b"another seed").digest()):
        ref, got, comb = _both(ctx, sigs, None, rows, L, True, seed=other)
        assert ref == got == [0, 0] and comb == A.ST_REJECT
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_per_item_headers(curve):
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, hdr0 = 3, b"ctx-header"
    gens = O.create_generators_cached(ocs, L + 1, ocs.api_id)
    ctx = A.BatchContext(suite, ocs.g2_compress(pk), hdr0, generators=P.gens_bytes(ocs, gens), per_item_headers=True)
    hdrs = [b"", b"short", P.rng_bytes("long", 100)]
    for core in (False, True):
        # every item carries the context's header: the shared-header calls' statuses
        sigs, msgs, rows, kinds = _mix(curve, sk, lambda i: hdr0, L, f"hu{curve}", core)
        n = len(sigs)
        ref, got, comb = _both(ctx, sigs, msgs, rows, L, core, headers=[hdr0] * n)
        shared, _, _ = _both(ctx, sigs, msgs, rows, L, core)
        assert ref == got == shared and comb == A.ST_REJECT
        # mixed headers with the mix: the per-item _hdr call and the oracle (fallback path)
        hof = lambda i: hdrs[i % 3]                              # noqa: E731
        sigs, msgs, rows, kinds = _mix(curve, sk, hof, L, f"hm{curve}", core, KINDS + ["ok"])
        n = len(sigs)
        exp = [_oracle(curve, pk, sk, hof(i), sigs[i], rows[i], L) for i in range(n)]
        _poison(ctx, n, L)
        ref, got, comb = _both(ctx, sigs, msgs, rows, L, core, headers=[hof(i) for i in range(n)])
        assert ref == got == exp and comb == A.ST_REJECT, (kinds, ref, got, exp)
        # without the items that fail at the pairing: the accept path
        keep = [i for i in range(n) if exp[i] != 0]
        _poison(ctx, len(keep), L)
        st, comb = _rlc_only(ctx, [sigs[i] for i in keep], [msgs[i] for i in keep], [rows[i] for i in keep], L, core,
                             headers=[hof(i) for i in keep])
        assert st == [exp[i] for i in keep] and comb == A.ST_ACCEPT
        # two valid items with their headers swapped
        ok = [i for i in keep if exp[i] == 1]
        ok = [ok[0], next(i for i in ok if hof(i) != hof(ok[0]))]
        ref, got, comb = _both(ctx, [sigs[i] for i in ok], [msgs[i] for i in ok], [rows[i] for i in ok], L, core,
                               headers=[hof(ok[1]), hof(ok[0])])
        assert ref == got == [0, 0] and comb == A.ST_REJECT
    # BBS_E_ARG: a context without the flag, decreasing offsets
    plain, _ = P.make_ctx(None, suite, ocs, pk, hdr0, L)
    sigs, msgs, rows, _ = _mix(curve, sk, lambda i: hdr0, L, f"ha{curve}", True, ["ok", "ok"])
    blob = np.frombuffer(b"".join(sigs), np.uint8)
    sc = np.frombuffer(b"".join(x for r in rows for x in r), np.uint8)
    hb = np.frombuffer(b"abcd", np.uint8)
    st = np.zeros(2, np.uint8)
    for c, hoff in ((plain, np.array([0, 2, 4], np.uint64)), (ctx, np.array([0, 3, 2], np.uint64))):
        for name in ("bbs_rlc_core_verify_batch_status_hdr",):
            rc = getattr(c.lib, name)(c.handle, 2, P.ptr(blob), P.ptr(sc), L, P.ptr(hb), P.ptr(hoff), None, P.ptr(st), None)
            assert rc == -1, name
        flat, offs = A._pack_ragged([m for ms in msgs for m in ms])
        rc = c.lib.bbs_rlc_verify_batch_status_hdr(c.handle, 2, P.ptr(blob), P.ptr(flat), P.ptr(offs), L, P.ptr(hb),
                                                   P.ptr(hoff), None, P.ptr(st), None)
        assert rc == -1
    plain.close()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_per_item_headers_at_the_largest_l(curve):
    """L = 256 (BBS_MAX_MESSAGES) on a small-table per-item-header context: the finish kernel's Fr sums fill every row"""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L = 256
    ctx = A.BatchContext(suite, ocs.g2_compress(pk), b"big", n_messages=L, small_tables=True, per_item_headers=True)
    n = 5
    hdrs = [b"", b"a", P.rng_bytes("big", 90), b"big", b"b"]
    msgs = [[P.rng_bytes(f"L256.{i}.{j}", 8) for j in range(L)] for i in range(n)]
    sigs, _, st = ctx.sign_batch(sk.to_bytes(32, "little"), msgs, headers=hdrs)
    assert st.tolist() == [1] * n
    sigs = sigs.reshape(-1)
    got, comb = ctx.rlc_verify_batch_status(sigs, msgs, headers=hdrs, seed=SEED)
    assert got.tolist() == [1] * n and comb == A.ST_ACCEPT
    bad = sigs.copy().reshape(n, -1)
    bad[2, suite.g1_bytes] ^= 1
    got, comb = ctx.rlc_verify_batch_status(bad.reshape(-1), msgs, headers=hdrs, seed=SEED)
    assert got.tolist() == ctx.verify_batch(bad.reshape(-1), msgs, headers=hdrs).tolist() == [1, 1, 0, 1, 1]
    assert comb == A.ST_REJECT
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_identity_public_key(curve):
    suite, ocs = P.SUITES[curve]
    sk, _ = P.keypair(ocs, 1)
    L, header = 2, b"idpk"
    ctx, _ = P.make_ctx(None, suite, ocs, None, header, L)
    for core in (False, True):
        sigs, msgs, rows, _ = _mix(curve, sk, lambda i: header, L, f"idpk{curve}", core)
        _poison(ctx, len(sigs), L)
        ref, got, comb = _both(ctx, sigs, msgs, rows, L, core)
        assert ref == got and 0 in ref and comb == A.ST_REJECT
    ctx.close()


@pytest.mark.gpu
def test_sharded_matches_one_context():
    from bbs_sign_b200.sharding import ShardedVerifier
    curve = "BLS12_381"
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    L, header = 3, b"shard"
    ctx, gens = P.make_ctx(None, suite, ocs, pk, header, L)
    sigs, msgs, rows, _ = _mix(curve, sk, lambda i: header, L, "shard", False)
    one, c1 = ctx.rlc_verify_batch_status(sigs, msgs)
    sv = ShardedVerifier(suite, ocs.g2_compress(pk), header, L, devices=[0, 0])
    two, c2 = sv.rlc_verify_batch_status(sigs, msgs)
    assert two.tolist() == one.tolist() == ctx.verify_batch(np.frombuffer(b"".join(sigs), np.uint8), msgs).tolist()
    assert c1 == c2 == A.ST_REJECT
    good = [i for i, s in enumerate(one.tolist()) if s != 0]
    two, c2 = sv.rlc_verify_batch_status([sigs[i] for i in good], [msgs[i] for i in good])
    assert two.tolist() == [one[i] for i in good] and c2 == A.ST_ACCEPT
    sv.close()
    ctx.close()
