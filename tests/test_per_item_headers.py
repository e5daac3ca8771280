"""Per-item headers and presentation headers (the bbs_*_hdr calls of include/bbs_b200.h): every item's result is the
reference's for its own header / ph.  The unmarked tests run the host simulation of the CUDA sources (tests/hostsim.py);
the `gpu` tests run the same cases, and batches above the chunking thresholds, on the CUDA library."""
import numpy as np
import pytest

import hostsim
import parity_cases as P
from bbs_sign_b200 import _native
from bbs_sign_b200 import api as A
from bbs_sign_b200.sharding import ShardedVerifier
from oracle import bbs_oracle as O

CURVES = ["BLS12_381", "BN254"]
HEADER_LENS = [0, 1, 55, 56, 63, 64, 65, 119, 200]     # around the SHA-256 block and padding boundaries
PH_LENS = [0, 1, 64, 300]


@pytest.fixture(scope="module")
def hs():
    path = hostsim.build()
    _native.load(path, allow_host_simulation=True)      # tests only: the product loader refuses non-CUDA builds
    return path


def ctx_for(lib_path, curve, L, header=b"", per_item=True, api_id=None, pk=None, small=None, split=None):
    suite, ocs = P.SUITES[curve]
    api_id = ocs.api_id if api_id is None else api_id
    gens = O.create_generators_cached(ocs, L + 1, api_id)
    pk = P.keypair(ocs, 1)[1] if pk is None else pk
    ctx = A.BatchContext(suite, ocs.g2_compress(pk), header, generators=P.gens_bytes(ocs, gens), api_id=api_id,
                         lib_path=lib_path, small_tables=P.SMALL_TABLES if small is None else small, per_item_headers=per_item)
    if split is not None:
        ctx.set_g1_split(split)
    return ctx, gens


def headers_of(lens, tag="h"):
    return [P.rng_bytes(f"{tag}{k}", n) for k, n in enumerate(lens)]


def sig_blob(ocs, sigs):
    return np.frombuffer(b"".join(O.signature_to_bytes(ocs, s) for s in sigs), dtype=np.uint8)


def scalar_blob(ocs, rows):
    flat = b"".join(ocs.scalar_le(x) for row in rows for x in row)
    return np.frombuffer(flat, dtype=np.uint8) if flat else np.zeros(0, np.uint8)


# ---- cases (host simulation: lib_path = the simulation; CUDA: lib_path = None) --------------------------------------
def case_uniform_equivalence(lib_path, curve, L, n=5, split=None, small=None):
    """every item carrying header h (and ph p) gives byte for byte what the calls without _hdr give on a context built
    with h (and the shared p): statuses, signatures, B points, proofs"""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    h, p = b"uniform-header", b"uniform-ph"
    ref, gens = ctx_for(lib_path, curve, L, header=h, per_item=False, split=split, small=small)
    flg, _ = ctx_for(lib_path, curve, L, header=b"something else", split=split, small=small)
    skb = sk.to_bytes(32, "little")
    msgs = [[P.rng_bytes(f"u{i}.{j}", 7 + j) for j in range(L)] for i in range(n)]
    s1, b1, st1 = ref.sign_batch(skb, msgs, want_b=True)
    s2, b2, st2 = flg.sign_batch(skb, msgs, want_b=True, headers=[h] * n)
    assert st1.tolist() == st2.tolist() == [1] * n
    assert s1.tobytes() == s2.tobytes() and b1.tobytes() == b2.tobytes()
    rows = [O.msg_to_scalars(ocs, m, ocs.api_id) for m in msgs]
    c1 = ref.core_sign_batch(skb, scalar_blob(ocs, rows), n, L, want_b=True)
    c2 = flg.core_sign_batch(skb, scalar_blob(ocs, rows), n, L, want_b=True, headers=[h] * n)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(c1, c2))
    # verify: good items and damaged ones
    blob = bytearray(s1.tobytes())
    blob[suite.signature_bytes + suite.g1_bytes] ^= 1                  # e of item 1
    if n > 3:
        blob[3 * suite.signature_bytes:3 * suite.signature_bytes + suite.g1_bytes] = b"\xff" * suite.g1_bytes   # malformed A
    sigs = np.frombuffer(bytes(blob), dtype=np.uint8)
    v1 = ref.verify_batch(sigs, msgs)
    assert v1.tolist() == flg.verify_batch(sigs, msgs, headers=[h] * n).tolist()
    assert v1[0] == 1 and v1[1] == 0
    assert ref.core_verify_batch(sigs, scalar_blob(ocs, rows), L).tolist() == \
        flg.core_verify_batch(sigs, scalar_blob(ocs, rows), L, headers=[h] * n).tolist() == v1.tolist()
    # proofs
    dis = [0] if L else []
    U = L - len(dis)
    rss = [[ocs.scalar_le(x) for x in O.seeded_random_scalars(ocs, b"u%d" % i, b"rs", 5 + U)] for i in range(n)]
    sl = [s1[i].tobytes() for i in range(n)]
    g1, gs1 = ref.proof_gen_batch(sl, msgs, [dis] * n, rss, p)
    g2, gs2 = flg.proof_gen_batch(sl, msgs, [dis] * n, rss, [p] * n, headers=[h] * n)
    assert gs1.tolist() == gs2.tolist() == [1] * n
    assert [(x.fixed, x.commitments) for x in g1] == [(x.fixed, x.commitments) for x in g2]
    proofs = list(g1)
    proofs[1] = A.ProofBytes(proofs[1].fixed[:-1] + bytes([proofs[1].fixed[-1] ^ 1]), proofs[1].commitments)
    dm = [[m[j] for j in dis] for m in msgs]
    w1 = ref.proof_verify_batch(proofs, p, dm, [dis] * n)
    assert w1.tolist()[0] == 1 and w1.tolist()[1] != 1
    assert flg.proof_verify_batch(proofs, [p] * n, dm, [dis] * n, headers=[h] * n).tolist() == w1.tolist()
    assert ref.proof_verify_batch(proofs, [p] * n, dm, [dis] * n).tolist() == w1.tolist()      # per-item ph, context header
    dsc = [[ocs.scalar_le(x) for x in O.msg_to_scalars(ocs, d, ocs.api_id)] for d in dm]
    assert flg.core_proof_verify_batch(proofs, [p] * n, dsc, [dis] * n, headers=[h] * n).tolist() == w1.tolist()
    ref.close()
    flg.close()


def case_mixed_headers(lib_path, curve, L, api_id=None, split=None, small=None):
    """one header per item over the SHA-256 boundaries: signatures byte-equal to the oracle's, verified; two items with
    their headers swapped are rejected.  api_id None: the interface calls; else core calls under that api_id."""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    skb = sk.to_bytes(32, "little")
    ctx, gens = ctx_for(lib_path, curve, L, api_id=api_id, split=split, small=small)
    hdrs = headers_of(HEADER_LENS, f"mx{L}")
    n = len(hdrs)
    if api_id is None:
        msgs = [[P.rng_bytes(f"mx{i}.{j}", 3 + 5 * j) for j in range(L)] for i in range(n)]
        sigs, bpts, st = ctx.sign_batch(skb, msgs, want_b=True, headers=hdrs)
        want = [O.sign(ocs, sk, msgs[i], hdrs[i]) for i in range(n)]
        rows = [O.msg_to_scalars(ocs, m, ocs.api_id) for m in msgs]
        aid = ocs.api_id
    else:
        rows = [[(11 * i + j + 1) % ocs.r for j in range(L)] for i in range(n)]
        sigs, bpts, st = ctx.core_sign_batch(skb, scalar_blob(ocs, rows), n, L, want_b=True, headers=hdrs)
        want = [O.core_sign(ocs, sk, gens, hdrs[i], rows[i], api_id) for i in range(n)]
        aid = api_id
    assert st.tolist() == [1] * n
    for i in range(n):
        assert sigs[i].tobytes() == O.signature_to_bytes(ocs, want[i]), (curve, L, api_id, i)
        dom = O.calculate_domain(ocs, pk, gens[0], gens[1:], hdrs[i], aid)
        assert bpts[i].tobytes() == ocs.g1_compress(O.compute_B(ocs, gens, dom, rows[i]))
    blob = sig_blob(ocs, want)
    swapped = list(hdrs)
    swapped[2], swapped[7] = swapped[7], swapped[2]
    exp_swapped = [0 if i in (2, 7) else 1 for i in range(n)]
    if api_id is None:
        assert ctx.verify_batch(blob, msgs, headers=hdrs).tolist() == [1] * n
        assert ctx.verify_batch(blob, msgs, headers=swapped).tolist() == exp_swapped
    assert ctx.core_verify_batch(blob, scalar_blob(ocs, rows), L, headers=hdrs).tolist() == [1] * n
    assert ctx.core_verify_batch(blob, scalar_blob(ocs, rows), L, headers=swapped).tolist() == exp_swapped
    # the pairing oracle (no trapdoor) on a subset agrees
    for i in (0, 7):
        assert O.core_verify(ocs, pk, want[i], gens, hdrs[i], rows[i], aid) is True
        assert O.core_verify(ocs, pk, want[i], gens, swapped[i], rows[i], aid) is (i not in (2, 7))
    ctx.close()


def case_proofs(lib_path, curve, L=3, dis=(0, 2), split=None, small=None):
    """proof_gen with a header and a ph per item (seeded scalars) byte-equal to the oracle; the proofs verify, and proofs
    with their phs swapped do not; per-item ph alone works on a context without the flag"""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    dis = list(dis)
    ctx, gens = ctx_for(lib_path, curve, L, split=split, small=small)
    hdrs = headers_of([0, 64, 65, 200], "ph-h")
    phs = headers_of(PH_LENS, "ph-p")
    n = len(phs)
    msgs = [[P.rng_bytes(f"pm{i}.{j}", 16) for j in range(L)] for i in range(n)]
    sigs = [O.sign(ocs, sk, msgs[i], hdrs[i]) for i in range(n)]
    U = L - len(set(dis))
    rss = [O.seeded_random_scalars(ocs, b"pr%d" % i, b"rs-dst", 5 + U) for i in range(n)]
    enc = [O.signature_to_bytes(ocs, s) for s in sigs]
    got, st = ctx.proof_gen_batch(enc, msgs, [dis] * n, [[ocs.scalar_le(x) for x in rs] for rs in rss], phs, headers=hdrs)
    assert st.tolist() == [1] * n
    for i in range(n):
        w = A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, O.proof_gen(ocs, pk, sigs[i], hdrs[i], phs[i], msgs[i], dis,
                                                                                  random_scalars=rss[i])))
        assert (got[i].fixed, got[i].commitments) == (w.fixed, w.commitments), (curve, i)
    dm = [[m[j] for j in sorted(set(dis))] for m in msgs]
    didx = [sorted(set(dis))] * n
    assert ctx.proof_verify_batch(got, phs, dm, didx, headers=hdrs).tolist() == [1] * n
    ph_sw = list(phs)
    ph_sw[1], ph_sw[2] = ph_sw[2], ph_sw[1]
    assert ctx.proof_verify_batch(got, ph_sw, dm, didx, headers=hdrs).tolist() == [1, 0, 0, 1]
    hd_sw = list(hdrs)
    hd_sw[0], hd_sw[3] = hd_sw[3], hd_sw[0]
    assert ctx.proof_verify_batch(got, phs, dm, didx, headers=hd_sw).tolist() == [0, 1, 1, 0]
    for i in (1, 2):   # the oracle's verdict without trapdoor
        assert O.proof_verify(ocs, pk, O.proof_gen(ocs, pk, sigs[i], hdrs[i], phs[i], msgs[i], dis, random_scalars=rss[i]),
                              hdrs[i], ph_sw[i], dm[i], didx[i]) is False
    ctx.close()
    # per-item ph with the context's header, on a context without the flag
    plain, _ = ctx_for(lib_path, curve, L, header=b"ctx-header", per_item=False, split=split, small=small)
    sigs = [O.sign(ocs, sk, msgs[i], b"ctx-header") for i in range(n)]
    enc = [O.signature_to_bytes(ocs, s) for s in sigs]
    got, st = plain.proof_gen_batch(enc, msgs, [dis] * n, [[ocs.scalar_le(x) for x in rs] for rs in rss], phs)
    assert st.tolist() == [1] * n
    for i in range(n):
        w = A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, O.proof_gen(ocs, pk, sigs[i], b"ctx-header", phs[i], msgs[i],
                                                                                  dis, random_scalars=rss[i])))
        assert (got[i].fixed, got[i].commitments) == (w.fixed, w.commitments)
    assert plain.proof_verify_batch(got, phs, dm, didx).tolist() == [1] * n
    assert plain.proof_verify_batch(got, ph_sw, dm, didx).tolist() == [1, 0, 0, 1]
    dsc = [[ocs.scalar_le(x) for x in O.msg_to_scalars(ocs, d, ocs.api_id)] for d in dm]
    assert plain.core_proof_verify_batch(got, ph_sw, dsc, didx).tolist() == [1, 0, 0, 1]
    with pytest.raises(A.BbsError):
        plain.proof_verify_batch(got, phs, dm, didx, headers=hdrs)
    plain.close()


def case_irtf_in_mixed_batch(lib_path):
    """the IRTF signature (header) and proof (header + ph) fixtures come out of mixed batches unchanged"""
    suite, ocs = P.SUITES["BLS12_381"]
    pk = O.sk_to_pk(ocs, P.IRTF_SK)
    ctx, gens = ctx_for(lib_path, "BLS12_381", 1, pk=pk)
    msgs = [[b"other"], [P.MSG], [b""]]
    hdrs = [b"", P.HEADER, P.HEADER + b"x"]
    sigs, b, st = ctx.sign_batch(P.IRTF_SK.to_bytes(32, "little"), msgs, want_b=True, headers=hdrs)
    assert st.tolist() == [1, 1, 1]
    got = sigs[1].tobytes()
    assert got[:48] + got[48:][::-1] == P.IRTF_SIG and b[1].tobytes() == P.IRTF_B
    assert ctx.verify_batch(sigs, msgs, headers=hdrs).tolist() == [1, 1, 1]
    sig = (ocs.g1_decompress(P.IRTF_SIG[:48]), int.from_bytes(P.IRTF_SIG[48:], "big"))
    pb = A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, O.proof_gen(ocs, pk, sig, P.HEADER, P.PH, [P.MSG], [0])))
    rs = [ocs.scalar_le(x) for x in O.mocked_calculate_random_scalars(ocs, 5)]
    enc = [sigs[k].tobytes() for k in range(3)]
    gen, gst = ctx.proof_gen_batch(enc, msgs, [[0]] * 3, [rs] * 3, [b"p0", P.PH, b""], headers=hdrs)
    assert gst.tolist() == [1, 1, 1]
    assert (gen[1].fixed, gen[1].commitments) == (pb.fixed, pb.commitments)
    assert ctx.proof_verify_batch(gen, [b"p0", P.PH, b""], msgs, [[0]] * 3, headers=hdrs).tolist() == [1, 1, 1]
    ctx.close()


def case_errors(lib_path, curve):
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    skb = sk.to_bytes(32, "little")
    L, n = 2, 4
    plain, _ = ctx_for(lib_path, curve, L, per_item=False)
    msgs = [[b"a%d" % i, b"b"] for i in range(n)]
    hdrs = [b"h%d" % i for i in range(n)]
    with pytest.raises(A.BbsError, match="BBS_CTX_PER_ITEM_HEADER"):
        plain.sign_batch(skb, msgs, headers=hdrs)
    with pytest.raises(A.BbsError, match="BBS_CTX_PER_ITEM_HEADER"):
        plain.verify_batch(np.zeros(n * suite.signature_bytes, np.uint8), msgs, headers=hdrs)
    plain.close()
    ctx, _ = ctx_for(lib_path, curve, L)
    sigs, _, st = ctx.sign_batch(skb, msgs, headers=hdrs)
    assert st.tolist() == [1] * n
    # decreasing offsets
    flat, offs = A._pack_ragged([m for item in msgs for m in item])
    hflat = np.frombuffer(b"".join(hdrs), dtype=np.uint8)
    hoff = np.array([0, 2, 1, 4, 8], dtype=np.uint64)
    out = np.zeros(n, np.uint8)
    rc = ctx.lib.bbs_verify_batch_hdr(ctx.handle, n, A._ptr(sigs.reshape(-1)), A._ptr(flat), A._ptr(offs), L, A._ptr(hflat),
                                      A._ptr(hoff), A._ptr(out))
    assert rc == -1 and b"offsets decrease" in ctx.lib.bbs_last_error()
    with pytest.raises(A.BbsError):
        ctx.verify_batch(sigs, msgs, headers=hdrs[:-1])                   # one header short
    # n_msgs != L per item
    sc = scalar_blob(ocs, [[5] * (L + 1)] * n)
    assert ctx.core_verify_batch(sigs, sc, L + 1, headers=hdrs).tolist() == [A.ST_ERR_MSG_GEN_LEN] * n
    assert ctx.core_sign_batch(skb, sc, n, L + 1, headers=hdrs)[2].tolist() == [A.ST_ERR_MSG_GEN_LEN] * n
    # a malformed item leaves its neighbours as they were
    bad = sigs.copy()
    bad[1, :suite.g1_bytes] = 0xff
    assert ctx.verify_batch(bad, msgs, headers=hdrs).tolist() == [1, A.ST_ERR_MALFORMED, 1, 1]
    # host-side length errors of proof_verify_batch stay aligned with the per-item phs / headers
    dis = [0]
    rss = [[ocs.scalar_le(x) for x in O.seeded_random_scalars(ocs, b"e%d" % i, b"rs", 5 + L - 1)] for i in range(n)]
    phs = [b"ph%d" % i for i in range(n)]
    enc = [sigs[i].tobytes() for i in range(n)]
    got, gst = ctx.proof_gen_batch(enc, msgs, [dis] * n, rss, phs, headers=hdrs)
    assert gst.tolist() == [1] * n
    dm = [[m[0]] for m in msgs]
    dm[1] = []                                                        # InvalidIndicesAndMessagesLength, answered on the host
    st = ctx.proof_verify_batch(got, phs, dm, [dis] * n, headers=hdrs)
    assert st.tolist() == [1, A.ST_ERR_IDX_MSG_LEN, 1, 1]
    dsc = [[ocs.scalar_le(x) for x in O.msg_to_scalars(ocs, d, ocs.api_id)] for d in dm]
    assert ctx.core_proof_verify_batch(got, phs, dsc, [dis] * n, headers=hdrs).tolist() == [1, A.ST_ERR_IDX_MSG_LEN, 1, 1]
    ctx.close()


def case_python_surfaces(lib_path, curve):
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    pkb = ocs.g2_compress(pk)
    hdrs = [b"credential-%d" % i for i in range(10)]
    msgs = [[b"m%d" % i, b"n"] for i in range(10)]
    skey = A.SecretKey(suite, sk.to_bytes(32, "little"), pkb)
    skey.pk.lib_path = lib_path
    sigs, _, st = skey.sign_batch(msgs, hdrs)
    assert st.tolist() == [1] * 10 and len(skey.pk._ctx) == 1
    for i in (0, 9):
        assert sigs[i].tobytes() == O.signature_to_bytes(ocs, O.sign(ocs, sk, msgs[i], hdrs[i]))
    key = A.PublicKey(suite, pkb, lib_path=lib_path)
    assert key.verify_batch(sigs, hdrs, msgs).tolist() == [1] * 10
    assert len(key._ctx) == 1                                         # one context for ten headers
    assert key.verify_batch(sigs, hdrs[::-1], msgs).tolist() == [0] * 10
    sh = ShardedVerifier(suite, pkb, b"", 2, [0], lib_path=lib_path, per_item_headers=True)
    flat = np.frombuffer(sigs.tobytes(), dtype=np.uint8)
    assert sh.verify_batch(flat, msgs, headers=hdrs).tolist() == key.verify_batch(sigs, hdrs, msgs).tolist()
    # proofs through PublicKey and the sharded verifier
    rss = [[ocs.scalar_le(x) for x in O.seeded_random_scalars(ocs, b"s%d" % i, b"rs", 6)] for i in range(10)]
    ctx = key.context(None, 2)
    phs = [b"nonce-%d" % i for i in range(10)]
    proofs, gst = ctx.proof_gen_batch([sigs[i].tobytes() for i in range(10)], msgs, [[0]] * 10, rss, phs, headers=hdrs)
    assert gst.tolist() == [1] * 10
    dm = [[m[0]] for m in msgs]
    want = key.proof_verify_batch(proofs, hdrs, phs, dm, [[0]] * 10)
    assert want.tolist() == [1] * 10 and len(key._ctx) == 1
    assert sh.proof_verify_batch(proofs, phs, dm, [[0]] * 10, headers=hdrs).tolist() == want.tolist()
    assert sh.proof_verify_batch(proofs, phs[::-1], dm, [[0]] * 10, headers=hdrs).tolist() == [0] * 10
    sh.close()


# ---- host simulation -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", CURVES)
@pytest.mark.parametrize("L", [0, 3])
def test_uniform_headers_match_the_shared_header_calls(hs, curve, L):
    case_uniform_equivalence(hs, curve, L)


@pytest.mark.parametrize("curve", CURVES)
@pytest.mark.parametrize("L,api_id", [(0, None), (1, None), (3, None), (1, b""), (3, b"abc")])
def test_mixed_headers_against_the_oracle(hs, curve, L, api_id):
    case_mixed_headers(hs, curve, L, api_id)


@pytest.mark.parametrize("curve", CURVES)
def test_proofs_with_per_item_header_and_ph(hs, curve):
    case_proofs(hs, curve)


def test_irtf_fixtures_in_mixed_batches(hs):
    case_irtf_in_mixed_batch(hs)


@pytest.mark.parametrize("curve", CURVES)
def test_errors(hs, curve):
    case_errors(hs, curve)


@pytest.mark.parametrize("curve", CURVES)
def test_split_path_and_small_tables_agree(hs, curve):
    """the one-thread and task-split G1 paths, and small tables, give the same bytes and verdicts"""
    case_uniform_equivalence(hs, curve, 3, n=4, split=1 << 62)
    case_uniform_equivalence(hs, curve, 3, n=4, small=True)
    case_mixed_headers(hs, curve, 1, split=1 << 62, small=True)
    case_proofs(hs, curve, split=1 << 62)
    case_proofs(hs, curve, small=True)


@pytest.mark.parametrize("curve", CURVES)
def test_public_key_and_sharded_verifier(hs, curve):
    case_python_surfaces(hs, curve)


# ---- CUDA library -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_gpu_cases(curve):
    _native.load()
    for L in (0, 3):
        case_uniform_equivalence(None, curve, L)
    for L, api_id in [(0, None), (3, None), (3, b"abc")]:
        case_mixed_headers(None, curve, L, api_id)
    case_mixed_headers(None, curve, 1, small=True)
    case_proofs(None, curve)
    case_proofs(None, curve, small=True)
    case_errors(None, curve)
    case_python_surfaces(None, curve)
    if curve == "BLS12_381":
        case_irtf_in_mixed_batch(None)


def _rand_scalars(rng, ocs, count):
    """`count` canonical LE32 scalars (top byte small enough to stay below r)"""
    s = rng.integers(0, 256, size=(count, 32), dtype=np.uint8)
    s[:, 31] &= 0x0f
    return s


@pytest.mark.gpu
def test_gpu_large_batch_with_distinct_headers():
    """300,000 BLS12-381 items at L = 10 (above the chunking threshold of the calls without _hdr), 1,024 distinct headers,
    1/16 of the items damaged by a header swap or a flipped message: statuses equal the construction, 64 items agree with
    the oracle, and a uniform header gives what the shared-header context gives"""
    _native.load()
    suite, ocs = P.SUITES["BLS12_381"]
    sk, pk = P.keypair(ocs, 3)
    skb = sk.to_bytes(32, "little")
    n, L = 300_000, 10
    rng = np.random.default_rng(7)
    distinct = headers_of([16 + (k % 97) for k in range(1024)], "big")
    hidx = rng.integers(0, 1024, size=n)
    hdrs = [distinct[k] for k in hidx]
    sc = _rand_scalars(rng, ocs, n * L)
    ctx, gens = ctx_for(None, "BLS12_381", L, pk=pk)
    sigs, _, st = ctx.core_sign_batch(skb, sc, n, L, headers=hdrs)
    assert (st == 1).all()
    exp = np.ones(n, np.uint8)
    bad = rng.choice(n, size=n // 16, replace=False)
    vh, vsc = list(hdrs), sc.reshape(n, L, 32).copy()
    for k, i in enumerate(bad):
        if k % 2 and distinct[(hidx[i] + 1) % 1024] != hdrs[i]:
            vh[i] = distinct[(hidx[i] + 1) % 1024]
        else:
            vsc[i, k % L, 0] ^= 1
        exp[i] = 0
    got = ctx.core_verify_batch(sigs, vsc.reshape(-1), L, headers=vh)
    assert np.array_equal(got, exp), np.flatnonzero(got != exp)[:10]
    for i in rng.choice(n, size=64, replace=False):
        rows = [int.from_bytes(vsc[i, j].tobytes(), "little") for j in range(L)]
        sig = (ocs.g1_decompress(sigs[i, :48].tobytes()), int.from_bytes(sigs[i, 48:].tobytes(), "little"))
        assert int(O.core_verify(ocs, pk, sig, gens, vh[i], rows, ocs.api_id, trapdoor_sk=sk)) == got[i], i
    # uniform header at the same size: what the shared-header context (chunked path) gives
    h = distinct[5]
    ref, _ = ctx_for(None, "BLS12_381", L, header=h, per_item=False, pk=pk)
    s_ref, _, st_ref = ref.core_sign_batch(skb, sc, n, L)
    s_u, _, st_u = ctx.core_sign_batch(skb, sc, n, L, headers=[h] * n)
    assert np.array_equal(s_ref, s_u) and np.array_equal(st_ref, st_u)
    s_ref[::13, 50] ^= 1
    assert np.array_equal(ref.core_verify_batch(s_ref, sc, L), ctx.core_verify_batch(s_ref, sc, L, headers=[h] * n))
    ref.close()
    ctx.close()


@pytest.mark.gpu
def test_gpu_proofs_with_per_item_header_and_ph():
    """4,096 proofs, each with its own header and ph, generated and verified on the GPU"""
    _native.load()
    suite, ocs = P.SUITES["BLS12_381"]
    sk, pk = P.keypair(ocs, 1)
    n, L, dis = 4096, 5, [1, 3]
    rng = np.random.default_rng(11)
    ctx, gens = ctx_for(None, "BLS12_381", L, pk=pk)
    hdrs = [P.rng_bytes(f"ph{i}", 8 + i % 70) for i in range(n)]
    phs = [P.rng_bytes(f"pp{i}", 32) for i in range(n)]
    sc = _rand_scalars(rng, ocs, n * L)
    sigs, _, st = ctx.core_sign_batch(sk.to_bytes(32, "little"), sc, n, L, headers=hdrs)
    assert (st == 1).all()
    rows = sc.reshape(n, L, 32)
    rand = _rand_scalars(rng, ocs, n * (5 + L - len(dis))).reshape(n, -1, 32)
    fixed = np.zeros(n * suite.proof_fixed_bytes, np.uint8)
    commit_off = np.arange(n + 1, dtype=np.uint64) * (L - len(dis))
    commit = np.zeros(int(commit_off[-1]) * 32, np.uint8)
    dis_off = np.arange(n + 1, dtype=np.uint64) * len(dis)
    idx = np.tile(np.array(dis, np.uint32), n)
    rand_off = np.arange(n + 1, dtype=np.uint64) * rand.shape[1]
    hb, hoff = A._pack_items(hdrs, n, "header")
    pb, poff = A._pack_items(phs, n, "ph")
    gst = np.zeros(n, np.uint8)
    rc = ctx.lib.bbs_core_proof_gen_batch_hdr(ctx.handle, n, A._ptr(sigs.reshape(-1)), A._ptr(sc), L, A._ptr(idx), A._ptr(dis_off),
                                              A._ptr(rand.reshape(-1)), A._ptr(rand_off), A._ptr(commit_off), A._ptr(hb),
                                              A._ptr(hoff), A._ptr(pb), A._ptr(poff), A._ptr(fixed), A._ptr(commit), A._ptr(gst))
    assert rc == 0 and (gst == 1).all()
    pf = suite.proof_fixed_bytes
    proofs = [A.ProofBytes(fixed[i * pf:(i + 1) * pf].tobytes(), commit[int(commit_off[i]) * 32:int(commit_off[i + 1]) * 32].tobytes())
              for i in range(n)]
    dsc = [[rows[i, j].tobytes() for j in dis] for i in range(n)]
    assert (ctx.core_proof_verify_batch(proofs, phs, dsc, [dis] * n, headers=hdrs) == 1).all()
    sw = list(phs)
    sw[0::2], sw[1::2] = phs[1::2], phs[0::2]
    assert (ctx.core_proof_verify_batch(proofs, sw, dsc, [dis] * n, headers=hdrs) == 0).all()
    for i in (0, 1, 4095):
        sig = (ocs.g1_decompress(sigs[i, :48].tobytes()), int.from_bytes(sigs[i, 48:].tobytes(), "little"))
        ms = [int.from_bytes(rows[i, j].tobytes(), "little") for j in range(L)]
        rs = [int.from_bytes(rand[i, k].tobytes(), "little") for k in range(rand.shape[1])]
        w = O.core_proof_gen(ocs, pk, sig, hdrs[i], gens, phs[i], ms, dis, ocs.api_id, random_scalars=rs)
        wb = A.ProofBytes.from_canonical(suite, O.proof_to_bytes(ocs, w))
        assert (proofs[i].fixed, proofs[i].commitments) == (wb.fixed, wb.commitments), i
    ctx.close()


@pytest.mark.gpu
def test_gpu_device_buffer_forms_and_profiling():
    """bbs_core_verify_batch_hdr_dev and bbs_core_proof_verify_batch_hdr_dev (with per-item headers, and with NULL headers on
    a context without the flag) give the statuses of the host-buffer _hdr calls; with profiling on, the per-item domain
    kernel is reported in slot 3 (verify, proof verify) / slot 2 (sign) and not after a call without per-item headers"""
    import ctypes as C
    import torch
    lib = _native.load()
    suite, ocs = P.SUITES["BLS12_381"]
    sk, pk = P.keypair(ocs, 1)
    skb = sk.to_bytes(32, "little")
    n, L, dis = 300, 3, [1]
    rng = np.random.default_rng(5)
    dev = torch.device("cuda", 0)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def d(a):
        a = np.ascontiguousarray(a)
        return torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a).to(dev)

    def p(t):
        return C.c_void_p(t.data_ptr())

    def times(ctx):
        ms = (C.c_float * 4)()
        assert lib.bbs_ctx_kernel_times(ctx.handle, ms, 4) == 0
        return list(ms)

    ctx, gens = ctx_for(None, "BLS12_381", L, pk=pk)
    hdrs = [P.rng_bytes(f"dv{i}", i % 90) for i in range(n)]
    sc = _rand_scalars(rng, ocs, n * L)
    lib.bbs_ctx_set_profiling(ctx.handle, 1)
    sigs, _, st = ctx.core_sign_batch(skb, sc, n, L, headers=hdrs)
    assert (st == 1).all()
    t = times(ctx)
    assert t[1] > 0 and t[2] > 0                                      # sign kernel, then the per-item domain kernel
    bad = sigs.copy()
    bad[::7, 60] ^= 1
    want = ctx.core_verify_batch(bad, sc, L, headers=hdrs)
    assert 0 < int(want.sum()) < n
    hb, hoff = A._pack_items(hdrs, n, "header")
    d_st = torch.zeros(n, dtype=torch.uint8, device=dev)
    d_hb, d_hoff = d(hb), d(hoff)
    assert lib.bbs_core_verify_batch_hdr_dev(ctx.handle, n, p(d(bad.reshape(-1))), p(d(sc)), L, p(d_hb), p(d_hoff), p(d_st),
                                             stream) == 0
    torch.cuda.synchronize()
    assert np.array_equal(d_st.cpu().numpy(), want)
    t = times(ctx)
    assert t[1] > 0 and t[2] > 0 and t[3] > 0                         # G1, pairing, per-item domain kernel
    # proofs: host-buffer _hdr generation, verification through the device-buffer form
    phs = [P.rng_bytes(f"dp{i}", 32) for i in range(n)]
    rss = [[r.tobytes() for r in _rand_scalars(rng, ocs, 5 + L - len(dis))] for _ in range(n)]
    msgs_sc = [[sc[i * L + j].tobytes() for j in range(L)] for i in range(n)]

    def gen_and_check(c, headers, ph_list):
        flat = np.ascontiguousarray(sc)
        fixed = np.zeros(n * suite.proof_fixed_bytes, np.uint8)
        commit_off = np.arange(n + 1, dtype=np.uint64) * (L - len(dis))
        commit = np.zeros(int(commit_off[-1]) * 32, np.uint8)
        dis_off = np.arange(n + 1, dtype=np.uint64) * len(dis)
        idx = np.tile(np.array(dis, np.uint32), n)
        rand = np.frombuffer(b"".join(b"".join(r) for r in rss), np.uint8)
        rand_off = np.arange(n + 1, dtype=np.uint64) * (5 + L - len(dis))
        s_here = c.core_sign_batch(skb, sc, n, L, headers=headers)[0] if headers is not None else c.core_sign_batch(skb, sc, n, L)[0]
        hb_, hoff_ = A._pack_items(headers, n, "header") if headers is not None else (None, None)
        pb, poff = A._pack_items(ph_list, n, "ph")
        g = np.zeros(n, np.uint8)
        assert lib.bbs_core_proof_gen_batch_hdr(c.handle, n, A._ptr(s_here.reshape(-1)), A._ptr(flat), L, A._ptr(idx), A._ptr(dis_off),
                                                A._ptr(rand), A._ptr(rand_off), A._ptr(commit_off), A._ptr(hb_), A._ptr(hoff_),
                                                A._ptr(pb), A._ptr(poff), A._ptr(fixed), A._ptr(commit), A._ptr(g)) == 0
        assert (g == 1).all()
        fixed[5 * suite.proof_fixed_bytes + 200] ^= 1                    # one damaged proof
        pf = suite.proof_fixed_bytes
        proofs = [A.ProofBytes(fixed[i * pf:(i + 1) * pf].tobytes(), commit[int(commit_off[i]) * 32:int(commit_off[i + 1]) * 32].tobytes())
                  for i in range(n)]
        dsc = [[msgs_sc[i][j] for j in dis] for i in range(n)]
        want = c.core_proof_verify_batch(proofs, ph_list, dsc, [dis] * n, headers=headers)
        assert want[5] != 1 and (np.delete(want, 5) == 1).all()
        dsc_flat = np.frombuffer(b"".join(x for row in dsc for x in row), np.uint8)
        d_st = torch.zeros(n, dtype=torch.uint8, device=dev)
        d_pb, d_poff = d(pb), d(poff)
        if headers is not None:
            d_hb_, d_hoff_ = d(hb_), d(hoff_)
            hp, ho = p(d_hb_), p(d_hoff_)
        else:
            hp = ho = None
        assert lib.bbs_core_proof_verify_batch_hdr_dev(c.handle, n, p(d(fixed)), p(d(commit)), p(d(commit_off)), p(d(idx)),
                                                       p(d(dsc_flat)), p(d(dis_off)), hp, ho, p(d_pb), p(d_poff), p(d_st),
                                                       stream) == 0
        torch.cuda.synchronize()
        assert np.array_equal(d_st.cpu().numpy(), want)
        return times(c)

    t = gen_and_check(ctx, hdrs, phs)
    assert t[1] > 0 and t[2] > 0 and t[3] > 0
    plain, _ = ctx_for(None, "BLS12_381", L, header=b"plain", per_item=False, pk=pk)
    lib.bbs_ctx_set_profiling(plain.handle, 1)
    t = gen_and_check(plain, None, phs)                                # NULL d_hdr_off: the context's header
    assert t[1] > 0 and t[2] > 0 and t[3] == 0
    plain.close()
    ctx.close()
