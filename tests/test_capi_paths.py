"""Every host-buffer batch entry point of the C ABI in each of its forms: plain, core_, _hdr with mixed headers, _multi and
per-item ph, for sign, verify, proof gen and proof verify, and bbs_msg_to_scalars.  For each call the outputs equal those
of the matching call in another form, the number of kernel launches it adds to bbs_ctx_launch_count is the one in PATHS,
and the context's scratch after the whole sequence has the size in MEMORY.  On the CUDA build (G1 task split on) the
launches are counted again, with the batches above the chunking thresholds, and PATHS names the bbs_ctx_kernel_times slots
that are non-zero after each call with profiling on.  The launches per step that bench.py reports come from these counts."""
import ctypes as C

import numpy as np
import pytest

import hostsim
import parity_cases as P
from bbs_sign_b200 import _native
from bbs_sign_b200 import api as A
from oracle import bbs_oracle as O
from test_per_item_headers import _rand_scalars, ctx_for, headers_of, scalar_blob

CURVES = ["BLS12_381", "BN254"]

# call: (launches on the host simulation, launches on the CUDA build, non-zero kernel_times slots on the CUDA build).
# Slots None: not checked (the call records no profiling mark).  Slot 0 is checked only where the call marks it, around
# its message hashing: a call that does not keeps an older call's slot-0 event.
PATHS = {
    "msg_to_scalars": (1, 1, None),
    "sign": (2, 2, "01"),
    "core_sign": (1, 1, "1"),
    "sign_hdr": (3, 3, "012"),
    "core_sign_hdr": (2, 2, "12"),
    "verify": (3, 4, "012"),
    "core_verify": (2, 3, "12"),
    "verify_hdr": (4, 5, "0123"),
    "core_verify_hdr": (3, 4, "123"),
    "proof_gen": (2, 2, None),
    "core_proof_gen": (1, 1, None),
    "proof_gen_ph": (2, 2, None),
    "proof_gen_hdr": (3, 3, None),
    "core_proof_gen_hdr": (2, 2, None),
    "proof_verify": (3, 4, "12"),
    "core_proof_verify": (2, 3, "12"),
    "proof_verify_ph": (3, 4, "12"),
    "core_proof_verify_ph": (2, 3, "12"),
    "proof_verify_hdr": (5, 5, "123"),
    "core_proof_verify_hdr": (4, 4, "123"),
    # CUDA build only
    "rlc_verify": (None, 8, "0123456"),
    "rlc_core_verify": (None, 7, "123456"),
    "rlc_partial": (None, 7, "012345"),
    "rlc_partial_core": (None, 6, "12345"),
    "verify_chunked": (None, 7, None),           # 262,144 items: two chunks, each hashed and G1-checked, one pairing
    "core_verify_chunked": (None, 5, None),
    "verify_hdr_large": (None, 5, "0123"),       # the _hdr calls take no chunks
    "core_verify_hdr_large": (None, 4, "123"),
    "sign_chunked": (None, 4, "1"),              # 524,288 items: two chunks, each hashed and signed
    "core_sign_chunked": (None, 2, "1"),
    "sign_hdr_large": (None, 3, "012"),
    "core_sign_hdr_large": (None, 2, "12"),
}
# (curve, L, n) -> (bbs_ctx_memory_bytes of the context, shared bytes of the issuer set) after run_small_paths
MEMORY = {
    ("BLS12_381", 3, 4): (2514145, 2015606),
    ("BN254", 3, 4): (1688205, 1353986),
}


class Recorder:
    """runs the calls of one context, checking each one's launch count and (profiling on) kernel_times slots"""

    def __init__(self, ctx, cuda):
        self.ctx, self.cuda = ctx, cuda
        if cuda:
            assert ctx.lib.bbs_ctx_set_profiling(ctx.handle, 1) == 0

    def __call__(self, name, fn, *args, **kw):
        before = self.ctx.launch_count()
        out = fn(*args, **kw)
        host, cuda, slots = PATHS[name]
        assert self.ctx.launch_count() - before == (cuda if self.cuda else host), name
        if self.cuda and slots is not None:
            ms = (C.c_float * 8)()
            assert self.ctx.lib.bbs_ctx_kernel_times(self.ctx.handle, ms, 8) == 0
            got = "".join(str(k) for k in range(8) if ms[k] > 0)
            if "0" not in slots:
                got = got.replace("0", "")
            assert got == slots, (name, list(ms))
        return out


def core_proof_gen(ctx, sigs, scalars, L, dis, rss, ph=b"", headers=None, phs=None):
    """bbs_core_proof_gen_batch, or bbs_core_proof_gen_batch_hdr when `phs` (one ph per item) is given"""
    n = len(sigs)
    U = L - len(dis)
    sigb = np.frombuffer(b"".join(sigs), np.uint8)
    idx = np.tile(np.array(dis, np.uint32), n)
    dis_off = np.arange(n + 1, dtype=np.uint64) * len(dis)
    rand = np.frombuffer(b"".join(s for r in rss for s in r), np.uint8)
    rand_off = np.arange(n + 1, dtype=np.uint64) * (5 + U)
    commit_off = np.arange(n + 1, dtype=np.uint64) * U
    pf = ctx.suite.proof_fixed_bytes
    fixed = np.zeros(n * pf, np.uint8)
    commit = np.zeros(max(n * U, 1) * 32, np.uint8)
    st = np.full(n, 255, np.uint8)
    if phs is not None:
        hb, hoff = A._pack_items(headers, n, "header") if headers is not None else (None, None)
        pb, poff = A._pack_items(phs, n, "ph")
        rc = ctx.lib.bbs_core_proof_gen_batch_hdr(ctx.handle, n, A._ptr(sigb), A._ptr(scalars), L, A._ptr(idx), A._ptr(dis_off),
                                                  A._ptr(rand), A._ptr(rand_off), A._ptr(commit_off), A._ptr(hb), A._ptr(hoff),
                                                  A._ptr(pb), A._ptr(poff), A._ptr(fixed), A._ptr(commit), A._ptr(st))
    else:
        phb = A._buf(ph) if ph else None
        rc = ctx.lib.bbs_core_proof_gen_batch(ctx.handle, n, A._ptr(sigb), A._ptr(scalars), L, A._ptr(idx), A._ptr(dis_off),
                                              A._ptr(rand), A._ptr(rand_off), A._ptr(commit_off), A._ptr(phb), len(ph), A._ptr(fixed),
                                              A._ptr(commit), A._ptr(st))
    assert rc == 0, ctx.lib.bbs_last_error()
    return [A.ProofBytes(fixed[i * pf:(i + 1) * pf].tobytes(), commit[i * U * 32:(i + 1) * U * 32].tobytes()) for i in range(n)], st


def pairs(proofs):
    return [(p.fixed, p.commitments) for p in proofs]


def run_small_paths(lib_path, curve, L=3, n=4):
    """the fixed call sequence on one per-item-header context whose own header is `h`: the items whose per-item header is
    `h` give what the calls without _hdr give.  Returns (context memory bytes, issuer set shared bytes)."""
    suite, ocs = P.SUITES[curve]
    sk, pk = P.keypair(ocs, 1)
    skb = sk.to_bytes(32, "little")
    h, p = b"paths-header", b"paths-ph"
    ctx, gens = ctx_for(lib_path, curve, L, header=h)
    iset = A.IssuerSet(suite, [ocs.g2_compress(pk)], h, generators=P.gens_bytes(ocs, gens), lib_path=lib_path)
    run = Recorder(ctx, lib_path is None)
    hdrs = [h if i % 2 == 0 else x for i, x in enumerate(headers_of([3 + 40 * i for i in range(n)], "paths"))]
    same = [i for i in range(n) if hdrs[i] == h]
    msgs = [[P.rng_bytes(f"pa{i}.{j}", 5 + 9 * j) for j in range(L)] for i in range(n)]

    sc = run("msg_to_scalars", ctx.msg_to_scalars, [m for item in msgs for m in item]).reshape(-1)
    assert sc.tobytes() == scalar_blob(ocs, [O.msg_to_scalars(ocs, m, ocs.api_id) for m in msgs]).tobytes()

    # sign
    s1, b1, st = run("sign", ctx.sign_batch, skb, msgs, want_b=True)
    assert st.tolist() == [1] * n
    s2, b2, st2 = run("core_sign", ctx.core_sign_batch, skb, sc, n, L, want_b=True)
    assert (s1.tobytes(), b1.tobytes(), st.tolist()) == (s2.tobytes(), b2.tobytes(), st2.tolist())
    hs1, hb1, hst = run("sign_hdr", ctx.sign_batch, skb, msgs, want_b=True, headers=hdrs)
    hs2, hb2, hst2 = run("core_sign_hdr", ctx.core_sign_batch, skb, sc, n, L, want_b=True, headers=hdrs)
    assert (hs1.tobytes(), hb1.tobytes(), hst.tolist()) == (hs2.tobytes(), hb2.tobytes(), hst2.tolist())
    assert hst.tolist() == [1] * n
    assert hs1[same].tobytes() == s1[same].tobytes() and hs1[1].tobytes() != s1[1].tobytes()

    # verify: item 1 damaged
    bad, hbad = s1.copy(), hs1.copy()
    bad[1, -1] ^= 1
    hbad[1, -1] ^= 1
    v = run("verify", ctx.verify_batch, bad, msgs)
    assert v.tolist() == [1, 0] + [1] * (n - 2)
    assert run("core_verify", ctx.core_verify_batch, bad, sc, L).tolist() == v.tolist()
    assert run("verify_hdr", ctx.verify_batch, hbad, msgs, headers=hdrs).tolist() == v.tolist()
    assert run("core_verify_hdr", ctx.core_verify_batch, hbad, sc, L, headers=hdrs).tolist() == v.tolist()
    assert iset.verify_batch([0] * n, bad, msgs).tolist() == v.tolist()
    assert iset.core_verify_batch([0] * n, bad, sc, L).tolist() == v.tolist()

    # proof gen
    dis = [0, 2] if L >= 3 else [0]
    rss = [[ocs.scalar_le(x) for x in O.seeded_random_scalars(ocs, b"pa%d" % i, b"rs", 5 + L - len(dis))] for i in range(n)]
    sl, hsl = [s1[i].tobytes() for i in range(n)], [hs1[i].tobytes() for i in range(n)]
    phs = headers_of([0, 1, 64, 300][:n] + [7] * max(0, n - 4), "paths-ph")
    g1, gst = run("proof_gen", ctx.proof_gen_batch, sl, msgs, [dis] * n, rss, p)
    assert gst.tolist() == [1] * n
    g2, gst2 = run("core_proof_gen", core_proof_gen, ctx, sl, sc, L, dis, rss, ph=p)
    assert pairs(g1) == pairs(g2) and gst2.tolist() == gst.tolist()
    g3, gst3 = run("proof_gen_ph", ctx.proof_gen_batch, sl, msgs, [dis] * n, rss, [p] * n)
    assert pairs(g1) == pairs(g3) and gst3.tolist() == gst.tolist()
    hg1, hgst = run("proof_gen_hdr", ctx.proof_gen_batch, hsl, msgs, [dis] * n, rss, phs, headers=hdrs)
    assert hgst.tolist() == [1] * n
    hg2, hgst2 = run("core_proof_gen_hdr", core_proof_gen, ctx, hsl, sc, L, dis, rss, headers=hdrs, phs=phs)
    assert pairs(hg1) == pairs(hg2) and hgst2.tolist() == hgst.tolist()

    # proof verify: proof 1 damaged
    proofs, hproofs = list(g1), list(hg1)
    for lst in (proofs, hproofs):
        lst[1] = A.ProofBytes(lst[1].fixed[:-1] + bytes([lst[1].fixed[-1] ^ 1]), lst[1].commitments)
    dm = [[m[j] for j in dis] for m in msgs]
    dsc = [[sc[(i * L + j) * 32:(i * L + j + 1) * 32].tobytes() for j in dis] for i in range(n)]
    w = run("proof_verify", ctx.proof_verify_batch, proofs, p, dm, [dis] * n)
    assert w.tolist()[0] == 1 and w.tolist()[1] != 1
    assert run("core_proof_verify", ctx.core_proof_verify_batch, proofs, p, dsc, [dis] * n).tolist() == w.tolist()
    assert run("proof_verify_ph", ctx.proof_verify_batch, proofs, [p] * n, dm, [dis] * n).tolist() == w.tolist()
    assert run("core_proof_verify_ph", ctx.core_proof_verify_batch, proofs, [p] * n, dsc, [dis] * n).tolist() == w.tolist()
    assert run("proof_verify_hdr", ctx.proof_verify_batch, hproofs, phs, dm, [dis] * n, headers=hdrs).tolist() == w.tolist()
    assert run("core_proof_verify_hdr", ctx.core_proof_verify_batch, hproofs, phs, dsc, [dis] * n,
               headers=hdrs).tolist() == w.tolist()
    assert iset.proof_verify_batch([0] * n, proofs, p, dm, [dis] * n).tolist() == w.tolist()
    assert iset.core_proof_verify_batch([0] * n, proofs, p, dsc, [dis] * n).tolist() == w.tolist()

    mem = (ctx.memory_bytes(), iset.memory_bytes()[1])
    if lib_path is None:
        run_rlc(ctx, run, bad, s1, msgs, sc, L)
    iset.close()
    ctx.close()
    return mem


def run_rlc(ctx, run, bad, good, msgs, sc, L):
    """the random-linear-combination calls in both forms (CUDA build only)"""
    n = len(msgs)
    seed = P.rng_bytes("paths-seed", 32)
    assert run("rlc_verify", ctx.rlc_verify_batch, good, msgs, seed) == 1
    v = np.zeros(1, np.uint8)
    assert run("rlc_core_verify", ctx.lib.bbs_rlc_core_verify_batch, ctx.handle, n, A._ptr(A._buf(bad)), A._ptr(sc), L,
               A._ptr(A._buf(seed)), A._ptr(v)) == 0
    assert v[0] == ctx.rlc_verify_batch(bad, msgs, seed) == 0
    parts, st = run("rlc_partial", ctx.rlc_partial, good, msgs, seed, 3)
    cparts = np.zeros(2 * ctx.suite.g1_bytes, np.uint8)
    cst = np.zeros(1, np.uint8)
    assert run("rlc_partial_core", ctx.lib.bbs_rlc_partial_core, ctx.handle, n, A._ptr(A._buf(good)), A._ptr(sc), L,
               A._ptr(A._buf(seed)), 3, A._ptr(cparts), A._ptr(cst)) == 0
    assert (parts, st) == (cparts.tobytes(), int(cst[0])) and st == 1


@pytest.fixture(scope="module")
def hs():
    path = hostsim.build()
    _native.load(path, allow_host_simulation=True)      # tests only: the product loader refuses non-CUDA builds
    return path


@pytest.mark.parametrize("curve", CURVES)
def test_host_paths(hs, curve):
    assert run_small_paths(hs, curve) == MEMORY[(curve, 3, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_gpu_paths(curve):
    _native.load()
    run_small_paths(None, curve)


@pytest.mark.gpu
def test_gpu_chunked_paths():
    """verify at 262,144 items and sign at 524,288 items take the chunked pipelines; the _hdr calls with the context's
    header for every item take none and give the same bytes"""
    _native.load()
    suite, ocs = P.SUITES["BLS12_381"]
    sk, pk = P.keypair(ocs, 2)
    skb = sk.to_bytes(32, "little")
    h, L = b"chunk-header", 2
    ctx, _ = ctx_for(None, "BLS12_381", L, header=h, pk=pk)
    run = Recorder(ctx, True)
    rng = np.random.default_rng(3)
    n = 262_144
    msgs = [[b"chunk-%d.%d" % (i, j) for j in range(L)] for i in range(n)]
    sc = ctx.msg_to_scalars([m for item in msgs for m in item]).reshape(-1)
    sigs, _, st = ctx.core_sign_batch(skb, sc, n, L)
    assert (st == 1).all()
    sigs[rng.choice(n, size=n // 16, replace=False), -1] ^= 1
    want = run("verify_hdr_large", ctx.verify_batch, sigs, msgs, headers=[h] * n)
    assert 0 < int(want.sum()) < n
    assert np.array_equal(run("verify_chunked", ctx.verify_batch, sigs, msgs), want)
    assert np.array_equal(run("core_verify_chunked", ctx.core_verify_batch, sigs, sc, L), want)
    assert np.array_equal(run("core_verify_hdr_large", ctx.core_verify_batch, sigs, sc, L, headers=[h] * n), want)
    n = 524_288
    msgs = [[i.to_bytes(4, "little"), b"m"] for i in range(n)]
    sc = _rand_scalars(rng, ocs, n * L).reshape(-1)
    a = run("core_sign_chunked", ctx.core_sign_batch, skb, sc, n, L, want_b=True)
    b = run("core_sign_hdr_large", ctx.core_sign_batch, skb, sc, n, L, want_b=True, headers=[h] * n)
    assert all(np.array_equal(x, y) for x, y in zip(a, b)) and (a[2] == 1).all()
    a = run("sign_chunked", ctx.sign_batch, skb, msgs, want_b=True)
    b = run("sign_hdr_large", ctx.sign_batch, skb, msgs, want_b=True, headers=[h] * n)
    assert all(np.array_equal(x, y) for x, y in zip(a, b)) and (a[2] == 1).all()
    ctx.close()
