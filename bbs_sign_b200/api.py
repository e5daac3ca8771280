"""Host-side mirror of the reference's interface for the hot path, as batch calls over the C ABI.

Reference (Rust, /root/reference/src)                     here
---------------------------------------------------------------------------------------------
PublicKey::verify        (verify.rs:18-50)                PublicKey.verify_batch
PublicKey::core_verify   (verify.rs:53-93)                PublicKey.core_verify_batch
proof_verify             (proof_verify.rs:19-61)          proof_verify_batch
core_proof_verify        (proof_verify.rs:64-116)         core_proof_verify_batch
SecretKey::sign          (sign.rs:32-60)                  SecretKey.sign_batch
SecretKey::core_sign     (sign.rs:63-133)                 SecretKey.core_sign_batch
msg_to_scalars           (interface_utilities.rs:76-88)   BatchContext.msg_to_scalars
Bls12381Const / Bn254Const (constants.rs)                 BLS12_381 / BN254

Results follow the reference's `Result<bool, Error>`: every batch call returns a `numpy.uint8` status
vector with 1 = Ok(true), 0 = Ok(false), 2.. = the Err variants (see include/bbs_b200.h).

All arithmetic happens in the CUDA library; this module only packs bytes.  There is no CPU fallback:
importing works anywhere, creating a context needs the built library and a GPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _native

ST_REJECT, ST_ACCEPT, ST_ERR_MSG_GEN_LEN, ST_ERR_DISCLOSED_INDEX, ST_ERR_IDX_MSG_LEN, ST_ERR_MALFORMED = range(6)
ST_ERR_DISCLOSED_LEN, ST_ERR_RANDOM_LEN = 6, 7
CTX_SMALL_TABLES = 1          # BBS_CTX_SMALL_TABLES (bbs_ctx_create_ex)
CTX_PER_ITEM_HEADER = 2       # BBS_CTX_PER_ITEM_HEADER (bbs_ctx_create_ex)



class BbsError(RuntimeError):
    pass


@dataclass(frozen=True)
class Ciphersuite:
    """The reference's `Constants` impls (constants.rs:27-89)."""
    name: str
    curve_id: int
    g1_bytes: int
    g2_bytes: int
    ciphersuite_id: bytes

    @property
    def api_id(self) -> bytes:  # verify.rs:31
        return self.ciphersuite_id + b"H2G_HM2S_"

    @property
    def signature_bytes(self) -> int:
        return self.g1_bytes + 32

    @property
    def proof_fixed_bytes(self) -> int:
        return 3 * self.g1_bytes + 128

    def create_generators(self, count: int, api_id: Optional[bytes] = None, device: int = 0,
                          lib_path: Optional[str] = None) -> bytes:
        """`create_generators(count, api_id)` (interface_utilities.rs:47-73) as `count` compressed G1 points, derived on
        the GPU by bbs_create_generators with the suite's hash-to-G1 (csrc/h2c.cuh).  `api_id` defaults to the suite's."""
        lib = _native.load(lib_path)
        aid = self.api_id if api_id is None else api_id
        out = np.zeros(max(count, 1) * self.g1_bytes, dtype=np.uint8)
        rc = lib.bbs_create_generators(self.curve_id, device, _ptr(_buf(aid)) if aid else None, len(aid), count, _ptr(out))
        if rc != 0:
            raise BbsError(f"bbs_create_generators failed ({rc}): {lib.bbs_last_error().decode()}")
        return out[: count * self.g1_bytes].tobytes()

    derive_generators = create_generators


BLS12_381 = Ciphersuite("BLS12_381", 1, 48, 96, b"BBS_BLS12381G1_XMD:SHA-256_SSWU_RO_")
BN254 = Ciphersuite("BN254", 2, 32, 64, b"BBS_QUUX-V01-CS02-with-BN254G1_XMD:SHA-256_SVDW_RO_")


def _buf(b) -> np.ndarray:
    a = np.frombuffer(b, dtype=np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b).view(np.uint8).reshape(-1)
    return a


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pack_ragged(items: Sequence[bytes]):
    offs = np.zeros(len(items) + 1, dtype=np.uint64)
    if len(items):
        offs[1:] = np.cumsum([len(m) for m in items], dtype=np.uint64)
    flat = np.frombuffer(b"".join(items), dtype=np.uint8) if len(items) else np.zeros(0, dtype=np.uint8)
    if flat.size == 0:
        flat = np.zeros(1, dtype=np.uint8)
    return flat, offs


def _is_per_item(x) -> bool:
    """a header / ph argument given as a list / tuple of byte strings, one per item, rather than one shared byte string
    (bytes, bytearray, memoryview or a numpy uint8 array, as the calls have always accepted)"""
    return x is not None and not isinstance(x, (bytes, bytearray, memoryview, np.ndarray))


def _pack_items(items, n: int, what: str):
    """one byte string per item -> (flat bytes, n + 1 uint64 offsets) as the *_hdr calls take them"""
    items = [bytes(x) for x in items]
    if len(items) != n:
        raise BbsError(f"one {what} per item required ({len(items)} for {n} items)")
    return _pack_ragged(items)


class BatchContext:
    """Per (GPU, issuer key, header, generators) state: `bbs_ctx_create` of include/bbs_b200.h.  With
    `per_item_headers=True` (BBS_CTX_PER_ITEM_HEADER) the batch methods also accept `headers=` (one header per item), so
    one context serves every header of a key and L."""

    def __init__(self, suite: Ciphersuite, pk: bytes, header: bytes = b"", n_messages: Optional[int] = None,
                 generators: Optional[bytes] = None, api_id: Optional[bytes] = None, device: int = 0,
                 lib_path: Optional[str] = None, small_tables: bool = False, per_item_headers: bool = False):
        self.suite = suite
        self.lib = _native.load(lib_path)
        if generators is None:
            if n_messages is None:
                raise BbsError("n_messages or generators required")
            generators = suite.create_generators(n_messages + 1, device=device, lib_path=lib_path)
        if len(generators) % suite.g1_bytes:
            raise BbsError("generators must be a whole number of compressed G1 points")
        self.n_generators = len(generators) // suite.g1_bytes
        self.L = self.n_generators - 1
        self.api_id = suite.api_id if api_id is None else api_id
        self.header = header
        self.per_item_headers = per_item_headers
        self.pk = bytes(pk)
        if len(self.pk) != suite.g2_bytes:
            raise BbsError("public key has the wrong length")
        h = C.c_void_p()
        hdr = _buf(header) if header else None
        aid = _buf(self.api_id) if self.api_id else None
        flags = (CTX_SMALL_TABLES if small_tables else 0) | (CTX_PER_ITEM_HEADER if per_item_headers else 0)
        rc = self.lib.bbs_ctx_create_ex(suite.curve_id, device, flags, _ptr(_buf(self.pk)),
                                        _ptr(_buf(generators)), self.n_generators, _ptr(hdr), len(header), _ptr(aid),
                                        len(self.api_id), C.byref(h))
        if rc != 0:
            raise BbsError(f"bbs_ctx_create failed ({rc}): {self.lib.bbs_last_error().decode()}")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self.lib.bbs_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def _check(self, rc, what):
        if rc != 0:
            raise BbsError(f"{what} failed ({rc}): {self.lib.bbs_last_error().decode()}")

    def domain(self) -> bytes:
        out = np.zeros(32, dtype=np.uint8)
        self._check(self.lib.bbs_ctx_domain(self._h, _ptr(out)), "bbs_ctx_domain")
        return out.tobytes()

    def launch_count(self) -> int:
        return int(self.lib.bbs_ctx_launch_count(self._h))

    def memory_bytes(self) -> int:
        return int(self.lib.bbs_ctx_memory_bytes(self._h))

    # ---- interface_utilities.rs:76-88 ----
    def msg_to_scalars(self, messages: Sequence[bytes]) -> np.ndarray:
        flat, offs = _pack_ragged(messages)
        out = np.zeros((len(messages), 32), dtype=np.uint8)
        self._check(self.lib.bbs_msg_to_scalars(self._h, len(messages), _ptr(flat), _ptr(offs), _ptr(out)), "bbs_msg_to_scalars")
        return out

    # ---- verify.rs ----
    def core_verify_batch(self, signatures, msg_scalars, n_msgs: int, *, headers: Optional[Sequence[bytes]] = None) -> np.ndarray:
        """`headers`: one header per signature instead of the context's (needs `per_item_headers=True`)"""
        sigs = _buf(signatures)
        n = sigs.size // self.suite.signature_bytes
        sc = _buf(msg_scalars)
        if sc.size != n * n_msgs * 32:
            raise BbsError("msg_scalars has the wrong size")
        if sc.size == 0:
            sc = np.zeros(1, dtype=np.uint8)
        st = np.full(n, 255, dtype=np.uint8)
        if headers is not None:
            hdr, hoff = _pack_items(headers, n, "header")
            self._check(self.lib.bbs_core_verify_batch_hdr(self._h, n, _ptr(sigs), _ptr(sc), n_msgs, _ptr(hdr), _ptr(hoff), _ptr(st)),
                        "bbs_core_verify_batch_hdr")
            return st
        self._check(self.lib.bbs_core_verify_batch(self._h, n, _ptr(sigs), _ptr(sc), n_msgs, _ptr(st)), "bbs_core_verify_batch")
        return st

    def verify_batch(self, signatures, messages: Sequence[Sequence[bytes]], *,
                     headers: Optional[Sequence[bytes]] = None) -> np.ndarray:
        """`headers`: one header per signature instead of the context's (needs `per_item_headers=True`)"""
        sigs = _buf(signatures)
        n = sigs.size // self.suite.signature_bytes
        if len(messages) != n:
            raise BbsError("one message list per signature required")
        n_msgs = len(messages[0]) if n else 0
        if any(len(m) != n_msgs for m in messages):
            raise BbsError("all items of a batch must carry the same number of messages")
        flat, offs = _pack_ragged([m for item in messages for m in item])
        st = np.full(n, 255, dtype=np.uint8)
        if headers is not None:
            hdr, hoff = _pack_items(headers, n, "header")
            self._check(self.lib.bbs_verify_batch_hdr(self._h, n, _ptr(sigs), _ptr(flat), _ptr(offs), n_msgs, _ptr(hdr), _ptr(hoff),
                                                      _ptr(st)), "bbs_verify_batch_hdr")
            return st
        self._check(self.lib.bbs_verify_batch(self._h, n, _ptr(sigs), _ptr(flat), _ptr(offs), n_msgs, _ptr(st)), "bbs_verify_batch")
        return st

    # ---- random-linear-combination batch mode (not in the reference; include/bbs_b200.h) -------------------
    def rlc_partial(self, signatures, messages: Sequence[Sequence[bytes]], seed: bytes, index_base: int = 0):
        """This shard's two partial G1 points (compressed) and a status byte (ACCEPT = well-formed shard).  All shards of
        a batch share `seed`, which the coordinator draws (os.urandom) AFTER the whole batch is fixed."""
        n = len(messages)
        n_msgs = len(messages[0]) if n else 0
        flat, offs = _pack_ragged([m for ms in messages for m in ms])
        sigs = _buf(b"".join(signatures) if not isinstance(signatures, (bytes, bytearray)) else signatures)
        parts = np.zeros(2 * self.suite.g1_bytes, dtype=np.uint8)
        st = np.zeros(1, dtype=np.uint8)
        self._check(self.lib.bbs_rlc_partial(self._h, n, _ptr(sigs), _ptr(flat), _ptr(offs), n_msgs, _ptr(_buf(seed)),
                                             index_base, _ptr(parts), _ptr(st)), "bbs_rlc_partial")
        return parts.tobytes(), int(st[0])

    def rlc_combine(self, parts: Sequence[bytes]) -> int:
        blob = _buf(b"".join(parts))
        v = np.zeros(1, dtype=np.uint8)
        self._check(self.lib.bbs_rlc_combine(self._h, len(parts), _ptr(blob), _ptr(v)), "bbs_rlc_combine")
        return int(v[0])

    def rlc_verify_batch(self, signatures, messages: Sequence[Sequence[bytes]], seed: Optional[bytes] = None) -> int:
        """One verdict (ST_ACCEPT / ST_REJECT / ST_ERR_*) for the whole batch; see include/bbs_b200.h.  `seed=None` (the
        default) lets the library draw the coefficient seed from the OS CSPRNG after it has the batch; pass a seed only
        for reproducible tests: a seed the submitter of the batch can predict voids the verdict's soundness."""
        n = len(messages)
        n_msgs = len(messages[0]) if n else 0
        flat, offs = _pack_ragged([m for ms in messages for m in ms])
        sigs = _buf(b"".join(signatures) if not isinstance(signatures, (bytes, bytearray)) else signatures)
        v = np.zeros(1, dtype=np.uint8)
        self._check(self.lib.bbs_rlc_verify_batch(self._h, n, _ptr(sigs), _ptr(flat), _ptr(offs), n_msgs,
                                                  _ptr(_buf(seed)) if seed is not None else None, _ptr(v)), "bbs_rlc_verify_batch")
        return int(v[0])

    # ---- test hooks (include/bbs_b200.h) ----
    def use_per_thread_pairing(self, on: bool = True):
        self._check(self.lib.bbs_ctx_use_per_thread_pairing(self._h, 1 if on else 0), "bbs_ctx_use_per_thread_pairing")

    def set_g1_split(self, max_items: int):
        self._check(self.lib.bbs_ctx_set_g1_split(self._h, max_items), "bbs_ctx_set_g1_split")

    def set_pairing_split(self, max_items: int):
        """test hook: batches of up to `max_items` (<= 32) items run the pairing kernel with two warps per role; 0 = never"""
        self._check(self.lib.bbs_ctx_set_pairing_split(self._h, max_items), "bbs_ctx_set_pairing_split")

    def set_rlc_windows(self, windows: int):
        self._check(self.lib.bbs_ctx_set_rlc_windows(self._h, windows), "bbs_ctx_set_rlc_windows")

    # ---- sign.rs ----
    def core_sign_batch(self, sk_le32: bytes, msg_scalars, n: int, n_msgs: int, want_b: bool = False, *,
                        headers: Optional[Sequence[bytes]] = None):
        """`headers`: one header per signature instead of the context's (needs `per_item_headers=True`)"""
        sc = _buf(msg_scalars)
        if sc.size != n * n_msgs * 32:
            raise BbsError("msg_scalars has the wrong size")
        if sc.size == 0:
            sc = np.zeros(1, dtype=np.uint8)
        sigs = np.zeros((n, self.suite.signature_bytes), dtype=np.uint8)
        b = np.zeros((n, self.suite.g1_bytes), dtype=np.uint8) if want_b else None
        st = np.full(n, 255, dtype=np.uint8)
        if headers is not None:
            hdr, hoff = _pack_items(headers, n, "header")
            self._check(self.lib.bbs_core_sign_batch_hdr(self._h, _ptr(_buf(sk_le32)), n, _ptr(sc), n_msgs, _ptr(hdr), _ptr(hoff),
                                                         _ptr(sigs), _ptr(b), _ptr(st)), "bbs_core_sign_batch_hdr")
            return sigs, b, st
        self._check(self.lib.bbs_core_sign_batch(self._h, _ptr(_buf(sk_le32)), n, _ptr(sc), n_msgs, _ptr(sigs), _ptr(b), _ptr(st)),
                    "bbs_core_sign_batch")
        return sigs, b, st

    def sign_batch(self, sk_le32: bytes, messages: Sequence[Sequence[bytes]], want_b: bool = False, *,
                   headers: Optional[Sequence[bytes]] = None):
        """`headers`: one header per message list instead of the context's (needs `per_item_headers=True`)"""
        n = len(messages)
        n_msgs = len(messages[0]) if n else 0
        if any(len(m) != n_msgs for m in messages):
            raise BbsError("all items of a batch must carry the same number of messages")
        flat, offs = _pack_ragged([m for item in messages for m in item])
        sigs = np.zeros((n, self.suite.signature_bytes), dtype=np.uint8)
        b = np.zeros((n, self.suite.g1_bytes), dtype=np.uint8) if want_b else None
        st = np.full(n, 255, dtype=np.uint8)
        if headers is not None:
            hdr, hoff = _pack_items(headers, n, "header")
            self._check(self.lib.bbs_sign_batch_hdr(self._h, _ptr(_buf(sk_le32)), n, _ptr(flat), _ptr(offs), n_msgs, _ptr(hdr),
                                                    _ptr(hoff), _ptr(sigs), _ptr(b), _ptr(st)), "bbs_sign_batch_hdr")
            return sigs, b, st
        self._check(self.lib.bbs_sign_batch(self._h, _ptr(_buf(sk_le32)), n, _ptr(flat), _ptr(offs), n_msgs, _ptr(sigs), _ptr(b), _ptr(st)),
                    "bbs_sign_batch")
        return sigs, b, st

    # ---- proof_verify.rs ----
    def proof_gen_batch(self, signatures, messages: Sequence[Sequence[bytes]], disclosed_indexes: Sequence[Sequence[int]],
                        random_scalars: Sequence[Sequence[bytes]], ph=b"", *, headers: Optional[Sequence[bytes]] = None):
        """Batch form of `proof_gen` (proof_gen.rs:78-113) with caller-supplied random scalars (LE32 each, 5 + U per
        item).  `ph` is one presentation header for the batch or one per item; `headers` one header per item instead of the
        context's (needs `per_item_headers=True`).  Returns (list of ProofBytes or None, status array)."""
        n = len(messages)
        n_msgs = len(messages[0]) if n else 0
        flat, offs = _pack_ragged([m for ms in messages for m in ms])
        sigs = _buf(b"".join(signatures))
        idx = np.array([i for d in disclosed_indexes for i in d], dtype=np.uint32)
        if idx.size == 0:
            idx = np.zeros(1, np.uint32)
        dis_off = np.zeros(n + 1, dtype=np.uint64)
        rand_off = np.zeros(n + 1, dtype=np.uint64)
        commit_off = np.zeros(n + 1, dtype=np.uint64)
        if n:
            dis_off[1:] = np.cumsum([len(d) for d in disclosed_indexes], dtype=np.uint64)
            rand_off[1:] = np.cumsum([len(r) for r in random_scalars], dtype=np.uint64)
            commit_off[1:] = np.cumsum([max(len(r) - 5, 0) for r in random_scalars], dtype=np.uint64)
        rand = _buf(b"".join(s for r in random_scalars for s in r) or b"\0")
        fixed = np.zeros(max(n, 1) * self.suite.proof_fixed_bytes, dtype=np.uint8)
        commit = np.zeros(max(int(commit_off[n]), 1) * 32, dtype=np.uint8)
        st = np.full(n, 255, dtype=np.uint8)
        if headers is not None or _is_per_item(ph):
            phs, poff = _pack_items(ph if _is_per_item(ph) else [ph] * n, n, "ph")
            hdr, hoff = _pack_items(headers, n, "header") if headers is not None else (None, None)
            self._check(self.lib.bbs_proof_gen_batch_hdr(self._h, n, _ptr(sigs), _ptr(flat), _ptr(offs), n_msgs, _ptr(idx),
                                                         _ptr(dis_off), _ptr(rand), _ptr(rand_off), _ptr(commit_off), _ptr(hdr),
                                                         _ptr(hoff), _ptr(phs), _ptr(poff), _ptr(fixed), _ptr(commit), _ptr(st)),
                        "bbs_proof_gen_batch_hdr")
        else:
            phb = _buf(ph) if len(ph) else None
            self._check(self.lib.bbs_proof_gen_batch(self._h, n, _ptr(sigs), _ptr(flat), _ptr(offs), n_msgs, _ptr(idx),
                                                     _ptr(dis_off), _ptr(rand), _ptr(rand_off), _ptr(commit_off), _ptr(phb),
                                                     len(ph), _ptr(fixed), _ptr(commit), _ptr(st)), "bbs_proof_gen_batch")
        pf = self.suite.proof_fixed_bytes
        out = []
        for i in range(n):
            if st[i] != ST_ACCEPT:
                out.append(None)
                continue
            out.append(ProofBytes(fixed[i * pf:(i + 1) * pf].tobytes(),
                                  commit[int(commit_off[i]) * 32:int(commit_off[i + 1]) * 32].tobytes()))
        return out, st

    def _pack_proofs(self, proofs: Sequence["ProofBytes"], disclosed_indexes: Sequence[Sequence[int]]):
        n = len(proofs)
        fixed = np.frombuffer(b"".join(p.fixed for p in proofs), dtype=np.uint8) if n else np.zeros(1, np.uint8)
        commit_off = np.zeros(n + 1, dtype=np.uint64)
        dis_off = np.zeros(n + 1, dtype=np.uint64)
        if n:
            commit_off[1:] = np.cumsum([len(p.commitments) // 32 for p in proofs], dtype=np.uint64)
            dis_off[1:] = np.cumsum([len(d) for d in disclosed_indexes], dtype=np.uint64)
        commit = np.frombuffer(b"".join(p.commitments for p in proofs), dtype=np.uint8)
        if commit.size == 0:
            commit = np.zeros(1, np.uint8)
        idx = np.array([i for d in disclosed_indexes for i in d], dtype=np.uint32)
        if idx.size == 0:
            idx = np.zeros(1, np.uint32)
        return fixed, commit, commit_off, idx, dis_off

    def _per_item_ph_args(self, keep, n, ph, headers):
        """(headers, hdr_off, phs, ph_off) of the kept items for a *_proof_verify_batch_hdr call; headers None = the context's"""
        phs = list(ph) if _is_per_item(ph) else [ph] * n
        if len(phs) != n or (headers is not None and len(headers) != n):
            raise BbsError("one ph (and header) per proof required")
        pb, poff = _pack_items([phs[i] for i in keep], len(keep), "ph")
        hb, hoff = _pack_items([headers[i] for i in keep], len(keep), "header") if headers is not None else (None, None)
        return hb, hoff, pb, poff

    def core_proof_verify_batch(self, proofs, ph, disclosed_scalars: Sequence[Sequence[bytes]],
                                disclosed_indexes: Sequence[Sequence[int]], *, headers: Optional[Sequence[bytes]] = None) -> np.ndarray:
        """`ph`: one presentation header for the batch or one per proof; `headers`: one header per proof instead of the
        context's (needs `per_item_headers=True`)"""
        return self._proof_verify(True, proofs, ph, disclosed_scalars, disclosed_indexes, headers)[0]

    def _length_error_status(self, proof, idxs):
        # reference order (proof_verify.rs:139-146): index range check first, then the length check
        L = len(proof.commitments) // 32 + len(idxs)
        return ST_ERR_DISCLOSED_INDEX if any(i >= L for i in idxs) else ST_ERR_IDX_MSG_LEN

    def proof_verify_batch(self, proofs, ph, disclosed_messages: Sequence[Sequence[bytes]],
                           disclosed_indexes: Sequence[Sequence[int]], *, headers: Optional[Sequence[bytes]] = None) -> np.ndarray:
        """`ph`: one presentation header for the batch or one per proof; `headers`: one header per proof instead of the
        context's (needs `per_item_headers=True`)"""
        return self._proof_verify(False, proofs, ph, disclosed_messages, disclosed_indexes, headers)[0]

    def rlc_core_proof_verify_batch(self, proofs, ph, disclosed_scalars: Sequence[Sequence[bytes]],
                                    disclosed_indexes: Sequence[Sequence[int]], *, headers: Optional[Sequence[bytes]] = None,
                                    seed: Optional[bytes] = None):
        """`core_proof_verify_batch` with the pairing half checked by one random linear combination
        (bbs_rlc_core_proof_verify_batch*, include/bbs_b200.h).  Returns (status, combined): the statuses are those of
        `core_proof_verify_batch` (an ACCEPT holds except with probability 2^-128 over the seed); `combined` is ST_ACCEPT
        when the one combined pairing check held (or no proof reached it), ST_REJECT when it failed and the per-item
        pairing decided instead.  `seed=None` (the default) lets the library draw the seed after it has the batch; pass a
        seed only for reproducible tests: a seed the submitter of the batch can predict lets crafted proofs pass."""
        return self._proof_verify(True, proofs, ph, disclosed_scalars, disclosed_indexes, headers, rlc=True, seed=seed)

    def rlc_proof_verify_batch(self, proofs, ph, disclosed_messages: Sequence[Sequence[bytes]],
                               disclosed_indexes: Sequence[Sequence[int]], *, headers: Optional[Sequence[bytes]] = None,
                               seed: Optional[bytes] = None):
        """`proof_verify_batch` with the pairing half checked by one random linear combination; returns (status, combined)
        as `rlc_core_proof_verify_batch`."""
        return self._proof_verify(False, proofs, ph, disclosed_messages, disclosed_indexes, headers, rlc=True, seed=seed)

    def _proof_verify(self, core: bool, proofs, ph, disclosed, disclosed_indexes, headers, rlc: bool = False,
                      seed: Optional[bytes] = None):
        """(status, combined) of the proof verify calls: `disclosed` holds message scalars (core) or messages.  Proofs whose
        disclosed lists differ in length never reach the library; the combined verdict covers the rest (ST_ACCEPT when
        none is left, or without rlc)."""
        n = len(proofs)
        st = np.full(n, 255, dtype=np.uint8)
        combined = np.full(1, ST_ACCEPT, dtype=np.uint8)
        # InvalidIndicesAndMessagesLength (proof_verify.rs:144-146) is a property of the host-side lists
        bad = [len(disclosed[i]) != len(disclosed_indexes[i]) for i in range(n)]
        keep = [i for i in range(n) if not bad[i]]
        if keep:
            fixed, commit, commit_off, idx, dis_off = self._pack_proofs([proofs[i] for i in keep], [disclosed_indexes[i] for i in keep])
            if core:
                dis = (np.frombuffer(b"".join(s for i in keep for s in disclosed[i]), dtype=np.uint8),)
                if dis[0].size == 0:
                    dis = (np.zeros(1, np.uint8),)
            else:
                dis = _pack_ragged([m for i in keep for m in disclosed[i]])
            out = np.full(len(keep), 255, dtype=np.uint8)
            tail = (_ptr(_buf(seed)) if seed is not None else None, _ptr(out), _ptr(combined)) if rlc else (_ptr(out),)
            name = ("bbs_rlc_" if rlc else "bbs_") + ("core_" if core else "") + "proof_verify_batch"
            head = (self._h, len(keep), _ptr(fixed), _ptr(commit), _ptr(commit_off), _ptr(idx)) + tuple(_ptr(d) for d in dis) + (_ptr(dis_off),)
            if headers is not None or _is_per_item(ph):
                hb, hoff, pb, poff = self._per_item_ph_args(keep, n, ph, headers)
                name += "_hdr"
                self._check(getattr(self.lib, name)(*head, _ptr(hb), _ptr(hoff), _ptr(pb), _ptr(poff), *tail), name)
            else:
                phb = _buf(ph) if len(ph) else None
                self._check(getattr(self.lib, name)(*head, _ptr(phb), len(ph), *tail), name)
            st[keep] = out
        for i in range(n):
            if bad[i]:
                st[i] = self._length_error_status(proofs[i], disclosed_indexes[i])
        return st, int(combined[0])


class IssuerSet:
    """Many issuer keys over one generator list / header (`bbs_issuer_set_create`): the reference's `PublicKey::verify`
    takes the key per call (verify.rs:18-30), so a batch may name a different issuer per item.  The generator tables are
    shared; a key costs ~26 KB (BLS12-381).  `status[i]` = ST_ACCEPT for a usable key, ST_ERR_MALFORMED for one that ark's
    `PublicKey::deserialize_compressed` refuses; items naming such a key come back ST_ERR_MALFORMED."""

    def __init__(self, suite: Ciphersuite, pks: Sequence[bytes], header: bytes = b"", n_messages: Optional[int] = None,
                 generators: Optional[bytes] = None, api_id: Optional[bytes] = None, device: int = 0,
                 lib_path: Optional[str] = None):
        self.suite = suite
        self.lib = _native.load(lib_path)
        if generators is None:
            if n_messages is None:
                raise BbsError("n_messages or generators required")
            generators = suite.create_generators(n_messages + 1, device=device, lib_path=lib_path)
        self.n_generators = len(generators) // suite.g1_bytes
        self.L = self.n_generators - 1
        self.api_id = suite.api_id if api_id is None else api_id
        self.n_issuers = len(pks)
        if any(len(pk) != suite.g2_bytes for pk in pks):
            raise BbsError("public key has the wrong length")
        blob = _buf(b"".join(bytes(pk) for pk in pks))
        self.status = np.zeros(self.n_issuers, dtype=np.uint8)
        h = C.c_void_p()
        hdr = _buf(header) if header else None
        aid = _buf(self.api_id) if self.api_id else None
        rc = self.lib.bbs_issuer_set_create(suite.curve_id, device, self.n_issuers, _ptr(blob), _ptr(_buf(generators)),
                                            self.n_generators, _ptr(hdr), len(header), _ptr(aid), len(self.api_id),
                                            _ptr(self.status), C.byref(h))
        if rc != 0:
            raise BbsError(f"bbs_issuer_set_create failed ({rc}): {self.lib.bbs_last_error().decode()}")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self.lib.bbs_issuer_set_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def memory_bytes(self):
        """(bytes that grow with the number of issuers, shared bytes: generator tables + batch scratch)"""
        shared = C.c_uint64()
        per = self.lib.bbs_issuer_set_memory_bytes(self._h, C.byref(shared))
        return int(per), int(shared.value)

    def verify_batch(self, item_issuer: Sequence[int], signatures, messages: Sequence[Sequence[bytes]]) -> np.ndarray:
        """status[i] = `pks[item_issuer[i]].verify(signatures[i], header, messages[i])`"""
        sigs = _buf(b"".join(signatures) if not isinstance(signatures, (bytes, bytearray, np.ndarray)) else signatures)
        n = sigs.size // self.suite.signature_bytes
        if len(messages) != n or len(item_issuer) != n:
            raise BbsError("one message list and one issuer index per signature required")
        n_msgs = len(messages[0]) if n else 0
        if any(len(m) != n_msgs for m in messages):
            raise BbsError("all items of a batch must carry the same number of messages")
        flat, offs = _pack_ragged([m for item in messages for m in item])
        iss = np.ascontiguousarray(np.asarray(item_issuer, dtype=np.uint32))
        st = np.full(n, 255, dtype=np.uint8)
        rc = self.lib.bbs_verify_batch_multi(self._h, n, _ptr(iss), _ptr(sigs), _ptr(flat), _ptr(offs), n_msgs, _ptr(st))
        if rc != 0:
            raise BbsError(f"bbs_verify_batch_multi failed ({rc}): {self.lib.bbs_last_error().decode()}")
        return st

    def core_verify_batch(self, item_issuer: Sequence[int], signatures, msg_scalars, n_msgs: int) -> np.ndarray:
        sigs = _buf(signatures)
        n = sigs.size // self.suite.signature_bytes
        sc = _buf(msg_scalars)
        if sc.size != n * n_msgs * 32 or len(item_issuer) != n:
            raise BbsError("msg_scalars / item_issuer have the wrong size")
        if sc.size == 0:
            sc = np.zeros(1, dtype=np.uint8)
        iss = np.ascontiguousarray(np.asarray(item_issuer, dtype=np.uint32))
        st = np.full(n, 255, dtype=np.uint8)
        rc = self.lib.bbs_core_verify_batch_multi(self._h, n, _ptr(iss), _ptr(sigs), _ptr(sc), n_msgs, _ptr(st))
        if rc != 0:
            raise BbsError(f"bbs_core_verify_batch_multi failed ({rc}): {self.lib.bbs_last_error().decode()}")
        return st

    def proof_verify_batch(self, item_issuer: Sequence[int], proofs, ph: bytes, disclosed_messages: Sequence[Sequence[bytes]],
                           disclosed_indexes: Sequence[Sequence[int]]) -> np.ndarray:
        """status[i] = `pks[item_issuer[i]].proof_verify(proofs[i], header, ph, disclosed_messages[i], disclosed_indexes[i])`
        (proof_verify.rs:19-34)"""
        n = len(proofs)
        if len(item_issuer) != n:
            raise BbsError("one issuer index per proof required")
        st = np.full(n, 255, dtype=np.uint8)
        bad = [len(disclosed_messages[i]) != len(disclosed_indexes[i]) for i in range(n)]
        keep = [i for i in range(n) if not bad[i]]
        if keep:
            fixed, commit, commit_off, idx, dis_off = BatchContext._pack_proofs(self, [proofs[i] for i in keep],
                                                                                [disclosed_indexes[i] for i in keep])
            flat, moffs = _pack_ragged([m for i in keep for m in disclosed_messages[i]])
            iss = np.ascontiguousarray(np.asarray([item_issuer[i] for i in keep], dtype=np.uint32))
            phb = _buf(ph) if len(ph) else None
            out = np.full(len(keep), 255, dtype=np.uint8)
            rc = self.lib.bbs_proof_verify_batch_multi(self._h, len(keep), _ptr(iss), _ptr(fixed), _ptr(commit), _ptr(commit_off),
                                                       _ptr(idx), _ptr(flat), _ptr(moffs), _ptr(dis_off), _ptr(phb), len(ph), _ptr(out))
            if rc != 0:
                raise BbsError(f"bbs_proof_verify_batch_multi failed ({rc}): {self.lib.bbs_last_error().decode()}")
            st[keep] = out
        for i in range(n):
            if bad[i]:
                st[i] = BatchContext._length_error_status(self, proofs[i], disclosed_indexes[i])
        return st

    def core_proof_verify_batch(self, item_issuer: Sequence[int], proofs, ph: bytes, disclosed_scalars: Sequence[Sequence[bytes]],
                                disclosed_indexes: Sequence[Sequence[int]]) -> np.ndarray:
        """as proof_verify_batch with the disclosed messages already mapped to scalars (32-byte little-endian)"""
        n = len(proofs)
        if len(item_issuer) != n or any(len(disclosed_scalars[i]) != len(disclosed_indexes[i]) for i in range(n)):
            raise BbsError("one issuer index per proof and one scalar per disclosed index required")
        if not n:
            return np.zeros(0, dtype=np.uint8)
        fixed, commit, commit_off, idx, dis_off = BatchContext._pack_proofs(self, proofs, disclosed_indexes)
        sc = np.frombuffer(b"".join(s for d in disclosed_scalars for s in d), dtype=np.uint8)
        if sc.size == 0:
            sc = np.zeros(1, np.uint8)
        iss = np.ascontiguousarray(np.asarray(item_issuer, dtype=np.uint32))
        phb = _buf(ph) if len(ph) else None
        st = np.full(n, 255, dtype=np.uint8)
        rc = self.lib.bbs_core_proof_verify_batch_multi(self._h, n, _ptr(iss), _ptr(fixed), _ptr(commit), _ptr(commit_off), _ptr(idx),
                                                        _ptr(sc), _ptr(dis_off), _ptr(phb), len(ph), _ptr(st))
        if rc != 0:
            raise BbsError(f"bbs_core_proof_verify_batch_multi failed ({rc}): {self.lib.bbs_last_error().decode()}")
        return st


@dataclass
class ProofBytes:
    """`Proof<E,F>` (proof_gen.rs:29-39) split as the ABI wants it: the fixed-size fields
    comp(Abar)||comp(Bbar)||comp(D)||LE32(e^)||LE32(r1^)||LE32(r3^)||LE32(c), and the LE32 commitments."""
    fixed: bytes
    commitments: bytes

    @staticmethod
    def from_canonical(suite: Ciphersuite, blob: bytes) -> "ProofBytes":
        """Parse ark `CanonicalSerialize` of Proof: 3 points, 3 scalars, u64 LE length, commitments, challenge."""
        g = suite.g1_bytes
        head = blob[: 3 * g + 96]
        u = int.from_bytes(blob[3 * g + 96: 3 * g + 104], "little")
        commitments = blob[3 * g + 104: 3 * g + 104 + 32 * u]
        challenge = blob[3 * g + 104 + 32 * u: 3 * g + 136 + 32 * u]
        if len(challenge) != 32:
            raise BbsError("truncated proof")
        return ProofBytes(head + challenge, commitments)


class PublicKey:
    """`PublicKey<E>` (key_gen.rs:12-15) with the batch entry points the north star adds."""

    MAX_CONTEXTS = 4       # contexts kept per key: one is 0.55 GB of HBM at L = 10 (header and L vary per call in the reference)

    def __init__(self, suite: Ciphersuite, pk: bytes, lib_path: Optional[str] = None):
        self.suite, self.pk, self.lib_path = suite, bytes(pk), lib_path
        self._ctx = {}         # (header, L, device) -> BatchContext, least recently used first; header None = per-item headers

    def context(self, header: Optional[bytes], n_messages: int, device: int = 0) -> BatchContext:
        """the context for `header`, or (header None) the one context serving every header of (L, device)"""
        key = (header, n_messages, device)
        ctx = self._ctx.pop(key, None)
        if ctx is None:
            while len(self._ctx) >= self.MAX_CONTEXTS:
                self._ctx.pop(next(iter(self._ctx))).close()
            ctx = BatchContext(self.suite, self.pk, header or b"", n_messages, device=device, lib_path=self.lib_path,
                               per_item_headers=header is None)
        self._ctx[key] = ctx
        return ctx

    def verify_batch(self, signatures, header, messages: Sequence[Sequence[bytes]], device: int = 0) -> np.ndarray:
        """verify.rs:18-50; messages[i] is the message list of signature i, `header` one header for the batch or one per
        signature."""
        n_msgs = len(messages[0]) if len(messages) else 0
        if _is_per_item(header):
            return self.context(None, n_msgs, device).verify_batch(signatures, messages, headers=header)
        return self.context(header, n_msgs, device).verify_batch(signatures, messages)

    def proof_verify_batch(self, proofs: Sequence[ProofBytes], header, ph,
                           disclosed_messages: Sequence[Sequence[bytes]], disclosed_indexes: Sequence[Sequence[int]],
                           device: int = 0) -> np.ndarray:
        """proof_verify.rs:19-61 for a batch with the same total message count; `header` and `ph` are each one byte string
        for the batch or one per proof."""
        if not proofs:
            return np.zeros(0, dtype=np.uint8)
        L = len(proofs[0].commitments) // 32 + len(disclosed_indexes[0])
        if _is_per_item(header):
            return self.context(None, L, device).proof_verify_batch(proofs, ph, disclosed_messages, disclosed_indexes,
                                                                    headers=header)
        return self.context(header, L, device).proof_verify_batch(proofs, ph, disclosed_messages, disclosed_indexes)


class SecretKey:
    """`SecretKey<F>` (key_gen.rs:29-32); `sk` is the 32-byte little-endian scalar, `pk` its public key
    (the reference derives it with sk_to_pk on every sign call, sign.rs:81)."""

    def __init__(self, suite: Ciphersuite, sk_le32: bytes, pk: bytes):
        self.suite, self.sk, self.pk = suite, bytes(sk_le32), PublicKey(suite, pk)

    def sign_batch(self, messages: Sequence[Sequence[bytes]], header, want_b: bool = False, device: int = 0):
        """sign.rs:32-60; `header` is one header for the batch or one per message list."""
        n_msgs = len(messages[0]) if len(messages) else 0
        if _is_per_item(header):
            return self.pk.context(None, n_msgs, device).sign_batch(self.sk, messages, want_b, headers=header)
        return self.pk.context(header, n_msgs, device).sign_batch(self.sk, messages, want_b)
