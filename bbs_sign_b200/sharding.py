"""Multi-GPU sharding of a batch by signature index (SURVEY 8e): contiguous split, one context and one
host thread per GPU, statuses written straight into the caller's slice, no collective on the data path.
MultiIssuerVerifier: batches whose items name different issuer keys (SURVEY 8f-4), grouped per key."""
from __future__ import annotations

import os
import threading
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .api import BatchContext, Ciphersuite, IssuerSet, _is_per_item


def shard_bounds(n: int, world: int) -> List[Tuple[int, int]]:
    """GPU g gets [g*n/world, (g+1)*n/world) -- the split the north star names."""
    return [(g * n // world, (g + 1) * n // world) for g in range(world)]


class ShardedVerifier:
    """`verify_batch` over several GPUs of one box (one BatchContext per device).  `per_item_headers=True` builds contexts
    that also take one header per item (`headers=`)."""

    def __init__(self, suite: Ciphersuite, pk: bytes, header: bytes, n_messages: int, devices: Sequence[int],
                 lib_path: Optional[str] = None, per_item_headers: bool = False):
        self.suite = suite
        self.ctxs = [BatchContext(suite, pk, header, n_messages, device=d, lib_path=lib_path, per_item_headers=per_item_headers)
                     for d in devices]

    def verify_batch(self, signatures, messages: Sequence[Sequence[bytes]], *,
                     headers: Optional[Sequence[bytes]] = None) -> np.ndarray:
        sigs = np.frombuffer(signatures, dtype=np.uint8) if not isinstance(signatures, np.ndarray) else signatures.reshape(-1)
        sb = self.suite.signature_bytes
        n = sigs.size // sb
        out = np.full(n, 255, dtype=np.uint8)
        errs: list = []

        def work(ctx, lo, hi):
            try:
                if hi > lo:
                    out[lo:hi] = ctx.verify_batch(sigs[lo * sb: hi * sb], messages[lo:hi],
                                                  headers=None if headers is None else headers[lo:hi])
            except Exception as e:  # pragma: no cover
                errs.append(e)

        ts = [threading.Thread(target=work, args=(c, lo, hi)) for c, (lo, hi) in zip(self.ctxs, shard_bounds(n, len(self.ctxs)))]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errs:
            raise errs[0]
        return out

    def _run_sharded(self, n, work):
        errs: list = []

        def guarded(ctx, g, lo, hi):
            try:
                if hi > lo:
                    work(ctx, g, lo, hi)
            except Exception as e:  # pragma: no cover
                errs.append(e)

        ts = [threading.Thread(target=guarded, args=(c, g, lo, hi))
              for g, (c, (lo, hi)) in enumerate(zip(self.ctxs, shard_bounds(n, len(self.ctxs))))]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errs:
            raise errs[0]

    def proof_verify_batch(self, proofs, ph, disclosed_messages, disclosed_indexes, *,
                           headers: Optional[Sequence[bytes]] = None) -> np.ndarray:
        """`proof_verify_batch` split by proof index (same contract as BatchContext.proof_verify_batch: `ph` shared or
        one per proof, `headers` one per proof)."""
        n = len(proofs)
        out = np.full(n, 255, dtype=np.uint8)
        per_item_ph = _is_per_item(ph)

        def work(ctx, g, lo, hi):
            out[lo:hi] = ctx.proof_verify_batch(proofs[lo:hi], ph[lo:hi] if per_item_ph else ph, disclosed_messages[lo:hi],
                                                disclosed_indexes[lo:hi], headers=None if headers is None else headers[lo:hi])

        self._run_sharded(n, work)
        return out

    def rlc_proof_verify_batch(self, proofs, ph, disclosed_messages, disclosed_indexes, *,
                               headers: Optional[Sequence[bytes]] = None):
        """`BatchContext.rlc_proof_verify_batch` split by proof index: every GPU checks its slice with one combined pairing
        under its own library-drawn seed, so nothing is exchanged.  Returns (status, combined); `combined` is ST_ACCEPT
        only if every shard's was."""
        n = len(proofs)
        out = np.full(n, 255, dtype=np.uint8)
        combined = [1] * len(self.ctxs)
        per_item_ph = _is_per_item(ph)

        def work(ctx, g, lo, hi):
            out[lo:hi], combined[g] = ctx.rlc_proof_verify_batch(
                proofs[lo:hi], ph[lo:hi] if per_item_ph else ph, disclosed_messages[lo:hi], disclosed_indexes[lo:hi],
                headers=None if headers is None else headers[lo:hi])

        self._run_sharded(n, work)
        return out, (1 if all(c == 1 for c in combined) else 0)

    def rlc_verify_batch_status(self, signatures, messages: Sequence[Sequence[bytes]], *,
                                headers: Optional[Sequence[bytes]] = None):
        """`BatchContext.rlc_verify_batch_status` split by signature index: every GPU checks its slice with one combined
        pairing under its own library-drawn seed, so nothing is exchanged.  Returns (status, combined); `combined` is
        ST_ACCEPT only if every shard's was."""
        sigs = np.frombuffer(b"".join(signatures) if isinstance(signatures, (list, tuple)) else signatures, dtype=np.uint8) \
            if not isinstance(signatures, np.ndarray) else signatures.reshape(-1)
        sb = self.suite.signature_bytes
        n = sigs.size // sb
        out = np.full(n, 255, dtype=np.uint8)
        combined = [1] * len(self.ctxs)

        def work(ctx, g, lo, hi):
            out[lo:hi], combined[g] = ctx.rlc_verify_batch_status(sigs[lo * sb: hi * sb], messages[lo:hi],
                                                                  headers=None if headers is None else headers[lo:hi])

        self._run_sharded(n, work)
        return out, (1 if all(c == 1 for c in combined) else 0)

    def rlc_verify_batch(self, signatures: Sequence[bytes], messages: Sequence[Sequence[bytes]],
                         seed: Optional[bytes] = None) -> int:
        """Random-linear-combination verdict for the whole batch: every GPU reduces its slice to two compressed G1
        points (coefficients are indexed globally), GPU 0 adds them and does the single pairing check.  The coefficient
        seed is drawn here (os.urandom), after the batch has been handed over; pass one only for reproducible tests."""
        if seed is None:
            seed = os.urandom(32)
        n = len(messages)
        parts: list = [None] * len(self.ctxs)
        status: list = [1] * len(self.ctxs)

        def work(ctx, g, lo, hi):
            parts[g], status[g] = ctx.rlc_partial(signatures[lo:hi], messages[lo:hi], seed, index_base=lo)

        self._run_sharded(n, work)
        bad = [s for s in status if s != 1]
        if bad:
            return bad[0]
        got = [p for p in parts if p is not None]
        return self.ctxs[0].rlc_combine(got) if got else 1

    def close(self):
        for c in self.ctxs:
            c.close()


class MultiIssuerVerifier:
    """Batches with a public key PER ITEM (SURVEY 8f rank 4: "multi-issuer batches") on top of `api.IssuerSet`
    (`bbs_issuer_set_create` / `bbs_verify_batch_multi`): the distinct keys of a batch are registered once (the generator
    tables are shared, a key costs ~26 KB), items carry an index into the set, one call verifies the whole mixed batch.
    Per item the result is exactly `PublicKey::verify` under that item's key (verify.rs:18-30).  A new key rebuilds the
    set (all keys are processed in parallel on the GPU, one thread per key)."""

    def __init__(self, suite: Ciphersuite, header: bytes, n_messages: int, device: int = 0, lib_path: Optional[str] = None):
        self.suite, self.header, self.n_messages = suite, header, n_messages
        self.device, self.lib_path = device, lib_path
        self.index: dict = {}
        self.keys: list = []
        self.set: Optional[IssuerSet] = None

    def _ensure(self, pks: Sequence[bytes]):
        new = [bytes(pk) for pk in dict.fromkeys(bytes(pk) for pk in pks) if bytes(pk) not in self.index]
        if new or self.set is None:
            for pk in new:
                self.index[pk] = len(self.keys)
                self.keys.append(pk)
            if self.set is not None:
                self.set.close()
            self.set = IssuerSet(self.suite, self.keys, self.header, self.n_messages, device=self.device, lib_path=self.lib_path)

    def verify_batch(self, pks: Sequence[bytes], signatures: Sequence[bytes], messages: Sequence[Sequence[bytes]]) -> np.ndarray:
        """status[i] = verify of signatures[i] over messages[i] under pks[i] (compressed G2)"""
        self._ensure(pks)
        return self.set.verify_batch([self.index[bytes(pk)] for pk in pks], b"".join(bytes(x) for x in signatures), messages)

    def close(self):
        if self.set is not None:
            self.set.close()
            self.set = None
