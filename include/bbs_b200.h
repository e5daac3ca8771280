/* bbs_b200.h -- C ABI of the B200-native batch engine for the BBS verification hot path of
 * hashcloak/bbs_sign (`bbs_plus` crate).  Plain pointers and sizes only; every entry point names the
 * reference interface (file:line under /root/reference) it replaces for a whole batch.
 *
 * The reference has no FFI of its own (pure generic Rust); this header is the boundary the north star
 * asks for: the Rust side (`verify_batch`, `proof_verify_batch`, `sign_batch`, see INTEGRATION.md) binds
 * exactly these symbols.  All arithmetic runs on the GPU (sm_100a); there is no CPU fallback: without a
 * CUDA device every call returns BBS_E_CUDA.
 *
 * Wire formats are the reference's own `CanonicalSerialize` encodings (SURVEY Appendix A):
 *   scalar      : 32 bytes little-endian, canonical (< r)
 *   G1 / G2     : ark `serialize_compressed` -- BLS12-381: 48 / 96 bytes zcash format;
 *                 BN254: 32 / 64 bytes arkworks SW format
 *   Signature   : comp(A) || LE32(e)                                   (src/sign.rs:18-22)
 *   Proof fixed : comp(Abar) || comp(Bbar) || comp(D) || LE32(e^) || LE32(r1^) || LE32(r3^) || LE32(c)
 *                 (the fixed-size fields of src/proof_gen.rs:29-39; commitments travel separately)
 *
 * Threading: one context per (GPU, issuer key, header, L), or per (GPU, issuer key, L) for the *_hdr calls, which take a header
 * per item on a context created with BBS_CTX_PER_ITEM_HEADER.  A context is SINGLE-STREAM: every call on it (host-buffer or
 * *_dev) shares the context's grow-only device scratch, so calls on one context must be serialized by the caller and
 * consecutive *_dev calls on one context must use the same stream (or be ordered by the caller's events).  Different
 * contexts are independent (one host thread per GPU for multi-GPU sharding).
 *
 * Sizes: n and n * n_msgs (and every flat count) must fit in 32 bits; larger batches return BBS_E_ARG and must be split.
 *
 * Validation: every G1 / G2 encoding that enters (signatures, proofs, generators, public key) is checked like ark-serialize
 * `deserialize_compressed` (Validate::Yes: derived for Signature src/sign.rs:18, Proof src/proof_gen.rs:29, PublicKey
 * src/key_gen.rs:12): canonical x, flags, on the curve AND in the prime-order subgroup.  Failures: BBS_ST_ERR_MALFORMED
 * per item, BBS_E_ARG from bbs_ctx_create.
 *
 * Secrets: the signing key is copied into a device buffer that is cleared when the call's kernel has run, shared memory
 * that held sk-derived values is zeroed by the kernel, and the staged messages / scalars are wiped after signing and at
 * bbs_ctx_destroy (the reference's SecretKey is Zeroize + ZeroizeOnDrop, src/key_gen.rs:29).
 */
#ifndef BBS_B200_H
#define BBS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bbs_ctx bbs_ctx;
typedef struct bbs_issuer_set bbs_issuer_set;

/* curve_id: the reference's type parameter E (with its C / H / F companions) */
#define BBS_CURVE_BLS12_381 1 /* Bls12_381 + Bls12381Const + HashToG1Bls12381  (src/constants.rs:63-89) */
#define BBS_CURVE_BN254 2     /* Bn254 + Bn254Const + HashToG1Bn254            (src/constants.rs:27-61) */

/* return codes */
#define BBS_OK 0
#define BBS_E_ARG (-1)       /* null pointer, bad curve id, L too large, undecodable key or generator */
#define BBS_E_CUDA (-2)      /* CUDA runtime error (no device, out of memory, launch failure) */

/* per-item status bytes */
#define BBS_ST_REJECT 0              /* Ok(false) */
#define BBS_ST_ACCEPT 1              /* Ok(true)  */
#define BBS_ST_ERR_MSG_GEN_LEN 2     /* Err(InvalidMessageAndGeneratorsLength)  src/sign.rs:24-28, src/proof_gen.rs:66 */
#define BBS_ST_ERR_DISCLOSED_INDEX 3 /* Err(InvalidDisclosedIndex)              src/proof_gen.rs:62-65 */
#define BBS_ST_ERR_IDX_MSG_LEN 4     /* Err(InvalidIndicesAndMessagesLength)    src/proof_gen.rs:72-74 */
#define BBS_ST_ERR_MALFORMED 5       /* undecodable point (bad flags, x >= p, not on the curve, not in the prime-order
                                        subgroup), scalar >= r, or an input on which the reference panics (duplicate
                                        disclosed index src/proof_verify.rs:179; sk+e == 0 src/sign.rs:129) */

#define BBS_ST_ERR_DISCLOSED_LEN 6   /* Err(InvalidDisclosedIndicesLength)      src/proof_gen.rs:139-141 */
#define BBS_ST_ERR_RANDOM_LEN 7      /* Err(InvalidRandomScalarsAndUndisclosedIndicesLength)  src/proof_gen.rs:232-234 */

#define BBS_MAX_MESSAGES 256

/* Sizes of the encodings for a curve (bytes). */
size_t bbs_g1_bytes(int curve_id);
size_t bbs_g2_bytes(int curve_id);
size_t bbs_signature_bytes(int curve_id);   /* g1 + 32 */
size_t bbs_proof_fixed_bytes(int curve_id); /* 3*g1 + 4*32 */

/* Last error text of the calling thread ("" if none). */
const char* bbs_last_error(void);

/* What this library was compiled as: "cuda sm_100a" for the product, anything else (the host simulation that the
 * GPU-less logic tests build from the same sources) must never be bound by a product loader. */
const char* bbs_build_info(void);

/* create_generators(count, api_id) (src/utils/interface_utilities.rs:47-73) on the device, with the suite's hash-to-G1
 * (:24-44: BLS12381G1_XMD:SHA-256_SSWU_RO_ / BN254G1_XMD:SHA-256_SVDW_RO_): out = count compressed G1 points
 * Q1, H_1, .., H_{count-1}, ready for bbs_ctx_create. */
int bbs_create_generators(int curve_id, int device, const uint8_t* api_id, size_t api_id_len, uint32_t count,
                          uint8_t* out);

/* Builds the per-issuer state on `device`:
 *   decodes `pk` (G2) and the `n_generators` = L+1 generators Q1, H_1..H_L (G1) -- the `generators: &[E::G1]`
 *   argument of core_verify / core_sign / core_proof_verify (src/verify.rs:53-60, src/sign.rs:63-69,
 *   src/proof_verify.rs:64-73); computes `calculate_domain` (src/utils/core_utilities.rs:24-63) for
 *   (pk, generators, header, api_id) once; K = P1 + Q1*domain; fixed-base window tables for K and
 *   every H_j (16-bit windows over GLV half scalars: 50 MB per generator on BLS12-381, 34 MB on BN254);
 *   and the Miller-loop line tables of pk and BP2.
 * `api_id` is the reference's `api_id` (CIPHERSUITE_ID || "H2G_HM2S_" in the interface functions,
 * arbitrary in the core tests).  Identity pk is allowed (the reference returns Ok(false) for it).
 * Generators must be non-identity points of G1. */
int bbs_ctx_create(int curve_id, int device, const uint8_t* pk, const uint8_t* generators, uint32_t n_generators,
                   const uint8_t* header, size_t header_len, const uint8_t* api_id, size_t api_id_len,
                   bbs_ctx** out);
/* The same with creation flags:
 *   BBS_CTX_SMALL_TABLES  8-bit windows instead of 16-bit: 390 KB (BLS12-381) / 260 KB (BN254) of table per generator instead of
 *                         50 / 34 MB -- the whole table set stays resident in L2, the context is built ~100x faster and
 *                         thousands of (key, header, L) contexts fit in HBM -- for twice the fixed-base additions per item
 *                         (the G1 kernels run ~1.5x longer; results are identical).
 *   BBS_CTX_PER_ITEM_HEADER  the context can also serve the *_hdr calls (a header per item, below): it adds a window table for
 *                         Q1 in generator slot L + 1 (+50 MB on BLS12-381, +34 MB on BN254; ~390 / 260 KB with small tables)
 *                         and keeps the SHA-256 state of calculate_domain after its header-independent prefix.  The
 *                         context's own header, domain and K are built as without the flag and serve every other call.
 * The two flags may be combined. */
#define BBS_CTX_SMALL_TABLES 1u
#define BBS_CTX_PER_ITEM_HEADER 2u
int bbs_ctx_create_ex(int curve_id, int device, uint32_t flags, const uint8_t* pk, const uint8_t* generators,
                      uint32_t n_generators, const uint8_t* header, size_t header_len, const uint8_t* api_id,
                      size_t api_id_len, bbs_ctx** out);
void bbs_ctx_destroy(bbs_ctx* ctx);

/* 32-byte little-endian domain scalar of the context (src/utils/core_utilities.rs:24-63). */
int bbs_ctx_domain(bbs_ctx* ctx, uint8_t out_le32[32]);

/* ---- host-buffer entry points (copies inside) ---------------------------------------------------- */

/* msg_to_scalars (src/utils/interface_utilities.rs:76-88) for `count` messages:
 * message t = msgs[offsets[t] .. offsets[t+1]); out = count x LE32. */
int bbs_msg_to_scalars(bbs_ctx* ctx, size_t count, const uint8_t* msgs, const uint64_t* offsets, uint8_t* out);

/* PublicKey::core_verify (src/verify.rs:53-93) for n signatures, each over `n_msgs` scalar messages.
 * status[i] in {ACCEPT, REJECT, ERR_MSG_GEN_LEN (n_msgs != L), ERR_MALFORMED}. */
int bbs_core_verify_batch(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msg_scalars, uint32_t n_msgs,
                          uint8_t* status);

/* PublicKey::verify (src/verify.rs:18-50): byte messages; item i owns messages i*n_msgs .. (i+1)*n_msgs-1,
 * message t = msgs[offsets[t] .. offsets[t+1]), offsets has n*n_msgs + 1 entries. */
int bbs_verify_batch(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* offsets,
                     uint32_t n_msgs, uint8_t* status);

/* SecretKey::core_sign (src/sign.rs:63-133): sigs_out = n x Signature; b_out (may be NULL) = n x comp(B),
 * the B point of src/sign.rs:120-126.  The context's pk must be sk*BP2 (the reference derives pk from sk,
 * src/sign.rs:81).  status[i] = ACCEPT on success. */
int bbs_core_sign_batch(bbs_ctx* ctx, const uint8_t sk_le32[32], size_t n, const uint8_t* msg_scalars,
                        uint32_t n_msgs, uint8_t* sigs_out, uint8_t* b_out, uint8_t* status);

/* SecretKey::sign (src/sign.rs:32-60): byte messages, layout as bbs_verify_batch. */
int bbs_sign_batch(bbs_ctx* ctx, const uint8_t sk_le32[32], size_t n, const uint8_t* msgs, const uint64_t* offsets,
                   uint32_t n_msgs, uint8_t* sigs_out, uint8_t* b_out, uint8_t* status);

/* core_proof_verify (src/proof_verify.rs:64-116) for n proofs.
 *   proofs_fixed     : n x Proof-fixed encoding (above)
 *   commitments      : flat LE32 scalars; proof i owns commitments[commit_off[i] .. commit_off[i+1])
 *   disclosed_idx    : flat indexes; proof i discloses disclosed_idx[dis_off[i] .. dis_off[i+1])
 *   disclosed_scalars: flat LE32 message scalars, same indexing as disclosed_idx
 *   ph               : presentation header shared by the batch
 * status[i] in {ACCEPT, REJECT, ERR_DISCLOSED_INDEX, ERR_MSG_GEN_LEN, ERR_MALFORMED}. */
int bbs_core_proof_verify_batch(bbs_ctx* ctx, size_t n, const uint8_t* proofs_fixed, const uint8_t* commitments,
                                const uint64_t* commit_off, const uint32_t* disclosed_idx,
                                const uint8_t* disclosed_scalars, const uint64_t* dis_off, const uint8_t* ph,
                                size_t ph_len, uint8_t* status);

/* proof_verify (src/proof_verify.rs:19-61): disclosed messages as bytes;
 * disclosed message k (flat numbering, same as disclosed_idx) = dis_msgs[dis_msg_off[k] .. dis_msg_off[k+1]). */
int bbs_proof_verify_batch(bbs_ctx* ctx, size_t n, const uint8_t* proofs_fixed, const uint8_t* commitments,
                           const uint64_t* commit_off, const uint32_t* disclosed_idx, const uint8_t* dis_msgs,
                           const uint64_t* dis_msg_off, const uint64_t* dis_off, const uint8_t* ph, size_t ph_len,
                           uint8_t* status);

/* core_proof_gen (src/proof_gen.rs:116-365: proof_init, proof_challenge_calculate, proof_finalize) for n signatures.
 *   sigs, msg_scalars : as bbs_core_verify_batch (ALL n_msgs message scalars of every item)
 *   disclosed_idx     : flat indexes, item i discloses disclosed_idx[dis_off[i] .. dis_off[i+1]) (duplicates are
 *                       de-duplicated and the set is sorted, as the reference does, :154-158)
 *   random_scalars    : flat LE32; item i owns random_scalars[rand_off[i] .. rand_off[i+1]) = 5 + U_i scalars in the
 *                       order of proof_init (:254-263).  The reference draws them from the thread RNG
 *                       (`calculate_random_scalars`) or the mocked stream (feature testvector_bls12_381); here the
 *                       caller supplies them, so a proof is a deterministic function of its inputs.
 *   commit_off        : n+1 offsets (in scalars) into commitments_out; U_i = commit_off[i+1] - commit_off[i] must be
 *                       n_msgs - |disclosed set|
 *   outputs           : proofs_fixed_out = n x Proof-fixed encoding, commitments_out = flat LE32 (the two halves of
 *                       ark's serialisation of Proof, the format bbs_proof_verify_batch consumes)
 * status[i] in {ACCEPT (= Ok(proof)), ERR_DISCLOSED_LEN, ERR_DISCLOSED_INDEX, ERR_MSG_GEN_LEN, ERR_RANDOM_LEN,
 *               ERR_MALFORMED}. */
int bbs_core_proof_gen_batch(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msg_scalars, uint32_t n_msgs,
                             const uint32_t* disclosed_idx, const uint64_t* dis_off, const uint8_t* random_scalars,
                             const uint64_t* rand_off, const uint64_t* commit_off, const uint8_t* ph, size_t ph_len,
                             uint8_t* proofs_fixed_out, uint8_t* commitments_out, uint8_t* status);
/* proof_gen (src/proof_gen.rs:78-113): byte messages, layout as bbs_verify_batch. */
int bbs_proof_gen_batch(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* offsets,
                        uint32_t n_msgs, const uint32_t* disclosed_idx, const uint64_t* dis_off,
                        const uint8_t* random_scalars, const uint64_t* rand_off, const uint64_t* commit_off,
                        const uint8_t* ph, size_t ph_len, uint8_t* proofs_fixed_out, uint8_t* commitments_out,
                        uint8_t* status);

/* ---- per-item headers and presentation headers -----------------------------------------------------------------
 * In the reference `header` and `ph` are arguments of every call (src/verify.rs:18-30, src/sign.rs:32-43,
 * src/proof_verify.rs:19-34); these calls take them per item.  Item i's result is the reference's for header_i / ph_i;
 * statuses are those of the calls without _hdr.
 *   headers, hdr_off : header i = headers[hdr_off[i] .. hdr_off[i+1]), n + 1 offsets.  The verify and sign calls require
 *                      them and a context created with BBS_CTX_PER_ITEM_HEADER (else BBS_E_ARG); the proof calls accept
 *                      NULL for both, meaning the context's header for every item, and then work on any context.
 *   phs, ph_off      : the proof calls' presentation headers, ph i = phs[ph_off[i] .. ph_off[i+1]) (required).
 * Offsets must not decrease and every header / ph must be shorter than 2^28 bytes (BBS_E_ARG).  Per item the library hashes
 * calculate_domain from the context's stored prefix state and computes K_i = P1 + Q1 * domain_i (one extra kernel,
 * profiled in the slot after the call's others).  Per-item-header proof verification always takes the task-split G1 path
 * (as issuer sets do).  These calls never take the chunked pipelines of large host-buffer batches: any size runs in one
 * shot, with the same results. */
int bbs_core_verify_batch_hdr(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msg_scalars, uint32_t n_msgs,
                              const uint8_t* headers, const uint64_t* hdr_off, uint8_t* status);
int bbs_verify_batch_hdr(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* offsets,
                         uint32_t n_msgs, const uint8_t* headers, const uint64_t* hdr_off, uint8_t* status);
int bbs_core_sign_batch_hdr(bbs_ctx* ctx, const uint8_t sk_le32[32], size_t n, const uint8_t* msg_scalars, uint32_t n_msgs,
                            const uint8_t* headers, const uint64_t* hdr_off, uint8_t* sigs_out, uint8_t* b_out,
                            uint8_t* status);
int bbs_sign_batch_hdr(bbs_ctx* ctx, const uint8_t sk_le32[32], size_t n, const uint8_t* msgs, const uint64_t* offsets,
                       uint32_t n_msgs, const uint8_t* headers, const uint64_t* hdr_off, uint8_t* sigs_out, uint8_t* b_out,
                       uint8_t* status);
int bbs_core_proof_verify_batch_hdr(bbs_ctx* ctx, size_t n, const uint8_t* proofs_fixed, const uint8_t* commitments,
                                    const uint64_t* commit_off, const uint32_t* disclosed_idx,
                                    const uint8_t* disclosed_scalars, const uint64_t* dis_off, const uint8_t* headers,
                                    const uint64_t* hdr_off, const uint8_t* phs, const uint64_t* ph_off, uint8_t* status);
int bbs_proof_verify_batch_hdr(bbs_ctx* ctx, size_t n, const uint8_t* proofs_fixed, const uint8_t* commitments,
                               const uint64_t* commit_off, const uint32_t* disclosed_idx, const uint8_t* dis_msgs,
                               const uint64_t* dis_msg_off, const uint64_t* dis_off, const uint8_t* headers,
                               const uint64_t* hdr_off, const uint8_t* phs, const uint64_t* ph_off, uint8_t* status);
int bbs_core_proof_gen_batch_hdr(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msg_scalars, uint32_t n_msgs,
                                 const uint32_t* disclosed_idx, const uint64_t* dis_off, const uint8_t* random_scalars,
                                 const uint64_t* rand_off, const uint64_t* commit_off, const uint8_t* headers,
                                 const uint64_t* hdr_off, const uint8_t* phs, const uint64_t* ph_off,
                                 uint8_t* proofs_fixed_out, uint8_t* commitments_out, uint8_t* status);
int bbs_proof_gen_batch_hdr(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* offsets,
                            uint32_t n_msgs, const uint32_t* disclosed_idx, const uint64_t* dis_off,
                            const uint8_t* random_scalars, const uint64_t* rand_off, const uint64_t* commit_off,
                            const uint8_t* headers, const uint64_t* hdr_off, const uint8_t* phs, const uint64_t* ph_off,
                            uint8_t* proofs_fixed_out, uint8_t* commitments_out, uint8_t* status);

/* ---- multi-issuer batches ---------------------------------------------------------------------------------
 * In the reference the public key is `&self` of every call (src/verify.rs:18-30), so a stream of signatures may name a
 * different issuer per item.  An issuer set holds n_issuers keys over ONE generator list / header / api_id: what depends
 * only on (suite, api_id, L) -- the decoded generators and their fixed-base tables -- is built once and shared; per key
 * it keeps W, calculate_domain (src/utils/core_utilities.rs:24-63), K = P1 + Q1 * domain and the Miller-loop lines of W:
 * about 26 KB (BLS12-381) / 17 KB (BN254) per issuer instead of a whole context, so tens of thousands of issuers fit.
 *   pks           : n_issuers x compressed G2
 *   issuer_status : n_issuers bytes out: ACCEPT = key usable, ERR_MALFORMED = what ark `PublicKey::deserialize_compressed`
 *                   refuses (bad flags, not on the twist, not in the subgroup) -- every item naming such an issuer gets
 *                   ERR_MALFORMED.  (A key whose ate walk meets a line through the origin, probability ~2^-380, is
 *                   reported the same way; verify such a key through its own bbs_ctx_create context.)
 * bbs_verify_batch_multi / bbs_core_verify_batch_multi: item i is `pks[item_issuer[i]].verify(..)` /
 * `.core_verify(..)`; everything else as bbs_verify_batch / bbs_core_verify_batch (item_issuer[i] >= n_issuers gives
 * ERR_MALFORMED).  bbs_issuer_set_memory_bytes returns the bytes that grow with the number of issuers and, in
 * *shared_bytes, the shared part. */
int bbs_issuer_set_create(int curve_id, int device, size_t n_issuers, const uint8_t* pks, const uint8_t* generators,
                          uint32_t n_generators, const uint8_t* header, size_t header_len, const uint8_t* api_id,
                          size_t api_id_len, uint8_t* issuer_status, bbs_issuer_set** out);
void bbs_issuer_set_destroy(bbs_issuer_set* set);
uint64_t bbs_issuer_set_memory_bytes(bbs_issuer_set* set, uint64_t* shared_bytes);
int bbs_verify_batch_multi(bbs_issuer_set* set, size_t n, const uint32_t* item_issuer, const uint8_t* sigs,
                           const uint8_t* msgs, const uint64_t* offsets, uint32_t n_msgs, uint8_t* status);
int bbs_core_verify_batch_multi(bbs_issuer_set* set, size_t n, const uint32_t* item_issuer, const uint8_t* sigs,
                                const uint8_t* msg_scalars, uint32_t n_msgs, uint8_t* status);
/* bbs_proof_verify_batch_multi / bbs_core_proof_verify_batch_multi: proof i is `pks[item_issuer[i]].proof_verify(..)`
 * (src/proof_verify.rs:19-34) / core_proof_verify under that key; everything else as bbs_proof_verify_batch /
 * bbs_core_proof_verify_batch.  The issuer enters through its domain (challenge, src/proof_gen.rs:272-328),
 * K_i = P1 + Q1 * domain_i (the K_i * c term of proof_verify_init, :165, a variable-base product here) and the lines of W_i. */
int bbs_core_proof_verify_batch_multi(bbs_issuer_set* set, size_t n, const uint32_t* item_issuer, const uint8_t* proofs_fixed,
                                      const uint8_t* commitments, const uint64_t* commit_off, const uint32_t* disclosed_idx,
                                      const uint8_t* disclosed_scalars, const uint64_t* dis_off, const uint8_t* ph,
                                      size_t ph_len, uint8_t* status);
int bbs_proof_verify_batch_multi(bbs_issuer_set* set, size_t n, const uint32_t* item_issuer, const uint8_t* proofs_fixed,
                                 const uint8_t* commitments, const uint64_t* commit_off, const uint32_t* disclosed_idx,
                                 const uint8_t* dis_msgs, const uint64_t* dis_msg_off, const uint64_t* dis_off,
                                 const uint8_t* ph, size_t ph_len, uint8_t* status);

/* ---- random-linear-combination batch mode (the optional mode of the north star; not in the reference) ----------
 * One verdict for n signatures under the context's issuer key:
 *     e( sum r_i A_i , W ) * e( sum r_i (e_i A_i - B_i) , BP2 ) == 1,   B_i as in src/verify.rs:81-86,
 * r_i = the first 16 bytes, as a big-endian integer, of SHA-256(seed || BE64(index_base + i)) (1 if that is 0).
 * ACCEPT means every item verifies except with probability 2^-128 over the seed; REJECT means at least one item does
 * not; ERR_MALFORMED / ERR_MSG_GEN_LEN as in bbs_core_verify_batch.
 * THE SEED MUST BE UNPREDICTABLE TO WHOEVER SUBMITS THE BATCH.  With a known seed three colluding items
 * (A_i + a_i X with sum r_i a_i = sum r_i e_i a_i = 0) pass although none verifies, and deriving r_i from the item's own
 * bytes does not help (a generalised-birthday search over a large batch finds such a_i).  Therefore:
 *   - bbs_rlc_[core_]verify_batch: pass seed = NULL and the library draws 32 bytes from the OS CSPRNG after it has received
 *     the batch (the safe default; an explicit seed is for reproducible tests);
 *   - sharded use (bbs_rlc_partial* on every GPU + bbs_rlc_combine): the coordinator draws ONE fresh seed after the
 *     whole batch is fixed and hands it to every shard; it is never reused and never revealed before that.
 * Sharding: every GPU reduces its shard to two compressed G1 points with bbs_rlc_partial[_core] (index_base = the
 * shard's first global index); bbs_rlc_combine adds the shards' points on one GPU and does the single pairing check.
 * bbs_rlc_[core_]verify_batch = one shard + combine. */
int bbs_rlc_partial_core(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msg_scalars, uint32_t n_msgs,
                         const uint8_t seed[32], uint64_t index_base, uint8_t* parts_out /* 2 x G1 */, uint8_t* status);
int bbs_rlc_partial(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* offsets,
                    uint32_t n_msgs, const uint8_t seed[32], uint64_t index_base, uint8_t* parts_out, uint8_t* status);
int bbs_rlc_combine(bbs_ctx* ctx, size_t n_parts, const uint8_t* parts /* n_parts x 2 x G1 */, uint8_t* verdict);
int bbs_rlc_core_verify_batch(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msg_scalars, uint32_t n_msgs,
                              const uint8_t* seed32_or_null, uint8_t* verdict);
int bbs_rlc_verify_batch(bbs_ctx* ctx, size_t n, const uint8_t* sigs, const uint8_t* msgs, const uint64_t* offsets,
                         uint32_t n_msgs, const uint8_t* seed32_or_null, uint8_t* verdict);

/* Proof verification with the pairing half by one random linear combination.  Arguments as bbs_[core_]proof_verify_batch
 * and bbs_[core_]proof_verify_batch_hdr (per-item phs, NULL headers = the context's header), plus:
 *   seed32_or_null : the coefficient seed; r_i = the first 16 bytes, as a big-endian integer, of SHA-256(seed || BE64(i))
 *                    (1 if that is 0), i = the item's position in the call.  NULL: the library draws 32 bytes from the OS
 *                    CSPRNG after it has received the batch.
 *   status[i]      : what the call without rlc_ returns for item i.  An ACCEPT holds except with probability 2^-128 over
 *                    the seed; every other status is exact.
 *   combined       : (may be NULL) ACCEPT when the one combined check held for every item that reached the pairing, or
 *                    when no item did; REJECT when it failed and the per-item pairing decided those items instead.
 * After the G1 half (challenge comparison, Err variants, malformed input: exact per item, as in the call without rlc_),
 * every proof that reaches the pairing is checked at once by
 *     e( sum r_i Abar_i , W ) * e( sum r_i (-Bbar_i) , BP2 ) == 1
 * one bucket MSM and one pairing for the batch.  If that fails, the per-item pairing kernel decides the same items, so
 * the statuses stay exact at about the cost of the call without rlc_; `combined` tells a caller that this happened.
 * THE SEED MUST BE UNPREDICTABLE TO WHOEVER SUBMITS THE BATCH: with a known seed, two proofs whose pairing checks fail
 * can be built so that their failures cancel in the sum, and both are accepted.  Pass NULL; an explicit seed is for
 * reproducible tests.  One issuer key per call (no issuer sets).  n must be below 2^31. */
int bbs_rlc_core_proof_verify_batch(bbs_ctx* ctx, size_t n, const uint8_t* proofs_fixed, const uint8_t* commitments,
                                    const uint64_t* commit_off, const uint32_t* disclosed_idx,
                                    const uint8_t* disclosed_scalars, const uint64_t* dis_off, const uint8_t* ph,
                                    size_t ph_len, const uint8_t* seed32_or_null, uint8_t* status, uint8_t* combined);
int bbs_rlc_proof_verify_batch(bbs_ctx* ctx, size_t n, const uint8_t* proofs_fixed, const uint8_t* commitments,
                               const uint64_t* commit_off, const uint32_t* disclosed_idx, const uint8_t* dis_msgs,
                               const uint64_t* dis_msg_off, const uint64_t* dis_off, const uint8_t* ph, size_t ph_len,
                               const uint8_t* seed32_or_null, uint8_t* status, uint8_t* combined);
int bbs_rlc_core_proof_verify_batch_hdr(bbs_ctx* ctx, size_t n, const uint8_t* proofs_fixed, const uint8_t* commitments,
                                        const uint64_t* commit_off, const uint32_t* disclosed_idx,
                                        const uint8_t* disclosed_scalars, const uint64_t* dis_off, const uint8_t* headers,
                                        const uint64_t* hdr_off, const uint8_t* phs, const uint64_t* ph_off,
                                        const uint8_t* seed32_or_null, uint8_t* status, uint8_t* combined);
int bbs_rlc_proof_verify_batch_hdr(bbs_ctx* ctx, size_t n, const uint8_t* proofs_fixed, const uint8_t* commitments,
                                   const uint64_t* commit_off, const uint32_t* disclosed_idx, const uint8_t* dis_msgs,
                                   const uint64_t* dis_msg_off, const uint64_t* dis_off, const uint8_t* headers,
                                   const uint64_t* hdr_off, const uint8_t* phs, const uint64_t* ph_off,
                                   const uint8_t* seed32_or_null, uint8_t* status, uint8_t* combined);

/* ---- device-buffer entry points (no copies; all pointers are device pointers on the context's GPU;
 *      work is enqueued on `stream` (a cudaStream_t, NULL = default stream) and NOT synchronized) ------ */
int bbs_msg_to_scalars_dev(bbs_ctx* ctx, size_t count, const uint8_t* d_msgs, const uint64_t* d_offsets,
                           uint8_t* d_out, void* stream);
int bbs_core_verify_batch_dev(bbs_ctx* ctx, size_t n, const uint8_t* d_sigs, const uint8_t* d_msg_scalars,
                              uint32_t n_msgs, uint8_t* d_status, void* stream);
int bbs_verify_batch_dev(bbs_ctx* ctx, size_t n, const uint8_t* d_sigs, const uint8_t* d_msgs,
                         const uint64_t* d_offsets, uint32_t n_msgs, uint8_t* d_status, void* stream);
int bbs_core_sign_batch_dev(bbs_ctx* ctx, const uint8_t sk_le32[32], size_t n, const uint8_t* d_msg_scalars,
                            uint32_t n_msgs, uint8_t* d_sigs_out, uint8_t* d_b_out, uint8_t* d_status, void* stream);
int bbs_core_proof_verify_batch_dev(bbs_ctx* ctx, size_t n, const uint8_t* d_proofs_fixed,
                                    const uint8_t* d_commitments, const uint64_t* d_commit_off,
                                    const uint32_t* d_disclosed_idx, const uint8_t* d_disclosed_scalars,
                                    const uint64_t* d_dis_off, const uint8_t* d_ph, size_t ph_len,
                                    uint8_t* d_status, void* stream);

/* Device-buffer forms of bbs_core_verify_batch_hdr / bbs_core_proof_verify_batch_hdr (offsets in device memory, not checked). */
int bbs_core_verify_batch_hdr_dev(bbs_ctx* ctx, size_t n, const uint8_t* d_sigs, const uint8_t* d_msg_scalars,
                                  uint32_t n_msgs, const uint8_t* d_headers, const uint64_t* d_hdr_off, uint8_t* d_status,
                                  void* stream);
int bbs_core_proof_verify_batch_hdr_dev(bbs_ctx* ctx, size_t n, const uint8_t* d_proofs_fixed,
                                        const uint8_t* d_commitments, const uint64_t* d_commit_off,
                                        const uint32_t* d_disclosed_idx, const uint8_t* d_disclosed_scalars,
                                        const uint64_t* d_dis_off, const uint8_t* d_headers, const uint64_t* d_hdr_off,
                                        const uint8_t* d_phs, const uint64_t* d_ph_off, uint8_t* d_status, void* stream);

/* Number of kernels the library has launched on this context since creation (for bench accounting). */
uint64_t bbs_ctx_launch_count(bbs_ctx* ctx);
/* Device memory the context holds (tables, key state and the grow-only batch scratch), bytes. */
uint64_t bbs_ctx_memory_bytes(bbs_ctx* ctx);

/* ---- test hooks (CUDA kernels either way; results are identical) ---------------------------------------
 * bbs_ctx_use_per_thread_pairing: run the pairing check with the one-thread-per-item kernel that a context with a
 *   degenerate line (a tangent / chord of the public key's ate walk through the origin; impossible for an honest key)
 *   falls back to, instead of the cooperative role-warp kernel.
 * bbs_ctx_set_rlc_windows: digits per 128-bit value of the bucket MSM of the random-linear-combination mode
 *   (8..32; 0 = the cost model's choice).
 * bbs_ctx_set_g1_split: verify / core_verify batches of up to max_items items run their G1 half as two tasks per item
 *   (variable-base and fixed-base part in parallel, then a join) instead of one thread per item; the default is SIZE_MAX
 *   (always: it is faster at every batch size measured), 0 selects the one-thread-per-item kernel.
 * bbs_ctx_set_pairing_split: batches of up to max_items (<= 32, the default) items run the cooperative pairing kernel with
 *   TWO warps per role (a batch that fits one 32-item group is latency-bound: about half the time); 0 = always one. */
int bbs_ctx_use_per_thread_pairing(bbs_ctx* ctx, int on);
int bbs_ctx_set_rlc_windows(bbs_ctx* ctx, uint32_t windows);
int bbs_ctx_set_g1_split(bbs_ctx* ctx, size_t max_items);
int bbs_ctx_set_pairing_split(bbs_ctx* ctx, size_t max_items);

/* ---- measurement hooks ------------------------------------------------------------------------------
 * With profiling on, every *_dev batch call records CUDA events on its launching stream around each of its
 * kernels; bbs_ctx_kernel_times returns the durations (ms) of the last call in launch order:
 *   verify / proof verify: [msg_to_scalars (0 if absent), G1 kernel, pairing kernel];  sign: [h2s, sign].
 * The *_hdr calls with per-item headers append the per-item domain kernel: verify / proof verify slot 3, sign slot 2.
 * bbs_rlc_*proof_verify_batch*: [msg_to_scalars, G1 kernels, prep, scan + scatter, buckets, reduction, finish, combined
 *   pairing, acceptance or per-item pairing]; the scan slot and the combined-pairing slot also hold the host's read of one
 *   word (whether any item reached the pairing; the verdict).  Slots 3..8 are 0 when no item reached the pairing;
 *   per-item headers: slot 9. */
int bbs_ctx_set_profiling(bbs_ctx* ctx, int on);
int bbs_ctx_kernel_times(bbs_ctx* ctx, float* ms, int n);
/* Integer-multiply roofline probe: 8 independent multiply-accumulate chains per thread on every SM.
 * mode 0: one mad.lo.u32 + one mad.hi.u32 per product; mode 1: one mad.wide.u32 (IMAD.WIDE) per product.
 * Returns the measured rate of full 32x32->64 products in 1e9 products/s and the kernel time. */
int bbs_imad_peak(int device, int iters, int mode, double* gprod_per_s, float* ms);

/* ---- arithmetic self-test hooks (parity tests of the field / curve layers against the oracle) ------
 * op: 0 = Fp mul, 1 = Fp add, 2 = Fp sub, 3 = Fp inv, 4 = Fp sqrt (0 if none), 5 = Fr mul, 6 = Fr inv,
 *     7 = Fp inv / 8 = Fr inv by the variable-time binary Euclid used where one thread inverts public data,
 *     9 = Fp square (fe_sqr: on the device the dedicated squaring of the base fields), 10 = Fp neg,
 *     11 = Fr add, 12 = Fr sub, 13 = Fr neg.  Unary ops ignore b.
 * op | 0x100: Montgomery-domain I/O.  a, b and out are the Montgomery words A, B, op(...)·R mod m themselves (no
 *     conversion on the way in or out), so out = mont(op(A·R^-1, B·R^-1)) with R = 2^(32N).  Without the flag a chosen
 *     value is multiplied by R before the operation and its limb pattern is lost.
 * a, b, out: n x field-size little-endian values below the modulus (48 / 32 bytes for Fp, 32 for Fr). */
int bbs_selftest_field(int curve_id, int device, int op, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out);
/* out[i] = comp(k_i * P_i) for compressed G1 points and LE32 scalars. */
int bbs_selftest_g1_mul(int curve_id, int device, size_t n, const uint8_t* points, const uint8_t* scalars,
                        uint8_t* out);
/* out[i] = comp(op(...)) on the G1 group law.  Operands are Jacobian points (X, Y, Z), three canonical little-endian Fp
 * values each (48 / 32 bytes), Z = 0 the identity, so one point can be given under several Z: (l^2 x, l^3 y, l).
 * op: 0 = g1_add(p_i, q_i); 1 = g1_add_mixed(p_i, q_i), q_i read as the affine (X, Y) of a finite point (its Z ignored);
 *     2 = g1_dbl(p_i) (q ignored); 3 / 4 = the Straus product sum_j k_ij P_ij over 2 / 3 points (g1_msm_scalar):
 *     p holds 2 / 3 operands per item, read as affine (X, Y) with Z = 0 for the identity (Z's value otherwise ignored),
 *     scalars 2 / 3 canonical LE32 scalars per item (q ignored).  scalars is ignored by ops 0..2.  Other ops are refused. */
int bbs_selftest_g1(int curve_id, int device, int op, size_t n, const uint8_t* p, const uint8_t* q, const uint8_t* scalars,
                    uint8_t* out);
/* status[i] = (e(P_i, Q) * e(R_i, BP2) == 1) for compressed G1 points P_i, R_i and one compressed G2 point Q. */
int bbs_selftest_pairing(int curve_id, int device, size_t n, const uint8_t* p_points, const uint8_t* r_points,
                         const uint8_t* q_point, uint8_t* status);

#ifdef __cplusplus
}
#endif
#endif /* BBS_B200_H */
