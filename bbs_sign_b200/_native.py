"""ctypes binding of the C ABI declared in include/bbs_b200.h.

`load()` opens the CUDA library built in-tree (`bbs_sign_b200/libbbs_b200.so`) and fails loudly when
it is missing or is not a CUDA build: there is no CPU fallback on the product path.  (The GPU-less logic tests bind the
host-simulation build of the same sources with `load(path, allow_host_simulation=True)`.)"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbbs_b200.so")

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)

# every symbol include/bbs_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "bbs_g1_bytes": (C.c_size_t, [C.c_int]),
    "bbs_g2_bytes": (C.c_size_t, [C.c_int]),
    "bbs_signature_bytes": (C.c_size_t, [C.c_int]),
    "bbs_proof_fixed_bytes": (C.c_size_t, [C.c_int]),
    "bbs_last_error": (C.c_char_p, []),
    "bbs_build_info": (C.c_char_p, []),
    "bbs_create_generators": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]),
    "bbs_ctx_create": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t,
                                 C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "bbs_ctx_create_ex": (C.c_int, [C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t,
                                    C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "bbs_ctx_destroy": (None, [C.c_void_p]),
    "bbs_ctx_domain": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bbs_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
    "bbs_ctx_memory_bytes": (C.c_uint64, [C.c_void_p]),
    "bbs_issuer_set_create": (C.c_int, [C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t,
                                        C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_void_p)]),
    "bbs_issuer_set_destroy": (None, [C.c_void_p]),
    "bbs_issuer_set_memory_bytes": (C.c_uint64, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "bbs_verify_batch_multi": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                         C.c_void_p]),
    "bbs_core_verify_batch_multi": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "bbs_core_proof_verify_batch_multi": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 8 + [C.c_size_t, C.c_void_p]),
    "bbs_proof_verify_batch_multi": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 9 + [C.c_size_t, C.c_void_p]),
    "bbs_ctx_use_per_thread_pairing": (C.c_int, [C.c_void_p, C.c_int]),
    "bbs_ctx_set_rlc_windows": (C.c_int, [C.c_void_p, C.c_uint32]),
    "bbs_ctx_set_g1_split": (C.c_int, [C.c_void_p, C.c_size_t]),
    "bbs_ctx_set_pairing_split": (C.c_int, [C.c_void_p, C.c_size_t]),
    "bbs_msg_to_scalars": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bbs_core_verify_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "bbs_verify_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "bbs_core_sign_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "bbs_sign_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "bbs_core_proof_verify_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "bbs_proof_verify_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "bbs_core_proof_gen_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "bbs_proof_gen_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "bbs_core_verify_batch_hdr": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                            C.c_void_p, C.c_void_p]),
    "bbs_verify_batch_hdr": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "bbs_core_sign_batch_hdr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32] + [C.c_void_p] * 5),
    "bbs_sign_batch_hdr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 5),
    "bbs_core_proof_verify_batch_hdr": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 11),
    "bbs_proof_verify_batch_hdr": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 12),
    "bbs_core_proof_gen_batch_hdr": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 12),
    "bbs_proof_gen_batch_hdr": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
                                + [C.c_void_p] * 12),
    "bbs_core_verify_batch_hdr_dev": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 4),
    "bbs_core_proof_verify_batch_hdr_dev": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 12),
    "bbs_rlc_partial_core": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64,
                                       C.c_void_p, C.c_void_p]),
    "bbs_rlc_partial": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                  C.c_uint64, C.c_void_p, C.c_void_p]),
    "bbs_rlc_combine": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "bbs_rlc_core_verify_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                            C.c_void_p]),
    "bbs_rlc_verify_batch": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                       C.c_void_p, C.c_void_p]),
    "bbs_rlc_core_proof_verify_batch": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 7 + [C.c_size_t] + [C.c_void_p] * 3),
    "bbs_rlc_proof_verify_batch": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 8 + [C.c_size_t] + [C.c_void_p] * 3),
    "bbs_rlc_core_proof_verify_batch_hdr": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 13),
    "bbs_rlc_proof_verify_batch_hdr": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_void_p] * 14),
    "bbs_msg_to_scalars_dev": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bbs_core_verify_batch_dev": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                            C.c_void_p]),
    "bbs_verify_batch_dev": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                       C.c_void_p, C.c_void_p]),
    "bbs_core_sign_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "bbs_core_proof_verify_batch_dev": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                                  C.c_void_p, C.c_void_p]),
    "bbs_ctx_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "bbs_ctx_kernel_times": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.c_int]),
    "bbs_imad_peak": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    "bbs_selftest_field": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bbs_selftest_g1_mul": (C.c_int, [C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bbs_selftest_g1": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bbs_selftest_pairing": (C.c_int, [C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
}


class NativeLibraryMissing(RuntimeError):
    pass


_CACHE = {}


def load(path: str | None = None, allow_host_simulation: bool = False) -> C.CDLL:
    """Binds the library.  Only a CUDA build is accepted: a library whose `bbs_build_info()` is not "cuda ..." (the host
    simulation tests/hostsim.py makes from the same sources) is refused unless the caller is a test that says so
    explicitly (`allow_host_simulation=True`, tests/test_hostsim_logic.py); there is no environment-variable override."""
    path = path or LIB_PATH
    if path in _CACHE:
        return _CACHE[path]
    if not os.path.exists(path):
        raise NativeLibraryMissing(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  bbs_sign_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    info = lib.bbs_build_info().decode()
    if not info.startswith("cuda") and not allow_host_simulation:
        raise NativeLibraryMissing(f"{path} is not a CUDA build ({info}); bbs_sign_b200 has no CPU fallback")
    _CACHE[path] = lib
    return lib
