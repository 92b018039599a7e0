"""ctypes binding of include/bpe_cuda.h.  Loading fails loudly when the CUDA library is missing;
there is no Python or CPU stand-in for the engine."""
import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BPE_CUDA_LIB") or os.path.join(PKG, "libbpe_cuda.so")  # override: A/B builds of the kernels
CORPUS_LIB_PATH = os.path.join(PKG, "libbpe_corpus.so")


class Pair(C.Structure):  # == pair_t, reference bpe/inc/bpe.h:14-17
    _fields_ = [("a", C.c_uint32), ("b", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "n_input", "n_merges", "n_tokens", "ranks_applied", "same_bucket_ties", "threshold_edges", "resolver_runs",
        "census_runs", "table_rehashes", "table_capacity", "final_distinct", "kernel_launches", "replace_launches",
        "replace_bytes")] + [(n, C.c_double) for n in ("replace_ms", "ms_device", "ms_h2d", "ms_d2h", "ms_total")] + [
        ("worker_buckets", C.c_uint64 * 16)] + [(n, C.c_double) for n in ("select_ms", "apply_ms", "gap_ms")] + [
        (n, C.c_uint64) for n in ("replace_passes", "batch_merges", "batch_passes")]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n != "worker_buckets"}
        d["worker_buckets"] = list(self.worker_buckets)
        return d


EXPORTS = [
    "bpe_cuda_train", "bpe_cuda_encode", "bpe_cuda_free", "bpe_cuda_last_error", "bpe_cuda_device_count",
    "bpe_cuda_ctx_create", "bpe_cuda_ctx_destroy", "bpe_cuda_nccl_unique_id", "bpe_cuda_ctx_set_comm",
    "bpe_cuda_ctx_upload", "bpe_cuda_ctx_upload_device", "bpe_cuda_ctx_train", "bpe_cuda_ctx_encode",
    "bpe_cuda_ctx_result_sizes", "bpe_cuda_ctx_download", "bpe_cuda_ctx_device_tokens", "bpe_cuda_ctx_set_option",
    "bpe_cuda_decode", "bpe_cuda_ctx_decode", "bpe_cuda_ctx_decode_download", "bpe_cuda_ctx_decode_compare",
    "bpe_cuda_ctx_device_decoded", "bpe_cuda_train_file", "bpe_cuda_encode_file", "bpe_cuda_ctx_upload_file",
    "bpe_cuda_ctx_truncate", "bpe_cuda_ctx_download_pageable", "bpe_cuda_encode_batch", "bpe_cuda_ctx_encode_batch",
    "bpe_cuda_decode_batch", "bpe_cuda_ctx_decode_batch",
]

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m llmtokenizer_b200.build` (nvcc, sm_100a). "
            "The engine has no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    P = C.POINTER
    lib.bpe_cuda_train.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_int, P(P(Pair)), P(C.c_size_t),
                                   P(P(C.c_uint32)), P(C.c_size_t), P(Stats)]
    lib.bpe_cuda_train.restype = C.c_int
    lib.bpe_cuda_encode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, P(P(C.c_uint32)),
                                    P(C.c_size_t), P(Stats)]
    lib.bpe_cuda_encode.restype = C.c_int
    lib.bpe_cuda_train_file.argtypes = [C.c_char_p, C.c_uint64, C.c_int, P(P(Pair)), P(C.c_size_t), P(P(C.c_uint32)), P(C.c_size_t),
                                        P(Stats)]
    lib.bpe_cuda_train_file.restype = C.c_int
    lib.bpe_cuda_encode_file.argtypes = [C.c_char_p, C.c_void_p, C.c_size_t, C.c_int, P(P(C.c_uint32)), P(C.c_size_t), P(Stats)]
    lib.bpe_cuda_encode_file.restype = C.c_int
    lib.bpe_cuda_ctx_upload_file.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_uint64, P(C.c_size_t), P(C.c_int)]
    lib.bpe_cuda_ctx_upload_file.restype = C.c_int
    lib.bpe_cuda_ctx_truncate.argtypes = [C.c_void_p, C.c_size_t]
    lib.bpe_cuda_ctx_truncate.restype = C.c_int
    lib.bpe_cuda_ctx_download_pageable.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bpe_cuda_ctx_download_pageable.restype = C.c_int
    lib.bpe_cuda_encode_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, P(P(C.c_uint32)),
                                          P(P(C.c_uint64)), P(C.c_size_t), P(Stats)]
    lib.bpe_cuda_encode_batch.restype = C.c_int
    lib.bpe_cuda_ctx_encode_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                              C.c_void_p, C.c_void_p, P(Stats)]
    lib.bpe_cuda_ctx_encode_batch.restype = C.c_int
    lib.bpe_cuda_decode_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, P(P(C.c_uint8)),
                                          P(P(C.c_uint64)), P(C.c_size_t), P(Stats)]
    lib.bpe_cuda_decode_batch.restype = C.c_int
    lib.bpe_cuda_ctx_decode_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                              C.c_void_p, P(C.c_size_t), P(Stats)]
    lib.bpe_cuda_ctx_decode_batch.restype = C.c_int
    lib.bpe_cuda_free.argtypes = [C.c_void_p]
    lib.bpe_cuda_free.restype = None
    lib.bpe_cuda_last_error.restype = C.c_char_p
    lib.bpe_cuda_device_count.restype = C.c_int
    lib.bpe_cuda_ctx_create.argtypes = [C.c_int, P(C.c_void_p)]
    lib.bpe_cuda_ctx_create.restype = C.c_int
    lib.bpe_cuda_ctx_destroy.argtypes = [C.c_void_p]
    lib.bpe_cuda_ctx_destroy.restype = None
    lib.bpe_cuda_nccl_unique_id.argtypes = [C.c_void_p]
    lib.bpe_cuda_nccl_unique_id.restype = C.c_int
    lib.bpe_cuda_ctx_set_comm.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.bpe_cuda_ctx_set_comm.restype = C.c_int
    lib.bpe_cuda_ctx_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.bpe_cuda_ctx_upload.restype = C.c_int
    lib.bpe_cuda_ctx_upload_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.bpe_cuda_ctx_upload_device.restype = C.c_int
    lib.bpe_cuda_ctx_train.argtypes = [C.c_void_p, C.c_uint64, P(Stats)]
    lib.bpe_cuda_ctx_train.restype = C.c_int
    lib.bpe_cuda_ctx_encode.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, P(Stats)]
    lib.bpe_cuda_ctx_encode.restype = C.c_int
    lib.bpe_cuda_ctx_result_sizes.argtypes = [C.c_void_p, P(C.c_size_t), P(C.c_size_t)]
    lib.bpe_cuda_ctx_result_sizes.restype = C.c_int
    lib.bpe_cuda_ctx_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bpe_cuda_ctx_download.restype = C.c_int
    lib.bpe_cuda_ctx_device_tokens.argtypes = [C.c_void_p]
    lib.bpe_cuda_ctx_device_tokens.restype = C.c_void_p
    lib.bpe_cuda_ctx_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_longlong]
    lib.bpe_cuda_ctx_set_option.restype = C.c_int
    lib.bpe_cuda_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, P(P(C.c_uint8)), P(C.c_size_t), P(Stats)]
    lib.bpe_cuda_decode.restype = C.c_int
    lib.bpe_cuda_ctx_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, P(C.c_size_t)]
    lib.bpe_cuda_ctx_decode.restype = C.c_int
    lib.bpe_cuda_ctx_decode_download.argtypes = [C.c_void_p, C.c_void_p]
    lib.bpe_cuda_ctx_decode_download.restype = C.c_int
    lib.bpe_cuda_ctx_decode_compare.argtypes = [C.c_void_p, P(C.c_uint64)]
    lib.bpe_cuda_ctx_decode_compare.restype = C.c_int
    lib.bpe_cuda_ctx_device_decoded.argtypes = [C.c_void_p]
    lib.bpe_cuda_ctx_device_decoded.restype = C.c_void_p
    _lib = lib
    return lib


_corpus = None


def load_corpus():
    global _corpus
    if _corpus is None:
        if not os.path.exists(CORPUS_LIB_PATH):
            raise RuntimeError(f"{CORPUS_LIB_PATH} is missing: run `python -m llmtokenizer_b200.build`")
        lib = C.CDLL(CORPUS_LIB_PATH)
        lib.gen_corpus_fill.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]
        lib.gen_corpus_fill.restype = C.c_int
        lib.gen_corpus_fnv1a.argtypes = [C.c_void_p, C.c_uint64]
        lib.gen_corpus_fnv1a.restype = C.c_uint64
        _corpus = lib
    return _corpus
