"""ctypes binding of libgenztok.so (include/genztok.h).  No fallback: if the CUDA library is
missing or cannot be loaded, importing the tokenizer fails loudly."""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("GENZTOK_LIB") or os.path.join(_HERE, "libgenztok.so")   # GENZTOK_LIB: try another build of the library

MAX_LEN_NONE = -(2 ** 31)
WANT_TOKEN_TYPE, WANT_SEQUENCE_ID, WANT_SPANS, WANT_OFFSETS = 1, 2, 4, 8
LONGEST_FIRST, ONLY_FIRST, ONLY_SECOND = 16, 32, 64         # pair truncation strategies (at most one)
NONE, EOS_MARK, PAD_MARK = -1, -3, -4

E_INVALID, E_IO, E_UTF8, E_CUDA, E_NOMEM, E_NODEVICE, E_LIMIT = -1, -2, -3, -4, -5, -6, -7
QA_BYTES, QA_CHARS = 0, 1


class Encoded(C.Structure):
    _fields_ = [("n", C.c_int64), ("total", C.c_int64), ("width", C.c_int32), ("has_pair", C.c_int32),
                ("input_ids", C.POINTER(C.c_int32)), ("attention_mask", C.POINTER(C.c_uint8)),
                ("row_off", C.POINTER(C.c_int64)), ("row_len", C.POINTER(C.c_int32)),
                ("token_type_ids", C.POINTER(C.c_int8)), ("sequence_id", C.POINTER(C.c_int8)),
                ("tt_len", C.POINTER(C.c_int32)), ("seq_len", C.POINTER(C.c_int32)),
                ("row_status", C.POINTER(C.c_uint8)), ("span_off", C.POINTER(C.c_int64)),
                ("spans", C.POINTER(C.c_int32)), ("real_tokens", C.c_int64), ("_owner", C.c_void_p), ("d2h_bytes", C.c_int64),
                ("offsets", C.POINTER(C.c_int32))]


class Text(C.Structure):
    _fields_ = [("n", C.c_int64), ("total", C.c_int64), ("bytes", C.POINTER(C.c_uint8)),
                ("off", C.POINTER(C.c_int64)), ("_owner", C.c_void_p)]


class DevPlanes(C.Structure):
    _fields_ = [("input_ids", C.c_void_p), ("attention_mask", C.c_void_p), ("token_type_ids", C.c_void_p),
                ("sequence_id", C.c_void_p), ("row_len", C.c_void_p), ("seq_len", C.c_void_p), ("row_status", C.c_void_p),
                ("offsets", C.c_void_p)]


class Windows(C.Structure):
    _fields_ = [("enc", Encoded), ("n_docs", C.c_int64), ("win_off", C.POINTER(C.c_int64)), ("win_doc", C.POINTER(C.c_int64)),
                ("win_start", C.POINTER(C.c_int32))]


SIGNATURES = {
    # name: (restype, argtypes)
    "genztok_create": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "genztok_destroy": (None, [C.c_void_p]),
    "genztok_last_error": (C.c_char_p, [C.c_void_p]),
    "genztok_version": (C.c_char_p, []),
    "genztok_vocab_size": (C.c_int64, [C.c_void_p]),
    "genztok_special_ids": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "genztok_encoder_count": (C.c_int64, [C.c_void_p]),
    "genztok_encoder_entry": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "genztok_encoder_get": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_int64]),
    "genztok_decoder_get": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_int64)]),
    "genztok_merge_count": (C.c_int64, [C.c_void_p]),
    "genztok_merge_line": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_int64)]),
    "genztok_rank_get": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_int64, C.c_char_p, C.c_int64]),
    "genztok_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int, C.c_int, C.c_uint32, C.POINTER(Encoded)]),
    "genztok_free_encoded": (None, [C.c_void_p, C.POINTER(Encoded)]),
    "genztok_encode_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_uint32, C.POINTER(DevPlanes), C.c_void_p]),
    "genztok_encode_windows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(Windows)]),
    "genztok_free_windows": (None, [C.c_void_p, C.POINTER(Windows)]),
    "genztok_encode_windows_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32,
                                                C.c_uint32, C.c_void_p, C.POINTER(DevPlanes), C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]),
    "genztok_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.POINTER(Text)]),
    "genztok_free_text": (None, [C.c_void_p, C.POINTER(Text)]),
    "genztok_decode_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]),
    "genztok_gather_rows": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.c_int64, C.c_void_p, C.c_int64,
                                      C.POINTER(C.c_void_p), C.c_void_p]),
    "genztok_decode_device_into": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64),
                                             C.c_void_p]),
    "genztok_preprocess": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Text)]),
    "genztok_preprocess_device": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]),
    "genztok_bpe_word": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64, C.POINTER(C.c_int32), C.c_int64, C.POINTER(C.c_int64)]),
    "genztok_sequence_id": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "genztok_attention_mask": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "genztok_host_alloc": (C.c_void_p, [C.c_size_t]),
    "genztok_host_free": (None, [C.c_void_p]),
    "genztok_device_count": (C.c_int, [C.c_void_p]),
    "genztok_cache_reset": (C.c_int, [C.c_void_p]),
    "genztok_launch_count": (C.c_int64, [C.c_void_p]),
    "genztok_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "genztok_profile_report": (C.c_int64, [C.c_void_p, C.c_char_p, C.c_int64, C.c_int]),
    "genztok_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "genztok_check_errors": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int64)]),
    "genztok_synth_init": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64]),
    "genztok_synth_device": (C.c_int, [C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]),
    "genztok_qa_labels_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_int32, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "genztok_qa_best_spans_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int, C.c_void_p, C.c_int64,
                                              C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "genztok_mlm_mask_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_double,
                                         C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "genztok_encode_dropout": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint32, C.c_double, C.c_uint64,
                                         C.c_void_p, C.POINTER(Encoded)]),
    "genztok_encode_dropout_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32,
                                                C.c_uint32, C.c_double, C.c_uint64, C.c_void_p, C.POINTER(DevPlanes), C.c_void_p]),
    "genztok_bpe_word_dropout": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64, C.c_double, C.c_uint64, C.c_int64, C.POINTER(C.c_int32), C.c_int64,
                                           C.POINTER(C.c_int64)]),
    "genztok_digest_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]),
}

_lib = None


def build(force=False):
    """Compile libgenztok.so in-tree with nvcc for sm_100a (no GPU needed to build)."""
    srcdir = os.path.join(_HERE, "csrc")
    srcs = [os.path.join(srcdir, f) for f in os.listdir(srcdir) if f.endswith((".cu", ".cuh", ".hpp"))]
    srcs.append(os.path.join(_HERE, "..", "include", "genztok.h"))
    stale = not os.path.exists(SO_PATH) or any(os.path.getmtime(s) > os.path.getmtime(SO_PATH) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-C", srcdir, "-s"] + (["-B"] if force else []))
    return SO_PATH


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError("genz_tokenize_b200: %s is missing; build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C genz_tokenize_b200/csrc` (there is no CPU fallback)" % SO_PATH)
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError if the ABI lost a symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
