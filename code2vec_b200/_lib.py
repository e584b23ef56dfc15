"""ctypes binding of libc2v_b200.so (include/c2v_b200.h).

The product path has NO CPU fallback: if the CUDA library is missing or cannot be
loaded, importing it raises -- loudly -- instead of computing something slower.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("C2V_LIB", os.path.join(_HERE, "libc2v_b200.so"))   # C2V_LIB: variant builds (scripts/sanitize.sh)

C2V_OK, C2V_EINVAL, C2V_ECUDA, C2V_EWORKSPACE, C2V_EINDEX, C2V_EUNSUPPORTED = 0, -1, -2, -3, -4, -5
ALGO_AUTO, ALGO_FFMA, ALGO_TCGEN05 = 0, 1, 2
ABI_VERSION = 1

c_i32, c_i64, c_f32, c_vp, c_sz = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t


class Dims(ctypes.Structure):
    _fields_ = [("terminal_count", c_i64), ("path_count", c_i64), ("label_count", c_i64),
                ("terminal_embed", c_i32), ("path_embed", c_i32), ("encode", c_i32), ("reserved", c_i32)]


class Params(ctypes.Structure):
    _fields_ = [("terminal_embedding", c_vp), ("path_embedding", c_vp), ("input_linear", c_vp),
                ("ln_weight", c_vp), ("ln_bias", c_vp), ("attention", c_vp),
                ("output_weight", c_vp), ("output_bias", c_vp)]


class Grads(ctypes.Structure):
    _fields_ = [("terminal_embedding", c_vp), ("path_embedding", c_vp), ("input_linear", c_vp),
                ("ln_weight", c_vp), ("ln_bias", c_vp), ("attention", c_vp)]


class Dropout(ctypes.Structure):
    _fields_ = [("p", c_f32), ("training", c_i32), ("seed", ctypes.c_uint64)]


class DeviceInfo(ctypes.Structure):
    _fields_ = [("cc_major", c_i32), ("cc_minor", c_i32), ("sm_count", c_i32), ("reserved", c_i32),
                ("global_mem_bytes", c_i64), ("smem_per_block_optin", c_i64)]


class CorpusInfo(ctypes.Structure):
    _fields_ = [("n_items", c_i64), ("n_contexts", c_i64), ("n_aliases", c_i64), ("label_bytes", c_i64),
                ("alias_bytes", c_i64), ("alias_name_bytes", c_i64)]


# every symbol include/c2v_b200.h declares: (restype, argtypes)
_P = ctypes.POINTER
SYMBOLS = {
    "c2v_abi_version": (ctypes.c_int, []),
    "c2v_last_error": (ctypes.c_char_p, []),
    "c2v_get_device_info": (ctypes.c_int, [ctypes.c_int, _P(DeviceInfo)]),
    "c2v_encode_supports_tcgen05": (ctypes.c_int, [_P(Dims)]),
    "c2v_encode_workspace_bytes": (c_sz, [_P(Dims), c_i32, c_i32]),
    "c2v_encode_forward": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_vp, c_i32, c_i32, _P(Dropout),
                                          c_vp, c_vp, c_vp, c_sz, c_i32, c_vp]),
    "c2v_encode_forward_stash": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_vp, c_i32, c_i32, _P(Dropout),
                                                c_vp, c_vp, c_vp, c_vp, c_sz, c_i32, c_vp]),
    "c2v_workspace_status": (c_i64, [c_vp, c_vp]),
    "c2v_workspace_set_status_mirror": (ctypes.c_int, [c_vp, c_vp, c_vp]),
    "c2v_label_workspace_bytes": (c_sz, [_P(Dims), c_i32]),
    "c2v_label_logits": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_i32, c_vp, c_vp, c_sz, c_i32, c_vp]),
    "c2v_label_logits_argmax": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_sz, c_i32,
                                               c_vp]),
    "c2v_label_loss_supported": (ctypes.c_int, [_P(Dims), c_i32]),
    "c2v_label_loss_argmax": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz,
                                             c_i32, c_vp]),
    "c2v_label_dlogits": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_vp, c_i32, c_f32, c_vp, c_vp, c_vp, c_sz, c_i32,
                                         c_vp]),
    "c2v_angular_logits": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_i32, c_f32, c_f32, c_vp, c_vp]),
    "c2v_angular_forward_train": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp]),
    "c2v_angular_backward": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp,
                                            c_vp, c_vp, c_vp]),
    "c2v_build_batch": (ctypes.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i32, c_i32, ctypes.c_uint64, c_i64, c_i64, c_vp, c_vp,
                                       c_vp, c_vp, c_vp]),
    "c2v_build_batch_vars": (ctypes.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_i32, c_i32, ctypes.c_uint64,
                                            c_i64, c_vp, c_i64, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "c2v_adam_step": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_f32, c_f32, c_i64, c_f32, c_i32, c_vp]),
    "c2v_adam_step_sharded": (ctypes.c_int, [c_vp, c_vp, c_vp, _P(c_vp), _P(c_vp), c_i32, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64,
                                             c_f32, c_f32, c_f32, c_f32, c_f32, c_i64, c_f32, c_vp]),
    "c2v_adam_step_sharded_bulk": (ctypes.c_int, [c_vp, _P(c_vp), _P(c_vp), c_i32, c_vp, c_vp, c_i64, c_i64, c_f32, c_f32, c_f32,
                                                  c_f32, c_f32, c_i64, c_f32, c_i32, c_vp]),
    "c2v_loss_argmax": (ctypes.c_int, [c_vp, c_vp, c_i32, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "c2v_label_backward": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "c2v_label_backward_ws": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_sz, c_i32, c_vp]),
    "c2v_encode_backward_workspace_bytes": (c_sz, [_P(Dims), c_i32, c_i32]),
    "c2v_encode_backward": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_vp, c_i32, c_i32, _P(Dropout),
                                           c_vp, c_vp, c_vp, c_vp, _P(Grads), c_vp, c_sz, c_vp]),
    "c2v_encode_backward_stashed": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_vp, c_i32, c_i32, _P(Dropout),
                                                   c_vp, c_vp, c_vp, c_vp, c_vp, _P(Grads), c_vp, c_sz, c_vp]),
    "c2v_encode_backward_phased": (ctypes.c_int, [_P(Dims), _P(Params), c_vp, c_vp, c_vp, c_i32, c_i32, _P(Dropout),
                                                  c_vp, c_vp, c_vp, c_vp, c_vp, _P(Grads), c_vp, c_sz, c_i32, c_vp]),
    "c2v_session_create": (ctypes.c_int, [ctypes.c_int, _P(Dims), c_i32, c_i32, _P(c_vp)]),
    "c2v_session_destroy": (None, [c_vp]),
    "c2v_forward_host": (ctypes.c_int, [c_vp, _P(Params), c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp,
                                        c_vp, c_i32]),
    "c2v_forward_host_async": (ctypes.c_int, [c_vp, _P(Params), c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp,
                                              c_vp, c_vp, c_i32, _P(c_i64)]),
    "c2v_session_wait": (ctypes.c_int, [c_vp, c_i64]),
    "c2v_launch_count": (c_i64, []),
    "c2v_profile_enable": (ctypes.c_int, [c_i32]),
    "c2v_profile_read": (ctypes.c_int, [_P(ctypes.c_double), _P(c_i64)]),
    "c2v_corpus_parse_buffer": (ctypes.c_int, [ctypes.c_char_p, c_sz, c_i32, _P(c_vp)]),
    "c2v_corpus_parse_files": (ctypes.c_int, [_P(ctypes.c_char_p), c_i32, c_i32, _P(c_vp)]),
    "c2v_corpus_free": (None, [c_vp]),
    "c2v_corpus_get_info": (ctypes.c_int, [c_vp, _P(CorpusInfo)]),
    "c2v_corpus_export": (ctypes.c_int, [c_vp] + [c_vp] * 12),
    "c2v_corpus_save": (ctypes.c_int, [c_vp, ctypes.c_char_p]),
    "c2v_corpus_load": (ctypes.c_int, [ctypes.c_char_p, _P(c_vp)]),
    "c2v_format_float": (ctypes.c_int, [c_f32, ctypes.c_char_p, c_sz]),
    "c2v_write_code_vectors": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p, c_i64, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp,
                                              c_i64, ctypes.c_char_p, ctypes.c_char_p, c_vp, c_vp, c_vp]),
}

_lib = None


class C2VError(RuntimeError):
    pass


def load():
    """dlopen the in-tree CUDA library; raises if it is missing (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise C2VError(
            f"{LIB_PATH} is missing: build it with `python -m code2vec_b200.build` "
            "(or __graft_entry__.build()). code2vec_b200 has no CPU / eager fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    got = lib.c2v_abi_version()
    if got != ABI_VERSION:
        raise C2VError(f"libc2v_b200.so ABI {got} != binding ABI {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc, what):
    if rc == C2V_OK:
        return
    msg = load().c2v_last_error().decode("utf-8", "replace")
    if rc == C2V_EINDEX:
        raise IndexError(msg or "index out of range in self")      # what nn.Embedding raises
    if rc == C2V_EUNSUPPORTED:
        raise NotImplementedError(f"{what}: {msg}")
    raise C2VError(f"{what} failed ({rc}): {msg}")
