"""ctypes binding of libpamrec_b200.so (include/pamrec_b200.h).  There is no fallback: if the
CUDA library has not been built the import fails loudly."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpamrec_b200.so")

POOL_DENSE, POOL_BN, POOL_WORKSPACE = 0, 1, 2
F32, I32, F64, U8 = 0, 1, 2, 3
SEG_L2, SEG_POS, SEG_DEAD = 1, 2, 4
ADAM_DENSE_EXACT, ADAM_LAZY = 0, 1
TABLES_LOCAL, TABLES_SHARDED, TABLES_REPLICATED = 0, 1, 2
LOSS_XENT, LOSS_SOFTMAX = 0, 1
MODEL_PAMREC, MODEL_MMOE, MODEL_PLE, MODEL_SHAREBOTTOM, MODEL_SASREC = 0, 1, 2, 3, 4
COMM_ID_BYTES = 128
IPC_HANDLE_BYTES = 64
GROUP = 5
DEBUG_SAVE_FFN_HIDDEN = 1
DEBUG_HEAD_TRACE = 2


class PamrecConfig(C.Structure):
    _fields_ = [
        ("n_users", C.c_int32), ("n_items", C.c_int32), ("n_cates", C.c_int32),
        ("max_seq_len", C.c_int32), ("max_batch", C.c_int32),
        ("learning_rate", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("epsilon", C.c_float),
        ("embed_l2", C.c_float), ("layer_l2", C.c_float), ("max_grad_norm", C.c_float), ("is_clip_norm", C.c_int32),
        ("fuzhu_weight", C.c_float), ("order_weight", C.c_float), ("sparse_adam_mode", C.c_int32),
        ("world_size", C.c_int32), ("rank", C.c_int32), ("table_mode", C.c_int32),
        ("loss_kind", C.c_int32), ("softmax_group", C.c_int32), ("model_kind", C.c_int32),
        ("item_dim", C.c_int32), ("cate_dim", C.c_int32), ("user_dim", C.c_int32),
    ]


class PamrecBatch(C.Structure):
    _fields_ = [
        ("batch", C.c_int32),
        ("item_history", C.c_void_p), ("item_cate_history", C.c_void_p), ("item_loop_times_history", C.c_void_p),
        ("mask", C.c_void_p), ("users", C.c_void_p), ("items", C.c_void_p), ("cates", C.c_void_p),
        ("labels_satisfied", C.c_void_p), ("labels_play", C.c_void_p), ("plays", C.c_void_p),
        ("global_batch", C.c_int32),
        ("satisfied_item_history", C.c_void_p), ("satisfied_cate_history", C.c_void_p), ("satisfied_mask", C.c_void_p),
    ]


class PamrecBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "dense_param", "dense_grad", "dense_m", "dense_v", "bn_moving",
        "item_w", "item_m", "item_v", "cate_w", "cate_m", "cate_v",
        "ulong_w", "ulong_m", "ulong_v", "ushort_w", "ushort_m", "ushort_v", "workspace")] + [("workspace_bytes", C.c_size_t)]


class PamrecLines(C.Structure):
    _fields_ = [("n_lines", C.c_int64), ("offsets", C.c_void_p), ("items", C.c_void_p), ("cates", C.c_void_p),
                ("durs", C.c_void_p), ("sats", C.c_void_p), ("plays", C.c_void_p), ("user_ids", C.c_void_p),
                ("label_sat", C.c_void_p), ("label_play", C.c_void_p), ("tgt_item", C.c_void_p), ("tgt_cate", C.c_void_p),
                ("tgt_dur", C.c_void_p)]


class PamrecVocab(C.Structure):
    _fields_ = [("n", C.c_int64), ("bytes", C.c_void_p), ("offsets", C.c_void_p), ("values", C.c_void_p)]


class PamrecTensorInfo(C.Structure):
    _fields_ = [("name", C.c_char * 160), ("pool", C.c_int32), ("dtype", C.c_int32), ("flags", C.c_int32),
                ("offset", C.c_int64), ("numel", C.c_int64), ("ndim", C.c_int32), ("shape", C.c_int64 * 4)]


EXPORTS = {
    "pamrec_version": (C.c_char_p, []),
    "pamrec_abi_sizes": (C.c_int, [C.POINTER(C.c_int64)]),
    "pamrec_create": (C.c_int, [C.POINTER(PamrecConfig), C.POINTER(C.c_void_p)]),
    "pamrec_destroy": (C.c_int, [C.c_void_p]),
    "pamrec_last_error": (C.c_char_p, [C.c_void_p]),
    "pamrec_dense_numel": (C.c_int64, [C.c_void_p]),
    "pamrec_bn_numel": (C.c_int64, [C.c_void_p]),
    "pamrec_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "pamrec_tensor_count": (C.c_int, [C.c_void_p, C.c_int]),
    "pamrec_tensor_info": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(PamrecTensorInfo)]),
    "pamrec_bind": (C.c_int, [C.c_void_p, C.POINTER(PamrecBuffers), C.c_void_p]),
    "pamrec_gather_fwd": (C.c_int, [C.c_void_p, C.POINTER(PamrecBatch), C.c_void_p, C.c_void_p]),
    "pamrec_forward": (C.c_int, [C.c_void_p, C.POINTER(PamrecBatch), C.c_int, C.c_void_p, C.c_void_p]),
    "pamrec_backward": (C.c_int, [C.c_void_p, C.POINTER(PamrecBatch), C.c_void_p]),
    "pamrec_apply_gradients": (C.c_int, [C.c_void_p, C.POINTER(PamrecBatch), C.c_int64, C.c_void_p]),
    "pamrec_train_step": (C.c_int, [C.c_void_p, C.POINTER(PamrecBatch), C.c_int64, C.c_void_p, C.c_void_p]),
    "pamrec_comm_unique_id": (C.c_int, [C.c_char_p, C.c_char_p]),
    "pamrec_comm_init": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p]),
    "pamrec_comm_destroy": (C.c_int, [C.c_void_p]),
    "pamrec_comm_mailbox_create": (C.c_int, [C.c_void_p, C.c_char_p]),
    "pamrec_comm_mailbox_open": (C.c_int, [C.c_void_p, C.c_char_p]),
    "pamrec_shard_rows": (C.c_int64, [C.c_void_p, C.c_int64]),
    "pamrec_comm_all_reduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "pamrec_bench_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                      C.c_void_p, C.c_void_p]),
    "pamrec_bench_table_adam": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "pamrec_set_debug": (C.c_int, [C.c_void_p, C.c_int]),
    "pamrec_head_trace": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
    "pamrec_head_trace_ctas": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]),
    "pamrec_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "pamrec_profile_reset": (C.c_int, [C.c_void_p]),
    "pamrec_profile_count": (C.c_int, [C.c_void_p]),
    "pamrec_profile_get": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "pamrec_last_launch_count": (C.c_int64, [C.c_void_p]),
    "pamrec_batcher_create": (C.c_int, [C.POINTER(PamrecLines), C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "pamrec_batcher_destroy": (C.c_int, [C.c_void_p]),
    "pamrec_batcher_begin_train": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "pamrec_batcher_begin_eval": (C.c_int, [C.c_void_p, C.c_int]),
    "pamrec_batcher_next": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "pamrec_batcher_next_shard": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p,
                                            C.POINTER(C.c_int)]),
    "pamrec_tokenize_file": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(PamrecVocab), C.POINTER(PamrecVocab), C.POINTER(PamrecVocab),
                                       C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "pamrec_tokens_read": (C.c_int, [C.c_void_p, C.POINTER(PamrecLines)]),
    "pamrec_tokens_free": (C.c_int, [C.c_void_p]),
    "pamrec_crc32c": (C.c_uint32, [C.c_uint32, C.c_void_p, C.c_size_t]),
    "pamrec_crc32c_portable": (C.c_uint32, [C.c_uint32, C.c_void_p, C.c_size_t]),
}

_lib = None


def load():
    """Load the shared library once and type every export declared in include/pamrec_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m pamrec_b200.build` (nvcc, sm_100a). "
            "pamrec_b200 has no CPU or eager fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    sizes = (C.c_int64 * 6)()
    lib.pamrec_abi_sizes(sizes)
    mirror = [C.sizeof(t) for t in (PamrecConfig, PamrecBatch, PamrecBuffers, PamrecTensorInfo, PamrecLines, PamrecVocab)]
    if list(sizes) != mirror:
        raise RuntimeError(f"ctypes mirrors disagree with include/pamrec_b200.h as compiled: {list(sizes)} vs {mirror} (rebuild the library)")
    _lib = lib
    return lib
