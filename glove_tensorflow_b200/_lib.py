"""ctypes binding of libglove_b200.so (C ABI declared in include/glove_b200.h).

The product path has NO CPU fallback: if the shared library is missing or does not export the ABI, importing
this module raises immediately (build it with ``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C glove_tensorflow_b200/csrc``)."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libglove_b200.so")

OK, EINVAL, ECUDA, EWORKSPACE, EUNSUPPORTED = 0, -1, -2, -3, -4
HEADS = {"glove": 0, "logistic": 1}
OPTIMIZERS = {"Adam": 0, "Adagrad": 1, "SGD": 2}
# "replay" = closed-form replay of idle steps (default, reference semantics); "replay_exact" = step-by-step replay with the
# dense sweep's fp32 operations; "dense" = replay_exact + flush after every step (the literal legacy-Keras schedule)
ADAM_MODES = {"replay": 0, "lazy": 1, "replay_exact": 2, "dense": 2}
ABI_VERSION = 2
ANALOGY_METHODS = {"add": 0, "mul": 1}   # 3CosAdd, 3CosMul (glove_analogy_topk)

c_i32, c_i64, c_u32, c_f32 = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_float
c_void, c_size = ctypes.c_void_p, ctypes.c_size_t


class GloveScalars(ctypes.Structure):
    _fields_ = [("step", c_i32), ("error", c_i32), ("g", c_f32), ("g_s0", c_f32), ("g_s1", c_f32), ("loss", c_f32),
                ("ticket", c_i32), ("reserved", c_i32)]


class StepArgs(ctypes.Structure):
    _fields_ = [("struct_size", c_u32),
                ("row_table", c_void), ("col_table", c_void), ("scalars", c_void), ("plan", c_void),
                ("workspace", c_void), ("workspace_bytes", c_size), ("alpha", c_void), ("alpha_len", c_i32),
                ("loss_out", c_void), ("loss_cap", c_i32), ("plan_K", c_i32), ("V", c_i64), ("d", c_i32), ("B", c_i32),
                ("head", c_i32), ("optimizer", c_i32), ("adam_mode", c_i32), ("learning_rate", c_f32),
                ("l2_reg", c_f32), ("reg_scale", c_f32), ("neg_factor", c_f32), ("beta1", c_f32), ("beta2", c_f32),
                ("epsilon", c_f32), ("dp_rank", c_i32), ("dp_world", c_i32), ("n_shards", c_i32), ("shard", c_i32),
                ("peer_gather", c_i32)]


class CsvSchema(ctypes.Structure):
    _fields_ = [("n_cols", c_i32), ("column", c_i32 * 4), ("kind", c_i32 * 4)]


CSV_TOKEN, CSV_INT, CSV_FLOAT = 0, 1, 2

# name -> (restype, argtypes); every symbol include/glove_b200.h declares
SIGNATURES = {
    "glove_last_error": (ctypes.c_char_p, []),
    "glove_abi_version": (c_i32, []),
    "glove_table_stride": (c_i32, [c_i32]),
    "glove_table_planes": (c_i32, [c_i32]),
    "glove_table_init": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_i32, c_void]),
    "glove_pack_plane": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_i32, c_i32, c_void, c_void, c_void]),
    "glove_unpack_plane": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_i32, c_i32, c_void, c_void, c_void]),
    "glove_get_last_step": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_i32, c_void, c_void]),
    "glove_set_last_step": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_i32, c_void, c_void]),
    "glove_shuffle_indices": (ctypes.c_int, [c_u32, c_i64, c_i64, c_i64, c_void, c_void]),
    "glove_plan_bytes": (c_size, [c_i32, c_i32]),
    "glove_prepare_workspace_bytes": (c_size, [c_i32, c_i32]),
    "glove_prepare_batches": (ctypes.c_int, [c_void, c_void, c_size, c_void, c_void, c_void, c_void, c_i64, c_void,
                                             c_i64, c_u32, c_i32, c_i32, c_i32, c_i32, c_void]),
    "glove_prepare_batches_sharded": (ctypes.c_int, [c_void, c_void, c_size, c_void, c_void, c_void, c_void, c_i64, c_void,
                                                     c_i64, c_u32, c_i32, c_i32, c_i32, c_i32, c_i32, c_void]),
    "glove_plan_shard_info": (ctypes.c_int, [c_void, c_i32, c_i32, c_i32, ctypes.POINTER(c_i32), c_void]),
    "glove_plan_batch_counts": (ctypes.c_int, [c_void, c_i32, c_i32, c_i32, ctypes.POINTER(c_i32), c_void]),
    "glove_step_args_size": (c_size, []),
    "glove_step_workspace_bytes": (c_size, [c_i32, c_i32]),
    "glove_train_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void]),
    "glove_step_graph_create": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_i32, ctypes.POINTER(c_void)]),
    "glove_step_graph_launch": (ctypes.c_int, [c_void, c_void]),
    "glove_step_graph_destroy": (ctypes.c_int, [c_void]),
    "glove_catchup_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_i32, c_void]),
    "glove_train_step_profiled": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void, ctypes.POINTER(c_f32)]),
    "glove_grad_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void, c_void, c_void, c_void]),
    "glove_apply_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void, c_void, c_void, c_void]),
    "glove_shard_set_peers": (ctypes.c_int, [ctypes.POINTER(StepArgs), ctypes.POINTER(c_void), c_i32, c_void]),
    "glove_shard_pull_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void]),
    "glove_shard_signal_staged": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void]),
    "glove_shard_wait_staged": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void]),
    "glove_shard_finish_sync": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void, c_void]),
    "glove_shard_train_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void]),
    "glove_shard_stage_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void]),
    "glove_shard_pack_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void, c_void]),
    "glove_shard_unpack_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void, c_void]),
    "glove_plan_need_info": (ctypes.c_int, [c_void, c_i32, c_i32, ctypes.POINTER(c_i32), c_void]),
    "glove_plan_pull_slice": (ctypes.c_int, [c_void, c_void, c_i32, c_i32, c_i32, c_i32, c_void]),
    "glove_shard_update_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void, c_void]),
    "glove_shard_finish_step": (ctypes.c_int, [ctypes.POINTER(StepArgs), c_void, c_void]),
    "glove_step_snapshot_rows": (c_i64, [c_i32]),
    "glove_step_snapshot_offset": (c_size, [c_i32, c_i32, c_i32]),
    "glove_flush_lazy_state": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_i32, c_void, c_i32, c_i32, c_f32, c_f32, c_f32,
                                              c_void]),
    "glove_flush_lazy_state_exact": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_i32, c_void, c_i32, c_i32, c_f32, c_f32,
                                                    c_f32, c_void]),
    "glove_eval_workspace_bytes": (c_size, [c_i64, c_i32]),
    "glove_eval_loss": (ctypes.c_int, [c_void, c_void, c_void, c_i32, c_i32, c_void, c_void, c_void, c_void, c_i64,
                                       c_i64, c_i32, c_i32, c_void, c_void, c_size, c_void]),
    "glove_topk_kpad": (c_i32, [c_i32]),
    "glove_topk_vpad": (c_i64, [c_i64]),
    "glove_normalize_rows": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_void, c_void, c_void]),
    "glove_topk_workspace_bytes": (c_size, [c_i64, c_i32, c_i32, c_i32]),
    "glove_topk_cosine": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_void, c_void, c_void, c_i32, c_i32, c_void,
                                         c_void, c_void, c_size, c_void]),
    "glove_topk_cosine_queries": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_void, c_void, c_void, c_i32, c_void, c_void,
                                                 c_i32, c_i32, c_void, c_void, c_void, c_size, c_void]),
    "glove_topk_merge": (ctypes.c_int, [c_void, c_void, c_i32, c_i32, c_i32, c_void, c_void, c_void]),
    "glove_topk_flagged": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_i32, ctypes.POINTER(c_i32), c_void]),
    "glove_topk_cosine_fp32": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_void, c_void, c_i32, c_i32, c_void,
                                              c_void, c_void, c_size, c_void]),
    "glove_analogy_workspace_bytes": (c_size, [c_i64, c_i32, c_i32, c_i32, c_i32]),
    "glove_analogy_topk": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_void, c_void, c_void, c_i32, c_i32, c_i32, c_void,
                                          c_void, c_void, c_size, c_void]),
    "glove_pair_cosine": (ctypes.c_int, [c_void, c_i64, c_i32, c_i32, c_void, c_void, c_i32, c_void, c_void]),
    "glove_vocab_slots": (c_i64, [c_i64]),
    "glove_vocab_build": (ctypes.c_int, [c_void, c_i64, c_void, c_void, c_i64, c_void]),
    "glove_csv_workspace_bytes": (c_size, [c_i64]),
    "glove_csv_index": (ctypes.c_int, [c_void, c_i64, c_void, c_size, ctypes.POINTER(c_i64), c_void]),
    "glove_csv_parse": (ctypes.c_int, [c_void, c_i64, c_i32, c_void, c_size, ctypes.POINTER(CsvSchema), c_void, c_i64,
                                       c_void, c_void, c_i64, c_void, c_void, c_void, c_void, c_void, c_i64, c_i64,
                                       ctypes.POINTER(c_i64), ctypes.POINTER(c_i64), c_void]),
    "glove_parse_float32": (ctypes.c_int, [ctypes.c_char_p, c_i32, ctypes.POINTER(c_f32)]),
    "glove_tokens_workspace_bytes": (c_size, [c_i64, c_i64]),
    "glove_tokens_scan": (ctypes.c_int, [c_void, c_i64, c_void, c_size, c_void, c_void, c_i64, ctypes.POINTER(c_i64), c_void]),
    "glove_tokens_count": (ctypes.c_int, [c_void, c_i64, c_void, c_i64, c_void, c_size, c_void, c_void, c_void, c_i64,
                                          ctypes.POINTER(c_i64), c_void]),
    "glove_tokens_lookup": (ctypes.c_int, [c_void, c_void, c_void, c_i64, c_void, c_i64, c_void, c_void, c_void, c_void]),
    "glove_cooc_workspace_bytes": (c_size, [c_i64]),
    "glove_cooc_chunk": (ctypes.c_int, [c_void, c_i64, c_i64, c_i32, c_i32, c_void, c_size, c_void, c_void, c_i64,
                                        ctypes.POINTER(c_i64), c_void]),
    "glove_cooc_merge": (ctypes.c_int, [c_void, c_void, c_i64, c_void, c_void, c_i64, c_i32, c_void, c_size, c_void, c_void,
                                        c_i64, ctypes.POINTER(c_i64), c_void]),
    "glove_cooc_finish": (ctypes.c_int, [c_void, c_void, c_i64, c_i32, c_i32, c_i64, c_void, c_i64, ctypes.c_uint64, c_void,
                                         c_size, c_void, c_void, c_void, c_void, c_void, c_void, c_void, c_i64,
                                         ctypes.POINTER(c_i64), c_void]),
    "glove_host_staging_bytes": (c_size, [c_i32, c_i32]),
    "glove_host_plan_bytes": (c_size, [c_i32, c_i32]),
    "glove_host_pipe_create": (ctypes.c_int, [ctypes.POINTER(c_void)]),
    "glove_host_pipe_destroy": (ctypes.c_int, [c_void]),
    "glove_train_steps_host": (ctypes.c_int, [c_void, ctypes.POINTER(StepArgs), c_void, c_void, c_size, c_void, c_size,
                                              c_void, c_void, c_void, c_void, c_i32, c_void, c_void]),
}

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "glove_tensorflow_b200: %s is missing. There is no CPU fallback; build the CUDA library first "
        "(python -c 'import __graft_entry__ as g; g.build()' or make -C glove_tensorflow_b200/csrc)." % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = ABI mismatch: fail loudly
    _fn.restype = _res
    _fn.argtypes = _args

if lib.glove_abi_version() != ABI_VERSION:
    raise ImportError("glove_tensorflow_b200: ABI version mismatch in %s (library %d, binding %d)"
                      % (LIB_PATH, lib.glove_abi_version(), ABI_VERSION))
if lib.glove_step_args_size() != ctypes.sizeof(StepArgs):
    raise ImportError("glove_tensorflow_b200: glove_step_args is %d bytes in %s, %d in the ctypes binding"
                      % (lib.glove_step_args_size(), LIB_PATH, ctypes.sizeof(StepArgs)))


class GloveError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != OK:
        msg = lib.glove_last_error()
        raise GloveError("%s failed (%d): %s" % (what or "glove call", rc, msg.decode() if msg else ""))
