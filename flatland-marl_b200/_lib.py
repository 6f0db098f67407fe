"""ctypes binding of the C ABI in include/flatland_b200.h.  There is no CPU fallback: if the CUDA
library is missing this module raises, and every compute entry point needs a CUDA device."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libflatland_b200.so")

MAX_NODES, NODE_F, ATTR_F, PRED_DEPTH = 31, 12, 83, 500
ACTION_ABSENT = 255
ST_STEP_AFTER_DONE, ST_AUTO_RESET, ST_BAD_CELL = 1, 2, 4
FLAG_AUTO_RESET, FLAG_FRESH_AGENTS = 1, 2
RESET_KEEP_SCHEDULE, RESET_KEEP_ARRIVAL = 1, 2
COPY_WORLD, COPY_STATE = 1, 2

# field order of struct FlBatch (include/flatland_b200.h)
_FIELDS = [("E", "i"), ("N", "i"), ("H", "i"), ("W", "i"), ("n_slots", "i"), ("S", "i"), ("ent_cap", "i"), ("grid_stride", "i"),
           ("dist_stride", "i"), ("debug_clocks", "p"), ("ridx_stride", "i"), ("state_stride", "i"), ("wlist_stride", "i"),
           ("whits_stride", "i"), ("seg_stride", "i"), ("pc_stride", "i"), ("ws_stride", "i")]
_PTR = ["grid", "slot_rc", "dist", "max_steps", "init_rc", "tgt_rc", "init_dir", "max_count", "slot", "speed",
        "earliest", "latest", "sched", "ridx", "srec", "wrec", "whoff", "wlist", "whits", "kcls", "sdist", "gtab", "walk_total",
        "rc", "old_rc", "dir", "old_dir", "state", "ctr", "mal", "saved", "sig_mal", "deadlocked", "done", "nmal",
        "arrival",
        "elapsed", "sched_pos", "done_all", "status", "stats",
        "entries", "segs", "obs_ws", "tree_cache", "path_cache"]
TREE_CACHE_WORDS = 160


class FlBatch(C.Structure):
    """Mirror of `struct FlBatch` (include/flatland_b200.h); the size is checked against the library."""
    _fields_ = [(n, C.c_int64 if k == "i" else C.c_void_p) for n, k in _FIELDS] + [(n, C.c_void_p) for n in _PTR]


class FlObsBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("agent_attr", "forest", "adjacency", "node_order", "edge_order",
                                          "valid_actions", "dist_target", "rewards", "dones")]


EXPORTS = ["fl_abi_version", "fl_batch_sizeof", "fl_error_string", "fl_distance_map", "fl_distance_map_ids", "fl_walk_tables", "fl_walk_tables_ids", "fl_reset", "fl_reset_ex", "fl_step",
           "fl_observe", "fl_observe_override", "fl_observe_plan", "fl_observe_ws_words", "fl_batch_slice", "fl_copy_envs", "fl_step_observe_host", "fl_step_observe_host_compact", "fl_wire_bytes", "fl_host_threads", "fl_launch_count", "fl_profile_num_kernels", "fl_profile_kernel_name",
           "fl_profile_enable", "fl_profile_collect"]

_lib = None


class FlatlandB200Error(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FlatlandB200Error(
            "CUDA library %s is not built (run `python __graft_entry__.py build` or "
            "`python flatland-marl_b200/build.py`); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    P = C.c_void_p
    L.fl_abi_version.restype = C.c_int
    L.fl_batch_sizeof.restype = C.c_size_t
    L.fl_error_string.restype = C.c_char_p
    L.fl_error_string.argtypes = [C.c_int]
    L.fl_launch_count.restype = C.c_uint64
    L.fl_distance_map.argtypes = [C.POINTER(FlBatch), P]
    L.fl_reset.argtypes = [C.POINTER(FlBatch), P, P]
    L.fl_reset_ex.argtypes = [C.POINTER(FlBatch), P, C.c_uint32, P]
    L.fl_observe_override.argtypes = [C.c_char_p, C.c_int]
    L.fl_observe_ws_words.argtypes = [C.POINTER(FlBatch)]
    L.fl_observe_ws_words.restype = C.c_int64
    L.fl_walk_tables.argtypes = [C.POINTER(FlBatch), C.c_int, P]
    L.fl_distance_map_ids.argtypes = [C.POINTER(FlBatch), P, C.c_int64, P]
    L.fl_walk_tables_ids.argtypes = [C.POINTER(FlBatch), C.c_int, P, C.c_int64, P]
    L.fl_step.argtypes = [C.POINTER(FlBatch), P, P, P, C.c_uint32, P]
    L.fl_observe.argtypes = [C.POINTER(FlBatch)] + [P] * 8
    L.fl_step_observe_host.argtypes = [C.POINTER(FlBatch), P, P, C.POINTER(FlObsBuffers), C.POINTER(FlObsBuffers),
                                       C.c_uint32, C.c_int, P, P]
    L.fl_step_observe_host_compact.argtypes = [C.POINTER(FlBatch), P, P, C.POINTER(FlObsBuffers), C.POINTER(FlObsBuffers), P, P,
                                               C.POINTER(C.c_uint64), C.c_uint32, C.c_int, P, P]
    L.fl_step_observe_host_compact.restype = C.c_int
    L.fl_wire_bytes.argtypes = [C.POINTER(FlBatch), C.c_int]
    L.fl_wire_bytes.restype = C.c_size_t
    L.fl_host_threads.argtypes = [C.c_int]
    L.fl_host_threads.restype = C.c_int
    L.fl_observe_plan.argtypes = [C.POINTER(FlBatch), P, C.c_int]
    L.fl_observe_plan.restype = C.c_int
    L.fl_batch_slice.argtypes = [C.POINTER(FlBatch), C.c_int64, C.c_int64, C.POINTER(FlBatch)]
    L.fl_copy_envs.argtypes = [C.POINTER(FlBatch), C.POINTER(FlBatch), P, P, C.c_int64, C.c_uint32, C.POINTER(FlObsBuffers),
                               C.POINTER(FlObsBuffers), P]
    L.fl_profile_num_kernels.restype = C.c_int
    L.fl_profile_kernel_name.restype = C.c_char_p
    L.fl_profile_kernel_name.argtypes = [C.c_int]
    L.fl_profile_enable.argtypes = [C.c_int]
    L.fl_profile_enable.restype = None
    L.fl_profile_collect.argtypes = [P, P, C.c_int]
    L.fl_profile_collect.restype = C.c_int
    for f in ("fl_distance_map", "fl_distance_map_ids", "fl_walk_tables", "fl_walk_tables_ids", "fl_reset", "fl_reset_ex", "fl_step", "fl_observe", "fl_step_observe_host", "fl_batch_slice", "fl_copy_envs"):
        getattr(L, f).restype = C.c_int
    if L.fl_batch_sizeof() != C.sizeof(FlBatch):
        raise FlatlandB200Error("FlBatch layout mismatch: library %d bytes, binding %d bytes"
                                % (L.fl_batch_sizeof(), C.sizeof(FlBatch)))
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise FlatlandB200Error("%s (code %d)" % (lib().fl_error_string(rc).decode(), rc))
