"""ctypes binding of libddz_b200.so -- the C-ABI declared in include/ddz_b200.h.

There is no CPU fallback: if the library is missing this module raises at import, and every launcher
raises when the CUDA runtime reports an error (e.g. no device)."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DDZ_LIB") or os.path.join(HERE, "libddz_b200.so")   # DDZ_LIB: developer builds

E_ARG, E_CUDA = -1, -2
FACE_FIRST, FACE_COMPLICATED, FACE_COOPERATION, FACE_SIMPLIFY = range(4)
CHOICE_INDEX, CHOICE_MOD, CHOICE_PHILOX, CHOICE_MOVE = range(4)
MAX_LEGAL = 512
STEPNO_AUTO = 0xFFFFFFFF
PIPE_DEPTH = 4
ABI_VERSION = 3

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc, sm_100a). The batched env has no CPU fallback." % LIB_PATH)

EXPORTS = ("ddz_abi_version", "ddz_prob_form", "ddz_set_tile_order", "ddz_face_channels", "ddz_state_bytes", "ddz_workspace_bytes", "ddz_last_error",
           "ddz_reset", "ddz_observe", "ddz_step", "ddz_rollout_step", "ddz_legal_moves", "ddz_encode_actions",
           "ddz_encode_face", "ddz_select_actions", "ddz_kth_moves", "ddz_playout", "ddz_pipe_create", "ddz_pipe_destroy",
           "ddz_pipe_step", "ddz_pipe_wait", "ddz_pipe_refill", "ddz_pipe_flush", "ddz_rollout_steps", "ddz_encode_state_actions", "ddz_legal_count", "ddz_legal_emit", "ddz_rows_alloc", "ddz_rows_free",
           "ddz_mpipe_create", "ddz_mpipe_destroy", "ddz_mpipe_step", "ddz_mpipe_wait", "ddz_mpipe_refill", "ddz_mpipe_flush", "ddz_mpipe_join",
           "ddz_mcts_moves", "ddz_playout_pruned", "ddz_q_features", "ddz_uct_workspace_bytes", "ddz_uct_search",
           "ddz_determinize", "ddz_uct_pool", "ddz_encode_face_gather", "ddz_move_ids", "ddz_moves_of_ids", "ddz_legal_mask",
           "ddz_policy_sample", "ddz_policy_logprob", "ddz_policy_logprob_backward", "ddz_policy_linear_logits",
           "ddz_policy_linear_sample", "ddz_policy_linear_logprob", "ddz_policy_linear_backward",
           "ddz_policy_linear_workspace_bytes", "ddz_policy_linear_grad_weight")

lib = C.CDLL(LIB_PATH)
_missing = [name for name in EXPORTS if not hasattr(lib, name)]
if _missing:
    raise ImportError("%s is older than include/ddz_b200.h (no %s): rebuild it with "
                      "`python -c 'import __graft_entry__ as g; g.build()'`" % (LIB_PATH, ", ".join(_missing)))
_vp, _i, _i64, _u64, _u32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_uint32

lib.ddz_abi_version.restype = _i
lib.ddz_prob_form.restype = _i
lib.ddz_set_tile_order.argtypes = [_i]
TILES_AUTO, TILES_TICKET = 0, 1


def set_tile_order(mode):
    """"auto" (default) or "ticket": ask for ticket-ordered tiles when other kernels (a Q-network, a collective) share the
    GPU with the env launches (include/ddz_b200.h, ddz_set_tile_order).  Returns the previous mode."""
    m = {"auto": TILES_AUTO, "ticket": TILES_TICKET}[mode] if isinstance(mode, str) else int(mode)
    prev = lib.ddz_set_tile_order(m)
    if prev < 0:
        raise ValueError("unknown tile order %r" % (mode,))
    return "ticket" if prev == TILES_TICKET else "auto"

lib.ddz_face_channels.argtypes = [_i]
lib.ddz_state_bytes.argtypes = [_i]
lib.ddz_state_bytes.restype = C.c_size_t
lib.ddz_workspace_bytes.argtypes = [_i]
lib.ddz_workspace_bytes.restype = C.c_size_t
lib.ddz_last_error.restype = C.c_char_p
lib.ddz_reset.argtypes = [_vp, _vp, _vp, _i, _i, _vp, _i, _vp]
lib.ddz_observe.argtypes = [_vp, _vp, _i, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp]
lib.ddz_step.argtypes = [_vp, _vp, _vp, _vp, _i, _u64, _u64, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]
lib.ddz_rollout_step.argtypes = [_vp, _vp, _i, _vp, _vp, _vp, _i, _u64, _u64, _u32, _vp, _vp, _vp, _i,
                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp]
lib.ddz_rollout_steps.argtypes = [_vp, _vp, _i, _i, _vp, _vp, _vp, _i, _u64, _u64, _u32, _vp, _vp, _vp, _i,
                                  _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp]
lib.ddz_legal_moves.argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _i, _vp]
lib.ddz_encode_actions.argtypes = [_vp, _i64, _vp, _vp]
lib.ddz_encode_face.argtypes = [_vp, _i, _vp, _i, _vp]
lib.ddz_encode_face_gather.argtypes = [_vp, _i, _vp, _i64, _vp, _vp, _vp, _i, _i, _vp]
ROWS_SPLIT, ROWS_CONCAT = 0, 1
STATE_WORDS = 19                     # int32 words of one env in a library state (uint64 hand/hist/recent [3], uint32 meta)
lib.ddz_kth_moves.argtypes = [_vp, _vp, _vp, _vp, _vp, _i, _vp]
lib.ddz_playout.argtypes = [_vp, _i, _u64, _u64, _u32, _vp, _vp, _vp, _i, _vp]
lib.ddz_playout_pruned.argtypes = lib.ddz_playout.argtypes
lib.ddz_mcts_moves.argtypes = [_vp, _vp, _vp, _vp, _i, _vp]
MCTS_MAX_MOVES = 344
lib.ddz_uct_workspace_bytes.argtypes = [_i, _i]
lib.ddz_uct_workspace_bytes.restype = C.c_size_t
lib.ddz_uct_search.argtypes = [_vp, _vp, _vp, _i, _i, _i, C.c_double, _vp, _u64, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]
UCT_MAX_BUDGET, UCT_MAX_WIDTH, UCT_MAX_PLAYOUTS, UCT_NODE_BYTES = 65536, 1024, 1 << 24, 160
lib.ddz_determinize.argtypes = [_vp, _vp, _i, _u64, _u64, _vp, _vp, _i, _vp]
lib.ddz_uct_pool.argtypes = [_vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp]
PIMC_MAX_DETERMINIZATIONS = 4096
lib.ddz_q_features.argtypes = [_vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _vp]
lib.ddz_pipe_create.restype = _vp
lib.ddz_pipe_destroy.argtypes = [_vp]
lib.ddz_pipe_destroy.restype = None
lib.ddz_pipe_step.argtypes = [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _u64, _u64, _u32, _vp, _vp, _vp, _i,
                              _vp, _vp, C.c_size_t, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp]
lib.ddz_pipe_wait.argtypes = [_vp, _i]
lib.ddz_pipe_refill.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]
lib.ddz_pipe_flush.argtypes = [_vp, _vp]
lib.ddz_encode_state_actions.argtypes = [_vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp]
lib.ddz_legal_count.argtypes = [_vp, _vp, _i, _vp]
lib.ddz_legal_emit.argtypes = [_vp, _vp, _vp, _vp, _i64, _vp, _i, _vp]
lib.ddz_rows_alloc.argtypes = [C.c_size_t, _i, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
lib.ddz_rows_free.argtypes = [_vp, C.c_size_t]


class GroupStep(C.Structure):
    """ddz_group_step of include/ddz_b200.h"""
    _fields_ = [("state", _vp), ("workspace", _vp), ("prev_offsets", _vp), ("prev_actions_u64", _vp),
                ("out_offsets", _vp), ("out_actions_u64", _vp), ("out_actions_f32", _vp), ("face", _vp),
                ("perm", _vp), ("lord_pile", _vp), ("reward", _vp),
                ("cap", _i64), ("env0", _u64), ("B", _i), ("stream", _vp)]


MPIPE_MAX_GROUPS = 16
lib.ddz_mpipe_create.argtypes = [_i]
lib.ddz_mpipe_create.restype = _vp
lib.ddz_mpipe_destroy.argtypes = [_vp]
lib.ddz_mpipe_destroy.restype = None
lib.ddz_mpipe_step.argtypes = [_vp, C.POINTER(GroupStep), _i, _vp, _vp, _u64, _u32, _vp, _i, _vp, _vp, _vp]
lib.ddz_mpipe_wait.argtypes = [_vp, _i]
lib.ddz_mpipe_refill.argtypes = [_vp, C.POINTER(GroupStep), C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _vp, _vp]
lib.ddz_mpipe_flush.argtypes = [_vp, C.POINTER(GroupStep)]
lib.ddz_mpipe_join.argtypes = [_vp, _vp]
lib.ddz_select_actions.argtypes = [_vp, _vp, C.c_float, _u64, _u64, _u32, _vp, _i, _vp]
lib.ddz_move_ids.argtypes = [_vp, _i64, _vp, _vp]
lib.ddz_moves_of_ids.argtypes = [_vp, _i64, _vp, _vp]
lib.ddz_legal_mask.argtypes = [_vp, _vp, _i64, _i, _vp, _vp, _i, _vp]
NUM_ACTION_IDS, MOVE_INVALID, MASK_WORDS = 13551, 0xFFFFFFFFFFFFFFFF, 424
MASK_BITS, MASK_BYTES = 0, 1
lib.ddz_policy_sample.argtypes = [_vp, _vp, _vp, _i64, _vp, _i, _i64, C.c_float, _u64, _u64, _u32, _vp, _vp, _vp, _vp, _vp,
                                  _vp, _i, _vp]
lib.ddz_policy_logprob.argtypes = [_vp, _vp, _i64, _vp, _i, _i64, _vp, _vp, _vp, _vp, _vp, _i, _vp]
lib.ddz_policy_logprob_backward.argtypes = [_vp, _vp, _i64, _vp, _i, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _i, _vp]
DTYPE_F32, DTYPE_BF16 = 0, 1
lib.ddz_policy_linear_logits.argtypes = [_vp, _vp, _i64, _vp, _vp, _vp, _i, _i, _i64, _vp, _vp, _i, _vp]
lib.ddz_policy_linear_sample.argtypes = [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i, _i, _i64, C.c_float, _u64, _u64, _u32, _vp,
                                         _vp, _vp, _vp, _vp, _vp, _i, _vp]
lib.ddz_policy_linear_logprob.argtypes = [_vp, _vp, _i64, _vp, _vp, _vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _i, _vp]
lib.ddz_policy_linear_backward.argtypes = [_vp, _vp, _i64, _vp, _vp, _vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64,
                                           _i, _vp]
lib.ddz_policy_linear_workspace_bytes.argtypes = [_i64, _i]
lib.ddz_policy_linear_workspace_bytes.restype = C.c_size_t
lib.ddz_policy_linear_grad_weight.argtypes = [_vp, _i64, _vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]
LINEAR_MAX_HIDDEN = 1024

if lib.ddz_abi_version() != ABI_VERSION:
    raise ImportError("libddz_b200.so ABI %d != binding %d: rebuild" % (lib.ddz_abi_version(), ABI_VERSION))


class DdzError(RuntimeError):
    pass


def check(rc, what):
    if rc == 0:
        return
    if rc == E_CUDA:
        raise DdzError("%s: CUDA failure: %s" % (what, lib.ddz_last_error().decode()))
    raise DdzError("%s: bad argument (code %d)" % (what, rc))


class _RowMemory:
    """one compressible device allocation (ddz_rows_alloc), exposed through __cuda_array_interface__"""

    def __init__(self, nbytes, device_index):
        ptr, mapped = C.c_void_p(), C.c_size_t()
        check(lib.ddz_rows_alloc(nbytes, device_index, C.byref(ptr), C.byref(mapped)), "ddz_rows_alloc")
        self.ptr, self.mapped, self.nbytes = ptr.value, mapped.value, nbytes
        self.__cuda_array_interface__ = {"shape": (nbytes // 4,), "typestr": "<f4", "data": (self.ptr, False), "version": 2}

    def __del__(self):
        ptr, self.ptr = getattr(self, "ptr", None), None
        if ptr and lib is not None:
            lib.ddz_rows_free(ptr, self.mapped)


def row_tensor(shape, device):
    """float32 tensor for thermometer rows (face / action one-hots) in COMPRESSIBLE device memory when the GPU has it
    (the L2 compresses the 0/1 rows on their way to HBM: +15 % store bandwidth for this data), else plain torch memory.
    DDZ_NO_COMPRESSION=1 forces plain memory."""
    import torch
    n = 1
    for d in shape:
        n *= int(d)
    dev = torch.device(device)
    if n == 0 or os.environ.get("DDZ_NO_COMPRESSION"):
        return torch.empty(tuple(shape), dtype=torch.float32, device=dev)
    index = dev.index if dev.index is not None else torch.cuda.current_device()
    try:
        with torch.cuda.device(index):
            torch.cuda.current_stream()                  # the primary context exists
            mem = _RowMemory(4 * n, index)
    except DdzError:
        return torch.empty(tuple(shape), dtype=torch.float32, device=dev)
    t = torch.as_tensor(mem, device=dev).view(tuple(shape))
    t._ddz_rows = mem                                    # keep the allocation alive with the tensor object
    return t
