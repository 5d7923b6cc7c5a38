"""ctypes binding of libdpt_b200.so (the C ABI in include/dpt_b200.h).

There is no CPU fallback: if the library is missing or a call fails, an exception is raised.
Tensors are passed as raw device pointers (``tensor.data_ptr()``) and work is enqueued on the
current torch CUDA stream; the library never synchronises (except the *_host entry points).
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DPT_B200_LIB") or os.path.join(_HERE, "libdpt_b200.so")   # override: A/B builds of the same ABI
ABI_VERSION = 9

OK, ERR_INVALID_ARG, ERR_CUDA, ERR_UNSUPPORTED = 0, -1, -2, -3


class DptError(RuntimeError):
    pass


class BanditInject(Structure):
    _fields_ = [("cov_idx", c_void_p), ("dir_probs", c_void_p), ("rand_idx", c_void_p), ("u", c_void_p),
                ("actions", c_void_p), ("z", c_void_p)]


BanditDump = BanditInject  # same layout, non-const


class DarkroomInject(Structure):
    _fields_ = [("states", c_void_p), ("actions", c_void_p), ("query", c_void_p)]


DarkroomDump = DarkroomInject


class OnlineInject(Structure):
    _fields_ = [("reward_z", c_void_p), ("ctrl_z", c_void_p), ("first_arm", c_void_p)]


OnlineDump = OnlineInject


class Gpt2Weights(Structure):
    _fields_ = [("horizon", c_int), ("state_dim", c_int), ("action_dim", c_int), ("n_layer", c_int), ("n_embd", c_int),
                ("n_positions", c_int),
                ("wpe", c_void_p), ("embed_w", c_void_p), ("embed_b", c_void_p), ("pred_w", c_void_p),
                ("pred_b", c_void_p), ("lnf_w", c_void_p), ("lnf_b", c_void_p),
                ("ln1_w", POINTER(c_void_p)), ("ln1_b", POINTER(c_void_p)), ("attn_w", POINTER(c_void_p)),
                ("attn_b", POINTER(c_void_p)), ("proj_w", POINTER(c_void_p)), ("proj_b", POINTER(c_void_p)),
                ("ln2_w", POINTER(c_void_p)), ("ln2_b", POINTER(c_void_p)), ("fc_w", POINTER(c_void_p)),
                ("fc_b", POINTER(c_void_p)), ("fc2_w", POINTER(c_void_p)), ("fc2_b", POINTER(c_void_p))]


class Gpt2Grads(Structure):
    _fields_ = [("wpe", c_void_p), ("embed_w", c_void_p), ("embed_b", c_void_p), ("pred_w", c_void_p), ("pred_b", c_void_p),
                ("lnf_w", c_void_p), ("lnf_b", c_void_p),
                ("ln1_w", POINTER(c_void_p)), ("ln1_b", POINTER(c_void_p)), ("attn_w", POINTER(c_void_p)),
                ("attn_b", POINTER(c_void_p)), ("proj_w", POINTER(c_void_p)), ("proj_b", POINTER(c_void_p)),
                ("ln2_w", POINTER(c_void_p)), ("ln2_b", POINTER(c_void_p)), ("fc_w", POINTER(c_void_p)),
                ("fc_b", POINTER(c_void_p)), ("fc2_w", POINTER(c_void_p)), ("fc2_b", POINTER(c_void_p))]


class Gpt2OnlineInject(Structure):
    _fields_ = [("reward_z", c_void_p), ("ctrl_u", c_void_p)]


class Gpt2OnlineDump(Structure):
    _fields_ = [("reward_z", c_void_p), ("ctrl_u", c_void_p), ("logits", c_void_p)]


class ExploreInject(Structure):
    _fields_ = [("ctrl_u", c_void_p), ("random_arm", c_void_p), ("reward_z", c_void_p)]


class ExploreDump(Structure):
    _fields_ = [("ctrl_u", c_void_p), ("random_arm", c_void_p), ("reward_z", c_void_p), ("logits_explorer", c_void_p),
                ("logits_exploiter", c_void_p)]


class OfflineParams(Structure):
    _fields_ = [("N", c_int), ("d", c_int), ("H_stride", c_int), ("K", c_int), ("horizons_host", c_void_p), ("ctrl_mask", c_int),
                ("lcb_const", c_double), ("thmp_std", c_double), ("thmp_prior_mean", c_double), ("thmp_prior_var", c_double),
                ("n_draws", c_int), ("arms", c_void_p), ("lin_d", c_int), ("linreg_const", c_double),
                ("learner_logits", c_void_p), ("logits_T", c_int), ("seed", c_uint64), ("env_id0", c_uint64),
                ("inject_z", c_void_p), ("dump_z", c_void_p)]


# name -> (restype, argtypes); every symbol include/dpt_b200.h declares
PROTOTYPES = {
    "dpt_version": (c_int, []),
    "dpt_last_error": (c_char_p, []),
    "dpt_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "dpt_bandit_sample_means": (c_int, [c_uint64, c_uint64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dpt_bandit_opt_action": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dpt_bandit_rollin": (c_int, [c_void_p, c_float, c_int, c_uint64, c_uint64, c_int, c_int, c_int, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p, POINTER(BanditInject), POINTER(BanditDump), c_void_p]),
    "dpt_bandit_rollin_host_f64": (c_int, [c_void_p, c_float, c_uint64, c_uint64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_uint64, c_void_p]),
    "dpt_bandit_rollin_host_last_d2h_bytes": (c_uint64, []),
    "dpt_host_write_peak": (c_double, [c_void_p, c_uint64, c_int]),
    "dpt_bandit_rollin_p2p": (c_int, [c_void_p, c_float, c_uint64, c_uint64, c_int, c_int, c_int, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p]),
    "dpt_peer_buffer_create": (c_int, [c_uint64, POINTER(c_void_p), c_void_p]),
    "dpt_peer_buffer_open": (c_int, [c_void_p, POINTER(c_void_p)]),
    "dpt_peer_buffer_close": (c_int, [c_void_p]),
    "dpt_peer_buffer_destroy": (c_int, [c_void_p]),
    "dpt_peer_buffer_read": (c_int, [c_void_p, c_void_p, c_uint64, c_void_p]),
    "dpt_peer_buffer_zero": (c_int, [c_void_p, c_uint64, c_void_p]),
    "dpt_bandit_rollin_host_scratch_bytes": (c_uint64, [c_int, c_int, c_int]),
    "dpt_bandit_rollin_host": (c_int, [c_void_p, c_float, c_uint64, c_uint64, c_int, c_int, c_int, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_uint64, c_void_p]),
    "dpt_darkroom_rollin": (c_int, [c_void_p, c_void_p, c_int, c_int, c_uint64, c_uint64, c_int, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    POINTER(DarkroomInject), POINTER(DarkroomDump), c_void_p]),
    "dpt_darkroom_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dpt_darkroom_opt_action": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "dpt_gpu_bandit_step": (c_int, [c_void_p, c_void_p, c_float, c_int, c_uint64, c_uint64, c_int64, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "dpt_selftest_div": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "dpt_debug_online_impl": (c_int, [c_int]),
    "dpt_arm_stats": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dpt_online_loop": (c_int, [c_int, c_double, c_double, c_double, c_void_p, c_void_p, c_int, c_double, c_int, c_uint64,
                                c_uint64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p, POINTER(OnlineInject), POINTER(OnlineDump), c_void_p]),
    "dpt_offline_eval": (c_int, [POINTER(OfflineParams), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dpt_debug_umma_gemm": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "dpt_gpt2_create": (c_int, [POINTER(Gpt2Weights), POINTER(c_void_p), c_void_p]),
    "dpt_gpt2_destroy": (c_int, [c_void_p]),
    "dpt_gpt2_forward_workspace_bytes": (c_uint64, [c_void_p, c_int, c_int, c_int]),
    "dpt_gpt2_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                 c_int, c_int, c_int, c_void_p, c_void_p, c_uint64, c_void_p]),
    "dpt_gpt2_train_workspace_bytes": (c_uint64, [POINTER(Gpt2Weights), c_int, c_int]),
    "dpt_gpt2_train_forward": (c_int, [POINTER(Gpt2Weights), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                       c_int, c_void_p, c_void_p, c_uint64, c_void_p]),
    "dpt_gpt2_train_backward": (c_int, [POINTER(Gpt2Weights), c_void_p, c_int, c_int, c_int, POINTER(Gpt2Grads), c_void_p,
                                        c_uint64, c_void_p]),
    "dpt_gpt2_train_population_workspace_bytes": (c_uint64, [POINTER(Gpt2Weights), c_int, c_int, c_int]),
    "dpt_gpt2_train_population_forward": (c_int, [POINTER(Gpt2Weights), c_int, POINTER(c_void_p), POINTER(c_void_p),
                                                  POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int,
                                                  c_int, POINTER(c_void_p), c_void_p, c_uint64, c_void_p]),
    "dpt_gpt2_train_population_backward": (c_int, [POINTER(Gpt2Weights), c_int, POINTER(c_void_p), c_int, c_int, c_int,
                                                   POINTER(Gpt2Grads), c_void_p, c_uint64, c_void_p]),
    "dpt_gpt2_train_population_workspace_bytes_ex": (c_uint64, [POINTER(Gpt2Weights), c_int, c_int, c_int, c_int]),
    "dpt_gpt2_train_population_forward_ex": (c_int, [POINTER(Gpt2Weights), c_int, POINTER(c_void_p), POINTER(c_void_p),
                                                     POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int,
                                                     c_int, c_int, POINTER(c_void_p), c_void_p, c_uint64, c_void_p]),
    "dpt_gpt2_train_population_backward_ex": (c_int, [POINTER(Gpt2Weights), c_int, POINTER(c_void_p), c_int, c_int, c_int, c_int,
                                                      POINTER(Gpt2Grads), c_void_p, c_uint64, c_void_p]),
    "dpt_ordered_sum_f32": (c_int, [POINTER(c_void_p), c_int, c_int64, c_void_p, c_void_p]),
    "dpt_darkroom_policy_rollout": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_uint64, c_uint64, c_int64,
                                            c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                            c_void_p]),
    "dpt_gpt2_decode_step": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_uint64, c_void_p, c_void_p]),
    "dpt_gpt2_online_kv_bytes": (c_uint64, [c_void_p, c_int, c_int, c_int]),
    "dpt_gpt2_online_loop": (c_int, [c_void_p, c_void_p, c_double, c_int, c_int, c_uint64, c_uint64, c_int, c_int, c_int,
                                     c_void_p, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     POINTER(Gpt2OnlineInject), POINTER(Gpt2OnlineDump), c_void_p]),
    "dpt_gpt2_online_loop_population": (c_int, [POINTER(c_void_p), c_int, c_void_p, c_double, c_int, c_int, c_uint64, c_uint64,
                                                c_int, c_int, c_int, c_void_p, c_uint64, POINTER(c_void_p), POINTER(c_void_p),
                                                POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                                POINTER(Gpt2OnlineInject), POINTER(Gpt2OnlineDump), c_void_p]),
    "dpt_gpt2_explore_exploit_rollout": (c_int, [c_void_p, c_void_p, c_void_p, c_double, c_int, c_uint64, c_uint64, c_int, c_int,
                                                 c_void_p, c_void_p, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                 POINTER(ExploreInject), POINTER(ExploreDump), c_void_p]),
}

_lib = None


def lib():
    """The loaded library.  Raises DptError (never falls back) when it is missing or stale."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DptError("CUDA extension missing: %s not built (run `python -c 'import __graft_entry__ as g; "
                           "g.build()'` or `make -C %s/csrc`); there is no CPU fallback" % (LIB_PATH, _HERE))
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            try:
                fn = getattr(l, name)
            except AttributeError:
                raise DptError("libdpt_b200.so does not export %s (stale build?)" % name)
            fn.restype, fn.argtypes = res, args
        if l.dpt_version() != ABI_VERSION:
            raise DptError("libdpt_b200.so ABI %d != expected %d" % (l.dpt_version(), ABI_VERSION))
        _lib = l
    return _lib


def check(rc, what):
    if rc != OK:
        msg = lib().dpt_last_error().decode("utf-8", "replace")
        if rc == ERR_INVALID_ARG:
            raise ValueError("%s: %s" % (what, msg))
        if rc == ERR_UNSUPPORTED:
            raise NotImplementedError("%s: %s" % (what, msg))
        raise DptError("%s failed (%d): %s" % (what, rc, msg))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL).  The tensor must be contiguous."""
    if t is None:
        return None
    if not t.is_contiguous():
        raise ValueError("non-contiguous tensor passed to the C ABI")
    return t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise DptError("no CUDA device: the DPT rollout hot path runs on B200 (sm_100a) only; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())
