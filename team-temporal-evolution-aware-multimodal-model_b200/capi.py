"""ctypes binding of ``libteam_b200.so`` (declared in ``include/team_b200.h``).

The library handle is module-global (never stored on an ``nn.Module``) so that the
reference's ``copy.deepcopy(self._network)`` (models/proof.py:297) keeps working.
There is deliberately no fallback: if the shared library is missing or a call fails a
``TeamB200Error`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libteam_b200.so")

D = 512
NUM_STATES = 10
MAX_TASKS = 64
DTYPE_F32, DTYPE_BF16 = 0, 1
MODE_F32, MODE_BF16 = 0, 1

EXPORTS = [
    "team_last_error", "team_version", "team_device_check",
    "team_segsum_workspace_bytes", "team_segsum", "team_segmean_finalize",
    "team_cosine_logits",
]


class TeamB200Error(RuntimeError):
    pass


class HeadWeights(C.Structure):
    _fields_ = ([("num_tasks", C.c_int32), ("prompts_per_task", C.c_int32)] +
                [(n, C.c_void_p * MAX_TASKS) for n in
                 ("w_img", "b_img", "w_text", "b_text", "w_state", "b_state", "prompts")] +
                [(n, C.c_void_p) for n in
                 ("state_emb", "w_q", "w_k", "w_v", "w_fc", "b_fc", "ln_g", "ln_b", "prototypes")] +
                [("num_classes", C.c_int32), ("num_frozen", C.c_int32),
                 ("w_frozen", C.c_void_p * 3), ("b_frozen", C.c_void_p * 3)])


class PeerComm(C.Structure):
    _fields_ = [("bufs", C.c_void_p * 8), ("flags", C.c_void_p * 8), ("multicast", C.c_void_p),
                ("rank", C.c_int32), ("world", C.c_int32), ("n_total", C.c_int64), ("split_at", C.c_int64)]


class HeadGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("w_img", "b_img", "w_text", "b_text", "w_state", "b_state", "prompts", "state_emb",
                 "w_q", "w_k", "w_v", "w_fc", "b_fc", "ln_g", "ln_b", "ev_w_fc", "ev_w_qkv")] + [("comm", C.POINTER(PeerComm)),
                                                                                                  ("g_own_rows", C.c_void_p)]


class Dropout(C.Structure):
    _fields_ = [("p", C.c_float), ("seed", C.c_uint64), ("offset", C.c_uint64), ("offset_dev", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class TgcnBlock(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("msg_w", "msg_b", "msg_ln_g", "msg_ln_b", "upd_w", "upd_b", "upd_ln_g", "upd_ln_b", "gate_w", "gate_b")]


class TgcnWeights(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in
                 ("node_w", "node_b", "node_ln_g", "node_ln_b", "time_w", "time_b", "time_ln_g", "time_ln_b")] +
                [("blocks", TgcnBlock * 8), ("num_blocks", C.c_int32), ("reserved", C.c_int32),
                 ("out_w", C.c_void_p), ("out_b", C.c_void_p)])


class DgcnLayer(C.Structure):
    _fields_ = [("w", C.c_void_p), ("b", C.c_void_p), ("ln_g", C.c_void_p), ("ln_b", C.c_void_p),
                ("in_dim", C.c_int32), ("out_dim", C.c_int32)]


class GemmDesc(C.Structure):
    _fields_ = [("a_mn", C.c_int32), ("b_mn", C.c_int32), ("M", C.c_int64), ("N", C.c_int64), ("K", C.c_int64),
                ("alpha", C.c_float), ("beta", C.c_float), ("A", C.c_void_p), ("lda", C.c_int64),
                ("B", C.c_void_p), ("ldb", C.c_int64), ("C", C.c_void_p), ("ldc", C.c_int64),
                ("C_bf16", C.c_void_p), ("ldc_bf16", C.c_int64), ("bias", C.c_void_p),
                ("a_mn2", C.c_int32), ("b_mn2", C.c_int32), ("K2", C.c_int64),
                ("A2", C.c_void_p), ("lda2", C.c_int64), ("B2", C.c_void_p), ("ldb2", C.c_int64)]


class LossShard(C.Structure):
    _fields_ = ([("mode", C.c_int32), ("rank", C.c_int32), ("world", C.c_int32), ("num_evo", C.c_int32),
                 ("batch", C.c_int64), ("num_classes", C.c_int64)] +
                [(n, C.c_void_p) for n in ("image", "text", "state", "own_rows", "logits", "labels", "state_ids", "evo",
                                           "evo_mask")] +
                [(n, C.c_float) for n in ("temperature", "logit_scale", "w_clip", "w_unicl")] +
                [("send", C.c_void_p * 3), ("gathered", C.c_void_p * 3)] +
                [(n, C.c_void_p) for n in ("g_image", "g_text", "g_state", "g_own_rows", "losses6", "workspace")] +
                [("workspace_bytes", C.c_size_t)])


_lib = None
_lock = threading.Lock()


def _declare(lib):
    vp, i64, i32, sz = C.c_void_p, C.c_int64, C.c_int, C.c_size_t
    lib.team_last_error.restype = C.c_char_p
    lib.team_last_error.argtypes = []
    lib.team_version.restype = i32
    lib.team_device_check.restype = i32
    lib.team_launch_count.restype = C.c_longlong
    lib.team_launch_count.argtypes = []
    lib.team_prof_enable.restype = i32
    lib.team_prof_enable.argtypes = [i32]
    lib.team_prof_collect.restype = i32
    lib.team_prof_collect.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong)]
    lib.team_segsum_workspace_bytes.restype = sz
    lib.team_segsum_workspace_bytes.argtypes = [i64, i64]
    lib.team_segsum.restype = i32
    lib.team_segsum.argtypes = [vp, i32, vp, vp, i64, i64, i64, i64, i32, vp, vp, vp, sz, vp]
    lib.team_segmean_finalize.restype = i32
    lib.team_segmean_finalize.argtypes = [vp, vp, i64, vp, i64, vp, vp, vp]
    lib.team_cosine_logits.restype = i32
    lib.team_cosine_logits.argtypes = [vp, i32, i64, vp, i64, vp, vp, vp, vp]
    if hasattr(lib, "team_gemm_f32"):
        lib.team_gemm_f32.restype = i32
        lib.team_gemm_f32.argtypes = [i32, i32, i64, i64, i64, C.c_float, vp, i64, vp, i64, C.c_float,
                                      vp, i64, vp, vp, sz, vp]
    if hasattr(lib, "team_gemm_bf16"):
        lib.team_gemm_bf16.restype = i32
        lib.team_gemm_bf16.argtypes = [i32, i32, i64, i64, i64, C.c_float, vp, vp, i64, vp, i64, C.c_float,
                                       vp, i64, vp, vp, sz, vp]
        lib.team_f32_to_bf16.restype = i32
        lib.team_f32_to_bf16.argtypes = [vp, i64, i64, i64, vp, vp, i64, vp]
    if hasattr(lib, "team_gemm_bf16_group"):
        lib.team_gemm_bf16_group.restype = i32
        lib.team_gemm_bf16_group.argtypes = [C.POINTER(GemmDesc), C.c_int32, vp, sz, vp]
    if hasattr(lib, "team_head_workspace_bytes"):
        lib.team_head_workspace_bytes.restype = sz
        lib.team_head_workspace_bytes.argtypes = [i64, C.c_int32, C.c_int32, C.c_int32, i32]
        lib.team_head_frozen_sums.restype = i32
        lib.team_head_frozen_sums.argtypes = [C.POINTER(HeadWeights), i32, vp, vp, vp]
        lib.team_head_own_rows_offset.restype = sz
        lib.team_head_own_rows_offset.argtypes = [i64, C.c_int32, C.c_int32, C.c_int32, i32]
        lib.team_head_tri_fwd.restype = i32
        lib.team_head_tri_fwd.argtypes = [C.POINTER(HeadWeights), i32, i64, vp, vp, vp, vp, i64,
                                          vp, vp, vp, vp, vp, vp, vp, sz, vp, C.POINTER(Dropout)]
        lib.team_head_tri_bwd.restype = i32
        lib.team_head_tri_bwd.argtypes = [C.POINTER(HeadWeights), i32, i64, vp, vp, vp, vp, vp, vp, vp,
                                          C.POINTER(HeadGrads), vp, sz, vp, C.POINTER(Dropout)]
        lib.team_head_dropout_workspace_bytes.restype = sz
        lib.team_head_dropout_workspace_bytes.argtypes = [i64, C.c_int32, C.c_int32, i32]
        lib.team_u64_add.restype = i32
        lib.team_u64_add.argtypes = [vp, C.c_uint64, vp]
        lib.team_head_encode.restype = i32
        lib.team_head_encode.argtypes = [C.POINTER(HeadWeights), i32, i32, vp, i64, i32, vp, vp, sz, vp]
        lib.team_peer_allreduce_flag_bytes.restype = sz
        lib.team_peer_allreduce_flag_bytes.argtypes = []
        lib.team_peer_allreduce_f32.restype = i32
        lib.team_peer_allreduce_f32.argtypes = [C.POINTER(vp), C.POINTER(vp), vp, i32, i32, i64, vp]
        lib.team_peer_allreduce_status.restype = i32
        lib.team_peer_allreduce_status.argtypes = [vp, vp, C.POINTER(C.c_uint32)]
        lib.team_peer_allgather.restype = i32
        lib.team_peer_allgather.argtypes = [C.POINTER(vp), C.POINTER(vp), vp, i32, i32, i64, vp]
        lib.team_adamw_step.restype = i32
        lib.team_adamw_step.argtypes = [i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64),
                                        C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, i64, vp]
        lib.team_adamw_step_graph.restype = i32
        lib.team_adamw_step_graph.argtypes = [i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64),
                                              C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, vp, i32, vp]
        lib.team_copy_batch.restype = i32
        lib.team_copy_batch.argtypes = [vp, vp, vp, vp, i64, vp, vp, vp, vp, vp]
        lib.team_ce_total.restype = i32
        lib.team_ce_total.argtypes = [vp, vp, i64, i64, C.c_float, C.c_float, vp, vp]
        lib.team_loss_workspace_bytes.restype = sz
        lib.team_loss_workspace_bytes.argtypes = [i64]
        lib.team_unicl_loss.restype = i32
        lib.team_unicl_loss.argtypes = [i32, vp, vp, vp, vp, i64, C.c_float, C.c_float, vp, vp, vp, vp, vp, sz, vp]
        lib.team_loss_evo_workspace_bytes.restype = sz
        lib.team_loss_evo_workspace_bytes.argtypes = [i64, i32]
        lib.team_unicl_loss_evo.restype = i32
        lib.team_unicl_loss_evo.argtypes = [i32, vp, vp, vp, vp, vp, vp, vp, i32, i64, C.c_float, C.c_float, vp, vp, vp, vp, vp, sz, vp]
        lib.team_clip_loss.restype = i32
        lib.team_clip_loss.argtypes = [i32, vp, vp, i64, C.c_float, C.c_float, vp, vp, vp, vp, sz, vp]
        lib.team_loss_shard_phases.restype = i32
        lib.team_loss_shard_phases.argtypes = [C.c_int32]
        lib.team_loss_shard_workspace_bytes.restype = sz
        lib.team_loss_shard_workspace_bytes.argtypes = [C.c_int32, i64, C.c_int32, C.c_int32]
        lib.team_loss_shard_xchg_bytes.restype = sz
        lib.team_loss_shard_xchg_bytes.argtypes = [C.c_int32, i64, C.c_int32, C.c_int32]
        lib.team_loss_shard_run.restype = i32
        lib.team_loss_shard_run.argtypes = [C.c_int32, C.POINTER(LossShard), vp]
        lib.team_head_tri_classtext_fwd.restype = i32
        lib.team_head_tri_classtext_fwd.argtypes = [C.POINTER(HeadWeights), i32, i64, vp, vp, i64, vp, vp, vp, vp, vp, vp, sz, vp]
        lib.team_head_proof_fwd.restype = i32
        lib.team_head_proof_fwd.argtypes = [C.POINTER(HeadWeights), i32, i64, vp, vp, i64, i32, vp, vp, vp, vp, sz, vp]
        lib.team_head_encode_rows_bwd.restype = i32
        lib.team_head_encode_rows_bwd.argtypes = [C.POINTER(HeadWeights), i32, i32, vp, i64, i32, vp, vp, vp, vp, vp, sz, vp]
        lib.team_herding_workspace_bytes.restype = sz
        lib.team_herding_workspace_bytes.argtypes = [i64]
        lib.team_herding_select.restype = i32
        lib.team_herding_select.argtypes = [vp, vp, i32, i32, i64, vp, vp, vp, vp, sz, vp]
        lib.team_mha_workspace_bytes.restype = sz
        lib.team_mha_workspace_bytes.argtypes = [i64, i64, i64]
        lib.team_mha_fwd.restype = i32
        lib.team_mha_fwd.argtypes = [i32, i64, i64, i64] + [vp] * 10 + [C.c_float, C.c_uint64, C.c_uint64] + [vp, vp, sz, vp]
        lib.team_mha_bwd.restype = i32
        lib.team_mha_bwd.argtypes = [i32, i64, i64, i64] + [vp] * 8 + [C.c_float, C.c_uint64, C.c_uint64] + [vp] * 11 + [vp, sz, vp]
        lib.team_dropout_keep_mask.restype = i32
        lib.team_dropout_keep_mask.argtypes = [vp, i64, C.c_float, C.c_uint64, C.c_uint64, vp]
        lib.team_mean_mid.restype = i32
        lib.team_mean_mid.argtypes = [vp, vp, i64, i64, i64, vp]
        lib.team_mean_mid_bwd.restype = i32
        lib.team_mean_mid_bwd.argtypes = [vp, vp, i64, i64, i64, vp]
        lib.team_head_encode_bwd.restype = i32
        lib.team_head_encode_bwd.argtypes = [C.POINTER(HeadWeights), i32, i32, vp, i64, i32, vp, vp, vp, vp, sz, vp]


def _declare_graph(lib):
    vp, i64, i32, sz, dbl = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_double
    lib.team_tgcn_workspace_bytes.restype = sz
    lib.team_tgcn_workspace_bytes.argtypes = [i64]
    lib.team_tgcn_forward.restype = i32
    lib.team_tgcn_forward.argtypes = [C.POINTER(TgcnWeights), vp, vp, i64, vp, vp, vp, vp, vp, sz, vp]
    lib.team_pairwise_state_dist.restype = i32
    lib.team_pairwise_state_dist.argtypes = [vp, vp, i64, vp, vp, vp, sz, vp]
    lib.team_sync_prototypes.restype = i32
    lib.team_sync_prototypes.argtypes = [vp, vp, vp, vp, i64, vp, vp]
    lib.team_rows_normalize.restype = i32
    lib.team_rows_normalize.argtypes = [vp, i64, vp]
    lib.team_group_mean.restype = i32
    lib.team_group_mean.argtypes = [vp, vp, vp, i64, vp, vp]
    lib.team_dist_matrix.restype = i32
    lib.team_dist_matrix.argtypes = [vp, C.c_int32, vp, vp]
    lib.team_dist_ema.restype = i32
    lib.team_dist_ema.argtypes = [vp, C.c_int32, vp, vp, C.c_int32, dbl, vp]
    lib.team_state_dist_forward.restype = i32
    lib.team_state_dist_forward.argtypes = [vp, vp, vp, dbl, vp, vp]
    lib.team_dgcn_workspace_bytes.restype = sz
    lib.team_dgcn_workspace_bytes.argtypes = [i64, C.c_int32]
    lib.team_dgcn_forward.restype = i32
    lib.team_dgcn_forward.argtypes = [C.POINTER(DgcnLayer), C.c_int32, vp, i64, vp, vp, vp, vp, vp, sz, vp]


def lib():
    """The loaded shared library; raises TeamB200Error if it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise TeamB200Error(
                        f"{LIB_PATH} not found - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU/PyTorch fallback)")
                handle = C.CDLL(LIB_PATH)
                _declare(handle)
                _declare_graph(handle)
                _lib = handle
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().team_last_error().decode("utf-8", "replace")
        raise TeamB200Error(f"{what} failed with code {rc}: {msg}")


_device_ok = set()


def require_device():
    """Fail loudly unless torch sees a CUDA device of compute capability 10.x (checked once per device)."""
    import torch
    if not torch.cuda.is_available():
        raise TeamB200Error("team_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.cuda.current_device()
    if dev not in _device_ok:
        check(lib().team_device_check(), "team_device_check")
        _device_ok.add(dev)
