"""ctypes binding of liblec_b200.so (the C ABI declared in include/lec_b200.h).

There is no fallback: if the shared library has not been built (`python -c "import
__graft_entry__ as g; g.build()"` or `make -C learning_embeddings_b200/csrc`) every op raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "liblec_b200.so")

GEOM = {"euc": 0, "hyp": 1, "oe": 2, "poincare": 4, "lorentz": 5}
ROWS_NONE, ROWS_EUC_SOFTCLIP, ROWS_HYP_SHELL, ROWS_HYP_TANH, ROWS_HYP_TANH_FEAT = 0, 1, 2, 3, 4
PREC_F32, PREC_F64CORE = 0, 1
ABI_VERSION = 14

EXPORTS = (
    "lec_abi_version", "lec_error_string", "lec_launch_count", "lec_set_pdl", "lec_index_errors", "lec_rows_fwd", "lec_rows_bwd",
    "lec_featnet_supported", "lec_featnet_fwd", "lec_featnet_wgrad",
    "lec_reduce_replicas", "lec_pairs_flat", "lec_pairs_grouped", "lec_pairs_poincare", "lec_pairs_lorentz", "lec_energy_dense", "lec_energy_dense_bwd",
    "lec_rsgd_update", "lec_exchange_packets", "lec_exchange_bytes", "lec_update_rows", "lec_cone_step", "lec_score_topk", "lec_score_topk_ex",
    "lec_score_tc_supported",
    "lec_score_workspace_bytes", "lec_score_topk_tc", "lec_mt_seed", "lec_mt_uint32", "lec_mt_randbelow",
    "lec_sample_negatives", "lec_sample_negatives_philox", "lec_philox_below", "lec_f1_workspace_bytes", "lec_f1_sweep",
    "lec_classify_counts", "lec_caption_hinge",
    "lec_recon_workspace_bytes", "lec_recon_counter_bytes", "lec_recon_pass", "lec_recon_pass_dag", "lec_recon_finish",
    "lec_rank_workspace_bytes", "lec_rank_run", "lec_rank_run_heldout", "lec_recon_pass_heldout", "lec_recon_finish_at",
    "lec_host_pipe_create", "lec_host_pipe_destroy", "lec_host_pipe_submit", "lec_host_pipe_wait",
)


class LecError(RuntimeError):
    pass


class LecUpdate(ctypes.Structure):
    """lec_update_t of include/lec_b200.h."""
    _fields_ = [
        ("rule", ctypes.c_int), ("row_mode", ctypes.c_int), ("geom", ctypes.c_int), ("lambda_mode", ctypes.c_int),
        ("hyp_rescale", ctypes.c_int), ("project_shell", ctypes.c_int),
        ("K", ctypes.c_float), ("lr", ctypes.c_float), ("r_in", ctypes.c_float),
        ("momentum", ctypes.c_float), ("beta1", ctypes.c_float), ("beta2", ctypes.c_float), ("eps", ctypes.c_float),
        ("opt_step", ctypes.c_int64),
        ("table", ctypes.c_void_p), ("n", ctypes.c_int64), ("D", ctypes.c_int), ("ld", ctypes.c_int),
        ("grad_rows", ctypes.c_void_p), ("grad_replicas", ctypes.c_int), ("grad_stride", ctypes.c_int64),
        ("state_m", ctypes.c_void_p), ("state_v", ctypes.c_void_p),
        ("rows_out", ctypes.c_void_p), ("aux_out", ctypes.c_void_p), ("grad_out", ctypes.c_void_p),
        ("loss_acc", ctypes.c_void_p), ("loss_step", ctypes.c_void_p),
    ]


class LecExchange(ctypes.Structure):
    """lec_exchange_t of include/lec_b200.h."""
    _fields_ = [
        ("peer_bufs", ctypes.c_void_p), ("slot_packets", ctypes.c_int64), ("world", ctypes.c_int), ("rank", ctypes.c_int),
        ("slot", ctypes.c_int), ("tag", ctypes.c_uint32),
        ("loss_global", ctypes.c_void_p), ("error", ctypes.c_void_p), ("timeout_ms", ctypes.c_int64),
        ("mode", ctypes.c_int), ("phases", ctypes.c_int),
    ]


class LecStep(ctypes.Structure):
    """lec_step_t of include/lec_b200.h."""
    _fields_ = [
        ("geom", ctypes.c_int), ("precision", ctypes.c_int), ("fused", ctypes.c_int),
        ("alpha", ctypes.c_float),
        ("pos_from", ctypes.c_void_p), ("pos_to", ctypes.c_void_p), ("neg_to", ctypes.c_void_p),
        ("neg_from", ctypes.c_void_p), ("idx_bytes", ctypes.c_int),
        ("B", ctypes.c_int64), ("N", ctypes.c_int),
        ("w_pos", ctypes.c_void_p), ("w_neg", ctypes.c_void_p),
        ("E_pos", ctypes.c_void_p), ("E_neg", ctypes.c_void_p),
        ("ev_pairs_start", ctypes.c_void_p), ("ev_pairs_stop", ctypes.c_void_p),
        ("upd", LecUpdate), ("xchg", LecExchange),
    ]


class LecHostSample(ctypes.Structure):
    """lec_host_sample_t of include/lec_b200.h."""
    _fields_ = [("graph", ctypes.c_void_p), ("seed", ctypes.c_uint64), ("stream_id", ctypes.c_uint64), ("status", ctypes.c_void_p)]


class LecRecon(ctypes.Structure):
    """lec_recon_t of include/lec_b200.h."""
    _fields_ = [
        ("geom", ctypes.c_int), ("K", ctypes.c_float),
        ("rows", ctypes.c_void_p), ("n", ctypes.c_int64), ("D", ctypes.c_int), ("ld", ctypes.c_int),
        ("tin", ctypes.c_void_p), ("tout", ctypes.c_void_p),
        ("u_begin", ctypes.c_int64), ("u_end", ctypes.c_int64),
        ("workspace", ctypes.c_void_p), ("workspace_bytes", ctypes.c_int64),
    ]


class LecReconExtra(ctypes.Structure):
    """lec_recon_extra_t of include/lec_b200.h."""
    _fields_ = [("ptr", ctypes.c_void_p), ("lo", ctypes.c_void_p), ("hi", ctypes.c_void_p), ("count", ctypes.c_int64)]


class LecRank(ctypes.Structure):
    """lec_rank_t of include/lec_b200.h."""
    _fields_ = [
        ("geom", ctypes.c_int), ("K", ctypes.c_float),
        ("rows", ctypes.c_void_p), ("n", ctypes.c_int64), ("D", ctypes.c_int), ("ld", ctypes.c_int),
        ("tin", ctypes.c_void_p), ("tout", ctypes.c_void_p), ("extra", ctypes.POINTER(LecReconExtra)),
        ("pos_ptr", ctypes.c_void_p), ("n_pos", ctypes.c_int64),
        ("u_begin", ctypes.c_int64), ("u_end", ctypes.c_int64),
        ("workspace", ctypes.c_void_p), ("workspace_bytes", ctypes.c_int64),
        ("stage_ms", ctypes.POINTER(ctypes.c_float)),
    ]


class LecHeldout(ctypes.Structure):
    """lec_heldout_t of include/lec_b200.h."""
    _fields_ = [("closure_ptr", ctypes.c_void_p), ("slot_map", ctypes.c_void_p), ("xcum", ctypes.c_void_p),
                ("n_closure", ctypes.c_int64)]


UPD_NONE, UPD_RSGD, UPD_SGD, UPD_ADAM, UPD_RSGD_RETRACT, UPD_RSGD_LORENTZ = 0, 1, 2, 3, 4, 5
XCHG_ONE_SHOT, XCHG_TWO_SHOT = 0, 1

_lib = None


def _p(t):
    """device pointer of a tensor (or NULL)."""
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LecError(
                "liblec_b200.so is not built (%s). Run __graft_entry__.build(); there is no CPU or eager fallback."
                % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        c_i, c_i64, c_f, c_vp = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p
        L.lec_abi_version.restype = c_i
        L.lec_error_string.restype = ctypes.c_char_p
        L.lec_error_string.argtypes = [c_i]
        L.lec_launch_count.restype = c_i64
        L.lec_rows_fwd.argtypes = [c_vp, c_i64, c_i, c_i, c_i, c_f, c_vp, c_i, c_vp, c_vp, c_i, c_i64, c_vp, c_vp]
        L.lec_rows_bwd.argtypes = [c_vp, c_vp, c_i, c_i64, c_i64, c_i, c_i, c_i, c_f, c_vp, c_i, c_vp]
        L.lec_set_pdl.argtypes = [c_i]
        L.lec_featnet_supported.argtypes = [c_i, c_i]
        L.lec_featnet_fwd.argtypes = [c_vp, c_i64, c_i, c_vp, c_i, c_i64, c_vp, c_vp, c_i, c_vp, c_vp]
        L.lec_featnet_wgrad.argtypes = [c_vp, c_i64, c_i, c_vp, c_i, c_i64, c_vp, c_i, c_vp, c_i, c_i64, c_vp]
        L.lec_reduce_replicas.argtypes = [c_vp, c_i, c_i64, c_vp, c_vp]
        L.lec_pairs_flat.argtypes = [c_i, c_i, c_vp, c_vp, c_i64, c_i, c_i, c_vp, c_vp, c_i, c_vp, c_vp, c_i64, c_f, c_f,
                                     c_vp, c_vp, c_vp, c_i, c_vp]
        L.lec_pairs_grouped.argtypes = [c_i, c_i, c_vp, c_vp, c_i64, c_i, c_i, c_vp, c_vp, c_vp, c_vp, c_i, c_i64, c_i,
                                        c_vp, c_vp, c_f, c_f, c_vp, c_vp, c_vp, c_vp, c_i, c_vp]
        L.lec_pairs_poincare.argtypes = [c_i, c_vp, c_i64, c_i, c_i, c_vp, c_vp, c_vp, c_i, c_i64, c_i, c_vp, c_vp, c_vp,
                                         c_vp, c_i, c_vp]
        L.lec_pairs_lorentz.argtypes = [c_i, c_vp, c_i64, c_i, c_i, c_vp, c_vp, c_vp, c_i, c_i64, c_i, c_vp, c_vp, c_vp,
                                        c_vp, c_i, c_vp]
        L.lec_energy_dense.argtypes = [c_i, c_i, c_vp, c_vp, c_i64, c_i, c_f, c_vp, c_vp]
        L.lec_energy_dense_bwd.argtypes = [c_i, c_i, c_vp, c_vp, c_vp, c_i64, c_i, c_f, c_vp, c_vp, c_vp]
        L.lec_rsgd_update.argtypes = [c_vp, c_vp, c_i, c_i64, c_i, c_i, c_f, c_f, c_i, c_vp, c_vp]
        L.lec_index_errors.argtypes = [c_vp, c_i, c_vp]
        L.lec_exchange_packets.argtypes = [c_i64, c_i]
        L.lec_exchange_packets.restype = c_i64
        L.lec_exchange_bytes.argtypes = [c_i64, c_i, c_i, c_i]
        L.lec_exchange_bytes.restype = c_i64
        L.lec_update_rows.argtypes = [ctypes.POINTER(LecUpdate), ctypes.POINTER(LecExchange), c_vp]
        L.lec_cone_step.argtypes = [ctypes.POINTER(LecStep), c_vp]
        L.lec_score_topk.argtypes = [c_i, c_i, c_vp, c_i64, c_vp, c_i64, c_i, c_f, c_vp, c_vp, c_i, c_i, c_vp, c_vp,
                                     c_vp, c_vp]
        L.lec_score_topk_ex.argtypes = [c_i, c_i, c_vp, c_i64, c_vp, c_i64, c_i, c_f, c_vp, c_vp, c_i, c_i, c_vp, c_i,
                                        c_vp, c_vp, c_vp]
        L.lec_score_tc_supported.argtypes = [c_i, c_i, c_i, c_i64, c_i]
        L.lec_score_workspace_bytes.argtypes = [c_i64, c_i, c_i]
        L.lec_score_workspace_bytes.restype = c_i64
        L.lec_score_topk_tc.argtypes = [c_i, c_i, c_vp, c_i64, c_vp, c_i64, c_i, c_f, c_vp, c_vp, c_i, c_i, c_vp, c_vp,
                                        c_vp, c_vp, c_i64, c_vp]
        c_u32, c_u64 = ctypes.c_uint32, ctypes.c_uint64
        L.lec_mt_seed.argtypes = [c_vp, c_vp, c_i]
        L.lec_mt_uint32.argtypes = [c_vp]
        L.lec_mt_uint32.restype = c_u32
        L.lec_mt_randbelow.argtypes = [c_vp, c_u32]
        L.lec_mt_randbelow.restype = c_i64
        L.lec_sample_negatives.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_i, c_vp, c_vp]
        L.lec_sample_negatives_philox.argtypes = [c_vp, c_vp, c_vp, c_i, c_i64, c_i, c_u64, c_u64, c_vp, c_vp, c_vp, c_vp]
        L.lec_philox_below.argtypes = [c_u64, c_u64, c_u64, c_u64]
        L.lec_philox_below.restype = c_i64
        L.lec_f1_workspace_bytes.restype = c_i64
        L.lec_f1_sweep.argtypes = [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp]
        L.lec_classify_counts.argtypes = [c_vp, c_vp, c_i64, c_i, c_i, c_vp, c_i, c_i64, c_vp, c_vp, c_vp, c_vp]
        L.lec_recon_workspace_bytes.argtypes = [c_i]
        L.lec_recon_workspace_bytes.restype = c_i64
        L.lec_recon_counter_bytes.argtypes = [c_i64]
        L.lec_recon_counter_bytes.restype = c_i64
        L.lec_recon_pass.argtypes = [ctypes.POINTER(LecRecon), c_vp]
        L.lec_recon_pass_dag.argtypes = [ctypes.POINTER(LecRecon), ctypes.POINTER(LecReconExtra), c_vp]
        L.lec_recon_finish.argtypes = [ctypes.POINTER(LecRecon), c_vp, c_vp, c_vp]
        L.lec_rank_workspace_bytes.argtypes = [c_i64, c_i64]
        L.lec_rank_workspace_bytes.restype = c_i64
        L.lec_rank_run.argtypes = [ctypes.POINTER(LecRank), c_vp, c_vp, c_vp, c_vp]
        L.lec_rank_run_heldout.argtypes = [ctypes.POINTER(LecRank), ctypes.POINTER(LecHeldout), c_vp, c_vp, c_vp, c_vp]
        L.lec_recon_pass_heldout.argtypes = [ctypes.POINTER(LecRecon), ctypes.POINTER(LecReconExtra),
                                             ctypes.POINTER(LecHeldout), c_vp]
        L.lec_recon_finish_at.argtypes = [ctypes.POINTER(LecRecon), c_f, c_vp, c_vp, c_vp]
        L.lec_caption_hinge.argtypes = [c_vp, c_vp, c_i64, c_i, c_f, c_vp, c_vp, c_vp, c_vp, c_vp]
        L.lec_host_pipe_create.argtypes = [ctypes.POINTER(c_vp), c_i]
        L.lec_host_pipe_destroy.argtypes = [c_vp]
        L.lec_host_pipe_destroy.restype = None
        L.lec_host_pipe_submit.argtypes = [c_vp, c_i, ctypes.POINTER(LecStep), ctypes.POINTER(LecHostSample), c_vp, c_i64, c_vp,
                                           c_vp, c_vp, c_vp]
        L.lec_host_pipe_wait.argtypes = [c_vp, c_i]
        for name in EXPORTS:
            getattr(L, name)
        if L.lec_abi_version() != ABI_VERSION:
            raise LecError("liblec_b200.so has ABI version %d, host expects %d: rebuild" % (L.lec_abi_version(), ABI_VERSION))
        _lib = L
    return _lib


def check(code, what):
    if code != 0:
        raise LecError("%s failed: %s (code %d)" % (what, lib().lec_error_string(code).decode(), code))


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise LecError("learning_embeddings_b200 runs on CUDA tensors only (got %s); there is no CPU path" % t.device)


def launch_count():
    return int(lib().lec_launch_count())


def index_errors(device=None, reset=True):
    """Pairs whose endpoint id fell outside the table since the last reset (lec_index_errors; synchronises the stream)."""
    n = ctypes.c_int64(0)
    check(lib().lec_index_errors(ctypes.byref(n), 1 if reset else 0, stream_ptr(device)), "lec_index_errors")
    return int(n.value)


def raise_on_index_errors(device=None):
    bad = index_errors(device)
    if bad:
        raise IndexError("%d pair endpoint ids were outside the embedding table (nn.Embedding raises IndexError in the "
                         "reference); those pairs got energy NaN and no gradient" % bad)
