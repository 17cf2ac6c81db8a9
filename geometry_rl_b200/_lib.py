"""ctypes binding of libgrl_b200.so (the C ABI declared in include/grl_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, a
RuntimeError is raised.  Only raw device pointers, sizes and the current CUDA stream cross the ABI.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgrl_b200.so")

GRL_OK = 0
BASIS_GRAD_FLOATS = 64 * 16 + 64 + 64 * 64 + 64
NODE_GRAD_FLOATS = 256 * 64 + 256 + 64 * 256 + 64 + 64 + 64 + 64 + 16 * 16 * 64
EDGE_GRAD_FLOATS = 64 * 64
FUSED_EDGE_GRAD_FLOATS = 64 * 64 + 64 * 16 + 64 * 64 + 64

_fp = C.c_void_p
_i32 = C.c_int32


class GrlEmbedDesc(C.Structure):
    _fields_ = [("n_nodes", _i32), ("n_scalars", _i32), ("n_vectors", _i32), ("dim", _i32),
                ("scalars", _fp), ("vectors", _fp), ("ori", _fp), ("weight", _fp), ("x", _fp),
                ("grad_x", _fp), ("grad_weight_partials", _fp), ("n_partials", _i32), ("node_ids", _fp)]


class GrlBasisDesc(C.Structure):
    _fields_ = [("n_edges", _i32), ("dim", _i32), ("edge_src", _fp), ("edge_dst", _fp), ("pos_src", _fp),
                ("pos_dst", _fp), ("ori", _fp), ("w1t", _fp), ("b1", _fp), ("w2t", _fp), ("b2", _fp), ("basis", _fp),
                ("w2", _fp), ("grad_basis", _fp), ("grad_partials", _fp), ("n_partials", _i32),
                ("basis_bf16", _fp), ("grad_basis_bf16", _fp)]


class GrlConvDesc(C.Structure):
    _fields_ = [("n_src", _i32), ("n_dst", _i32), ("n_edges", _i32),
                ("rowptr_dst", _fp), ("edge_src", _fp), ("edge_dst", _fp), ("rowptr_src", _fp), ("src_eid", _fp),
                ("x_src", _fp), ("x_dst", _fp), ("basis", _fp), ("fiber_kernel", _fp), ("wk_t", _fp), ("wk", _fp),
                ("bias", _fp), ("ln_g", _fp), ("ln_b", _fp), ("w1_t", _fp), ("w1", _fp), ("b1", _fp), ("w2_t", _fp),
                ("w2_c", _fp), ("b2", _fp), ("x1", _fp), ("out", _fp), ("accumulate_out", _i32),
                ("grad_out", _fp), ("grad_x1", _fp), ("grad_x_src", _fp), ("grad_x_src_init", _fp),
                ("grad_basis", _fp), ("accumulate_grad_basis", _i32), ("node_grad_partials", _fp),
                ("n_partials_node", _i32), ("edge_grad_partials", _fp), ("n_partials_edge", _i32), ("w2", _fp),
                ("basis_bf16", _fp), ("grad_basis_bf16", _fp), ("grad_x2", _fp), ("x2", _fp), ("grad_amax", _fp),
                ("basis_row", _fp), ("grad_basis_acc_mask", _fp)]


class GrlFusedEdgeDesc(C.Structure):
    _fields_ = [("n_key", _i32), ("n_edges", _i32), ("dim", _i32), ("n_partials", _i32),
                ("rowptr", _fp), ("e_src", _fp), ("e_dst", _fp), ("pos_src", _fp), ("pos_dst", _fp), ("ori", _fp),
                ("w1", _fp), ("b1", _fp), ("w2", _fp), ("b2", _fp), ("wk", _fp), ("x_src", _fp), ("x1", _fp),
                ("grad_x1", _fp), ("grad_x_src", _fp), ("grad_x_src_init", _fp), ("grad_partials", _fp), ("n_other", _i32)]


class GrlEncoderDesc(C.Structure):
    _fields_ = [("n_graphs", _i32), ("n_tokens", _i32), ("n_partials", _i32), ("x", _fp), ("in_proj_weight", _fp),
                ("in_proj_bias", _fp), ("out_proj_weight", _fp), ("out_proj_bias", _fp), ("linear1_weight", _fp),
                ("linear1_bias", _fp), ("linear2_weight", _fp), ("linear2_bias", _fp), ("norm1_weight", _fp),
                ("norm1_bias", _fp), ("norm2_weight", _fp), ("norm2_bias", _fp), ("out", _fp), ("grad_out", _fp),
                ("grad_x", _fp), ("grad_partials", _fp)]


ENCODER_MAX_TOKENS = 56
ENCODER_GRAD_FLOATS = 192 * 64 + 192 + 3 * (64 * 64 + 64) + 4 * 64


class GrlCriticDesc(C.Structure):
    _fields_ = [("n_graphs", _i32), ("n_tokens", _i32), ("n_feat", _i32), ("n_partials", _i32), ("eps", C.c_float),
                ("count", C.c_double), ("x", _fp), ("w1", _fp), ("b1", _fp), ("gamma", _fp), ("beta", _fp), ("stats", _fp),
                ("stat_partials", _fp), ("ysum", _fp), ("grad_ysum", _fp), ("bstats", _fp), ("grad_partials", _fp),
                ("n_groups", _i32)]


CRITIC_GRAD_FLOATS = 3 * 64 + 64 * 16


class GrlProjDesc(C.Structure):
    _fields_ = [("batch", _i32), ("k", _i32), ("proj_type", _i32), ("eps_mean", C.c_float), ("eps_cov", C.c_float),
                ("mean", _fp), ("v", _fp), ("old_mean", _fp), ("old_v", _fp), ("proj_mean", _fp), ("proj_v", _fp),
                ("eta", _fp), ("grad_proj_mean", _fp), ("grad_proj_v", _fp), ("grad_mean", _fp), ("grad_v", _fp),
                ("grad_mean_add", _fp), ("grad_v_add", _fp), ("entropy_mode", _i32), ("entropy_first", _i32),
                ("entropy_beta", _fp), ("entropy_alpha", _fp)]


ENTROPY_MODE = {"ineq": 1, "eq": 2}  # GRL_ENTROPY_INEQ / _EQ (0 = off)
ENTROPY_SCHEDULE = {"linear": 1, "exp": 2}  # GRL_ENTROPY_LINEAR / _EXP


class GrlEntropyBoundDesc(C.Structure):
    _fields_ = [("batch", _i32), ("k", _i32), ("schedule", _i32), ("stage", _i32), ("total_train_steps", C.c_int64),
                ("target_entropy", C.c_double), ("temperature", C.c_double), ("old_v", _fp), ("step", _fp), ("sums", _fp),
                ("state", _fp)]


class GrlLossDesc(C.Structure):
    _fields_ = [("batch", _i32), ("k", _i32), ("proj_type", _i32), ("normalize_advantage", _i32),
                ("entropy_coef", C.c_float), ("trust_region_coeff", C.c_float),
                ("mean", _fp), ("v", _fp), ("proj_mean", _fp), ("proj_v", _fp), ("action", _fp), ("prev_log_prob", _fp),
                ("advantage", _fp), ("terms", _fp), ("stats", _fp), ("scalars", _fp), ("grad_losses", _fp),
                ("grad_proj_mean", _fp), ("grad_proj_v", _fp), ("grad_mean_direct", _fp), ("grad_v_direct", _fp),
                ("sums", _fp), ("stage", _i32)]


class GrlReadoutDesc(C.Structure):
    _fields_ = [("n_nodes", _i32), ("od", _i32), ("odv", _i32), ("dim", _i32), ("latent", _fp), ("weight", _fp),
                ("bias", _fp), ("ori", _fp), ("out", _fp), ("hidden", _fp), ("grad_out", _fp), ("grad_hidden", _fp),
                ("grad_latent", _fp), ("grad_partials", _fp), ("n_partials", _i32)]


class GrlHomoPart(C.Structure):
    _fields_ = [("coo", _fp), ("edge_ptr", _fp), ("coo_row_stride", C.c_int64), ("n_src", _i32), ("n_dst", _i32),
                ("off_src", _i32), ("off_dst", _i32)]


HOMO_MAX_PARTS = 8  # GRL_MAX_HOMO_PARTS


class GrlActDesc(C.Structure):
    _fields_ = [("batch", _i32), ("num_rows", _i32), ("action_dim", _i32), ("hidden_dim", _i32), ("post_fc", _i32),
                ("contextual_std", _i32), ("use_tanh_mean", _i32), ("deterministic", _i32), ("rank", _i32),
                ("pre_shift", C.c_float), ("minimal_std", C.c_float), ("hidden", _fp), ("mean", _fp),
                ("mean_weight", _fp), ("mean_bias", _fp), ("std_weight", _fp), ("std_bias", _fp), ("state", _fp),
                ("loc", _fp), ("cov", _fp), ("action", _fp), ("log_prob", _fp), ("eps", _fp)]


ACT_MAX_K = 32  # GRL_ACT_MAX_K


class GrlVecNormKey(C.Structure):
    _fields_ = [("batch", C.c_int64), ("feat", _i32), ("comps", _i32), ("x", _fp), ("out", _fp), ("sum", _fp),
                ("ssq", _fp), ("count", _fp)]


VECNORM_MAX_KEYS = 8  # GRL_VECNORM_MAX_KEYS
VECNORM_MAX_COMPS = 64  # GRL_VECNORM_MAX_COMPS
VECNORM_ROWS_PER_SLOT = 512  # GRL_VECNORM_ROWS_PER_SLOT
VECNORM_MAX_SLOTS = 1024  # GRL_VECNORM_MAX_SLOTS


class GrlVecNormDesc(C.Structure):
    _fields_ = [("n_keys", _i32), ("world", _i32), ("decay", C.c_float), ("eps", C.c_float),
                ("key", GrlVecNormKey * VECNORM_MAX_KEYS), ("partials", _fp), ("inc", _fp)]
READOUT_MAX_OUT = 8
MAX_KNN = 8  # GRL_MAX_KNN: k of grl_knn_graph, max_neighbors of the radius graph
LOSS_TERMS = 8
LOSS_SCALARS = 16
LOSS_STATS = 8
LOSS_SUMS = 16
# index of every scalar grl_trpl_loss_fwd writes (GRL_LS_* in include/grl_b200.h)
LOSS_SCALAR_INDEX = {"loss_objective": 0, "loss_trust_region": 1, "loss_entropy": 2, "dist_entropy": 3, "ESS": 4, "kl": 5,
                     "constraint": 6, "mean_constraint": 7, "mean_constraint_max": 8, "cov_constraint": 9,
                     "cov_constraint_max": 10, "entropy": 11, "entropy_diff": 12}


# name -> (restype, argtypes); every symbol include/grl_b200.h declares
SIGNATURES = {
    "grl_abi_version": (C.c_int, []),
    "grl_last_error": (C.c_char_p, []),
    "grl_sm_count": (C.c_int, []),
    "grl_reserve_sms": (C.c_int, [C.c_int]),
    "grl_knn_edge_ptr": (C.c_int, [_fp, C.c_int, C.c_int, C.c_int, _fp, _fp]),
    "grl_knn_graph": (C.c_int, [_fp, _fp, _fp, C.c_int, C.c_int, C.c_int, _fp, C.c_int64, _fp]),
    "grl_knn_topology": (C.c_int, [_fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int64, _fp, C.c_int64, _fp, _fp, _fp,
                                   _fp, _fp, _fp, _fp, _fp, _fp]),
    "grl_radius_neighbors": (C.c_int, [_fp, _fp, C.c_int, C.c_int, C.c_float, C.c_int, _fp, _fp, _fp]),
    "grl_radius_edge_ptr": (C.c_int, [_fp, C.c_int, C.c_int, C.c_int64, _fp, _fp]),
    "grl_radius_graph": (C.c_int, [_fp, _fp, _fp, C.c_int, C.c_int, C.c_int, _fp, C.c_int64, C.c_int64, _fp]),
    "grl_dense_edges": (C.c_int, [C.c_int, _fp, _fp, C.c_int, C.c_int, C.c_int, _fp, C.c_int64, _fp]),
    "grl_csr_build": (C.c_int, [_fp, C.c_int64, _fp, C.c_int, C.c_int, C.c_int, _fp, _fp, _fp, _fp]),
    "grl_homo_merge": (C.c_int, [C.POINTER(GrlHomoPart), C.c_int, C.c_int, C.c_int, C.c_int64, _fp, _fp, C.c_int64, _fp]),
    "grl_sub_edge_set": (C.c_int, [_fp, _fp, _fp, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, _fp, _fp, _fp,
                                   _fp, _fp, _fp, _fp, _fp, C.c_int64, _fp]),
    "grl_embed_fwd": (C.c_int, [C.POINTER(GrlEmbedDesc), _fp]),
    "grl_embed_bwd": (C.c_int, [C.POINTER(GrlEmbedDesc), _fp]),
    "grl_edge_basis_fwd": (C.c_int, [C.POINTER(GrlBasisDesc), _fp]),
    "grl_edge_basis_bwd": (C.c_int, [C.POINTER(GrlBasisDesc), _fp]),
    "grl_fbconv_edge_fwd": (C.c_int, [C.POINTER(GrlConvDesc), _fp]),
    "grl_fbconv_node_fwd": (C.c_int, [C.POINTER(GrlConvDesc), _fp]),
    "grl_fbconv_node_bwd": (C.c_int, [C.POINTER(GrlConvDesc), _fp]),
    "grl_fbconv_edge_bwd": (C.c_int, [C.POINTER(GrlConvDesc), _fp]),
    "grl_fbconv_node_fwd_tc": (C.c_int, [C.POINTER(GrlConvDesc), _fp]),
    "grl_edge_basis_fwd_tc": (C.c_int, [C.POINTER(GrlBasisDesc), _fp]),
    "grl_fbconv_edge_fwd_tc": (C.c_int, [C.POINTER(GrlConvDesc), _fp]),
    "grl_fbconv_edge_bwd_tc": (C.c_int, [C.POINTER(GrlConvDesc), _fp]),
    "grl_edge_basis_bwd_tc": (C.c_int, [C.POINTER(GrlBasisDesc), _fp]),
    "grl_fbconv_node_bwd_tc": (C.c_int, [C.POINTER(GrlConvDesc), _fp]),
    "grl_fbconv_edge_fused_fwd": (C.c_int, [C.POINTER(GrlFusedEdgeDesc), _fp]),
    "grl_fbconv_edge_fused_bwd": (C.c_int, [C.POINTER(GrlFusedEdgeDesc), _fp]),
    "grl_critic_inner_stats": (C.c_int, [C.POINTER(GrlCriticDesc), _fp]),
    "grl_critic_inner_fwd": (C.c_int, [C.POINTER(GrlCriticDesc), _fp]),
    "grl_critic_inner_bwd_stats": (C.c_int, [C.POINTER(GrlCriticDesc), _fp]),
    "grl_critic_inner_bwd": (C.c_int, [C.POINTER(GrlCriticDesc), _fp]),
    "grl_encoder_layer_fwd": (C.c_int, [C.POINTER(GrlEncoderDesc), _fp]),
    "grl_encoder_layer_bwd": (C.c_int, [C.POINTER(GrlEncoderDesc), _fp]),
    "grl_readout_fwd": (C.c_int, [C.POINTER(GrlReadoutDesc), _fp]),
    "grl_readout_bwd": (C.c_int, [C.POINTER(GrlReadoutDesc), _fp]),
    "grl_trpl_loss_fwd": (C.c_int, [C.POINTER(GrlLossDesc), _fp]),
    "grl_trpl_loss_bwd": (C.c_int, [C.POINTER(GrlLossDesc), _fp]),
    "grl_dp_combine": (C.c_int, [_fp, C.c_int, C.c_int, C.c_int, _fp, _fp]),
    "grl_absmax": (C.c_int, [_fp, C.c_int64, _fp, _fp]),
    "grl_reduce_partials": (C.c_int, [_fp, C.c_int, C.c_int64, _fp, C.c_int, _fp]),
    "grl_gae_scan": (C.c_int, [_fp, _fp, _fp, _fp, C.c_float, C.c_float, C.c_int, C.c_int, _fp, _fp, _fp]),
    "grl_gaussian_act": (C.c_int, [C.POINTER(GrlActDesc), _fp]),
    "grl_act_advance": (C.c_int, [_fp, _fp]),
    "grl_vecnorm_stats": (C.c_int, [C.POINTER(GrlVecNormDesc), _fp]),
    "grl_vecnorm_update": (C.c_int, [C.POINTER(GrlVecNormDesc), _fp]),
    "grl_vecnorm_apply": (C.c_int, [C.POINTER(GrlVecNormDesc), _fp]),
    "grl_trpl_fwd": (C.c_int, [C.POINTER(GrlProjDesc), _fp]),
    "grl_trpl_bwd": (C.c_int, [C.POINTER(GrlProjDesc), _fp]),
    "grl_trpl_entropy_bound": (C.c_int, [C.POINTER(GrlEntropyBoundDesc), _fp]),
    "grl_tc_selftest_gemm": (C.c_int, [_fp, _fp, _fp, C.c_int, C.c_int, _fp]),
    "grl_tc_selftest_gemm_ts": (C.c_int, [_fp, _fp, _fp, C.c_int, _fp]),
    "grl_tc_debug_mma": (C.c_int, [_fp, C.c_int, _fp, C.c_int, _fp, C.c_int, C.c_int] + [C.c_uint32] * 8 + [_fp]),
    "grl_tc_latency_probe": (C.c_int, [_fp, _fp]),
}

_lib = None
launch_count = 0  # number of kernel-launching ABI calls made by this process (bench.py reports it)


def load():
    """Load the shared library (once).  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(geometry_rl_b200 has no CPU or eager fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    return load().grl_last_error().decode()


def check(rc: int, what: str):
    if rc != GRL_OK:
        raise RuntimeError(f"{what} failed with code {rc}: {last_error()}")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("geometry_rl_b200 kernels need CUDA tensors (no CPU path exists)")
    if not t.is_contiguous():
        raise RuntimeError("geometry_rl_b200 kernels need contiguous tensors")
    return t.data_ptr()


def ptr_any(t):
    """Device pointer without the contiguity check (strided COO rows, fp64 workspaces)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("geometry_rl_b200 kernels need CUDA tensors (no CPU path exists)")
    return t.data_ptr()


_timing = None  # None | dict name -> list of (start_event, end_event, shape)


def event_timing(enable: bool):
    """bench.py's per-kernel pass: bracket every ABI launch with CUDA events on the launching stream.
    event_timing(True) starts recording; event_timing(False) returns {name: [(ms, *shape), ...]}."""
    global _timing
    if enable:
        _timing = {}
        return None
    rec, _timing = _timing, None
    torch.cuda.synchronize()
    return {k: [(a.elapsed_time(b),) + tuple(shape) for a, b, shape in v] for k, v in (rec or {}).items()}


def call(name: str, *args, shape=(0, 0, 0)):
    """Invoke an ABI function on the current torch stream and raise on a non-zero return code.
    `shape` = (n_src, n_dst, n_edges) of the launch, only used to label bench.py's per-kernel timings."""
    global launch_count
    lib = load()
    if _timing is not None:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = getattr(lib, name)(*args, stream_ptr())
        b.record()
        _timing.setdefault(name, []).append((a, b, shape))
    else:
        rc = getattr(lib, name)(*args, stream_ptr())
    launch_count += 1
    check(rc, name)


_sm = None


def sm_count() -> int:
    global _sm
    if _sm is None:
        _sm = load().grl_sm_count()
    return _sm


def reserve_sms(n: int) -> None:
    """Leave `n` SMs out of every persistent kernel's grid (see grl_reserve_sms in include/grl_b200.h)."""
    global _sm
    check(load().grl_reserve_sms(int(n)), "grl_reserve_sms")
    _sm = None
