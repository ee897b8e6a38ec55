"""ctypes binding of libomc.so (include/omc.h) — the only way the Python host code reaches the CUDA kernels.

There is no CPU fallback: if the shared library is missing `load()` raises, and every numeric entry point of the
package goes through it.
"""

import ctypes as C
import os

_LIB_NAME = "libomc.so"
_lib = None


class OmcError(RuntimeError):
    """Raised when a libomc call returns non-zero; carries omc_last_error()."""


class Vec(C.Structure):
    """omc_vec_t: per-chain operand (device pointer + element stride between chains, 0 = shared)."""

    _fields_ = [("ptr", C.c_void_p), ("chain_stride", C.c_longlong)]


class Rng(C.Structure):
    """omc_rng_t"""

    _fields_ = [
        ("seed", C.c_ulonglong),
        ("sweep", C.c_void_p),
        ("chain_offset", C.c_uint),
        ("site", C.c_uint),
    ]


class NNDense(C.Structure):
    """omc_nn_dense_t"""

    _fields_ = [
        ("n_chains", C.c_int),
        ("p", C.c_int),
        ("stats", Vec),
        ("tau", Vec),
        ("prior_kind", C.c_int),
        ("prior_P", Vec),
        ("lam", Vec),
        ("mu0", Vec),
        ("beta", C.c_void_p),
        ("rng", Rng),
        ("debug_z", C.c_void_p),
        ("debug_sweep_stride", C.c_longlong),
        ("probe_Q", C.c_void_p),
        ("probe_b", C.c_void_p),
        ("probe_L", C.c_void_p),
        ("probe_mu", C.c_void_p),
        ("status", C.c_void_p),
        ("truncated", C.c_int),
        ("trunc_lo", Vec),
        ("trunc_hi", Vec),
        ("trunc_lo_len", C.c_int),
        ("trunc_hi_len", C.c_int),
        ("debug_u", C.c_void_p),
        ("center", Vec),
        ("rss_out", C.c_void_p),
        ("mode", C.c_int),
        ("ridge_rel", C.c_double),
        ("workspace", C.c_void_p),
    ]


class DenseFactor(C.Structure):
    """omc_dense_factor_t"""

    _fields_ = [("n_mats", C.c_int), ("n", C.c_int), ("Q", C.c_void_p), ("Q_stride", C.c_longlong), ("b", C.c_void_p),
                ("z", C.c_void_p), ("L", C.c_void_p), ("logdet", C.c_void_p), ("mean", C.c_void_p), ("x", C.c_void_p),
                ("status", C.c_void_p), ("factored", C.c_int), ("backward_only", C.c_int), ("workspace", C.c_void_p)]


class Quadform(C.Structure):
    """omc_quadform_t"""

    _fields_ = [
        ("n_chains", C.c_int),
        ("p", C.c_int),
        ("x", Vec),
        ("mu", Vec),
        ("kind", C.c_int),
        ("P", Vec),
        ("ss", C.c_void_p),
        ("cnt", C.c_void_p),
    ]


class NGDraw(C.Structure):
    """omc_ng_draw_t"""

    _fields_ = [
        ("n_chains", C.c_int),
        ("a0", Vec),
        ("b0", Vec),
        ("ss", Vec),
        ("cnt", Vec),
        ("out", C.c_void_p),
        ("rng", Rng),
        ("debug_g", C.c_void_p),
        ("debug_sweep_stride", C.c_longlong),
        ("probe_a", C.c_void_p),
        ("probe_b", C.c_void_p),
        ("n_elem", C.c_int),
        ("a0_len", C.c_int),
        ("b0_len", C.c_int),
        ("ss_stride", C.c_longlong),
        ("cnt_stride", C.c_longlong),
    ]


class MixtureAlloc(C.Structure):
    """omc_mixture_alloc_t"""

    _fields_ = [("n_chains", C.c_int), ("n", C.c_int), ("K", C.c_int), ("x", Vec), ("mu", Vec), ("tau", Vec),
                ("prob", Vec), ("prob_rows", C.c_int), ("z", C.c_void_p), ("rng", Rng), ("debug_u", C.c_void_p),
                ("debug_sweep_stride", C.c_longlong)]


class MixtureStats(C.Structure):
    """omc_mixture_stats_t"""

    _fields_ = [("n_chains", C.c_int), ("n", C.c_int), ("K", C.c_int), ("x", Vec), ("mu", Vec), ("tau", Vec),
                ("z", C.c_void_p), ("stats", C.c_void_p), ("record", C.c_void_p), ("gather_mu", C.c_void_p),
                ("gather_tau", C.c_void_p), ("logp", C.c_void_p), ("accumulate", C.c_int)]


class LogpNormalSS(C.Structure):
    """omc_logp_normal_ss_t"""

    _fields_ = [("n_chains", C.c_int), ("dim", C.c_double), ("ss", Vec), ("scalar", Vec), ("logdet", Vec),
                ("out", C.c_void_p), ("accumulate", C.c_int)]


class LogpGamma(C.Structure):
    """omc_logp_gamma_t"""

    _fields_ = [("n_chains", C.c_int), ("n_elem", C.c_int), ("shape_len", C.c_int), ("rate_len", C.c_int),
                ("x", Vec), ("shape", Vec), ("rate", Vec), ("out", C.c_void_p), ("accumulate", C.c_int)]


class LogpPoisson(C.Structure):
    """omc_logp_poisson_t"""

    _fields_ = [("n_chains", C.c_int), ("n_elem", C.c_int), ("rate_len", C.c_int), ("k", Vec), ("rate", Vec),
                ("out", C.c_void_p), ("accumulate", C.c_int)]


class LinearPredictor(C.Structure):
    """omc_linear_predictor_t"""

    _fields_ = [("n_chains", C.c_int), ("n", C.c_int), ("n_terms", C.c_int), ("p", C.c_int * 4), ("X", Vec * 4),
                ("theta", Vec * 4), ("out", C.c_void_p), ("transform_exp", C.c_int * 4), ("residual_of", Vec)]


class Term(C.Structure):
    """omc_term_t"""

    _fields_ = [("kind", C.c_int), ("mat_kind", C.c_int), ("p1_len", C.c_int), ("p2_len", C.c_int), ("data", Vec),
                ("p1", Vec), ("p2", Vec), ("P", Vec), ("scalar", Vec), ("logdet", Vec), ("dom_lo", C.c_double),
                ("dom_hi", C.c_double), ("stats", Vec), ("n_data", C.c_int), ("transform_exp", C.c_int)]


class MHModel(C.Structure):
    """omc_mh_model_t"""

    _fields_ = [("n_chains", C.c_int), ("n_elem", C.c_int), ("n_terms", C.c_int), ("terms", Term * 4)]


class RandomWalkArgs(C.Structure):
    """omc_random_walk_t"""

    _fields_ = [("model", MHModel), ("theta", C.c_void_p), ("p_dim", C.c_int), ("n_rep", C.c_int), ("loop", C.c_int),
                ("step", Vec), ("step_rows", C.c_int), ("step_cols", C.c_int), ("limits", C.c_void_p), ("rng", Rng),
                ("debug_z", C.c_void_p), ("debug_u", C.c_void_p), ("debug_sweep_stride_z", C.c_longlong),
                ("debug_sweep_stride_u", C.c_longlong), ("counters", C.c_void_p), ("probe", C.c_void_p)]


class MMalaArgs(C.Structure):
    """omc_mmala_t"""

    _fields_ = [("model", MHModel), ("theta", C.c_void_p), ("step", C.c_double), ("method", C.c_int), ("rng", Rng),
                ("debug_z", C.c_void_p), ("debug_u", C.c_void_p), ("debug_sweep_stride_z", C.c_longlong),
                ("debug_sweep_stride_u", C.c_longlong), ("counters", C.c_void_p), ("status", C.c_void_p),
                ("probe_mu", C.c_void_p), ("probe_L", C.c_void_p), ("probe_prop", C.c_void_p),
                ("probe_scalars", C.c_void_p)]


class TridiagNN(C.Structure):
    """omc_tridiag_nn_t"""

    _fields_ = [("n_chains", C.c_int), ("n", C.c_longlong), ("pd", C.c_void_p), ("pe", C.c_void_p), ("lam", Vec),
                ("tau", Vec), ("w", Vec), ("y", Vec), ("h", Vec), ("mu0", Vec), ("x", C.c_void_p), ("rng", Rng),
                ("debug_z", C.c_void_p), ("debug_sweep_stride", C.c_longlong), ("ss_prior", C.c_void_p),
                ("ss_lik", C.c_void_p), ("logdet", C.c_void_p), ("probe_l", C.c_void_p), ("probe_c", C.c_void_p),
                ("status", C.c_void_p), ("workspace", C.c_void_p)]


class _FKonst(C.Structure):
    _fields_ = [("value", C.c_double), ("out", C.c_void_p), ("accumulate", C.c_int)]


class _FCopy(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("count", C.c_longlong), ("iter_counter", C.c_void_p),
                ("max_iter", C.c_longlong), ("ring", C.c_int)]


class _FUnion(C.Union):
    _fields_ = [("normal_ss", LogpNormalSS), ("gamma", LogpGamma), ("poisson", LogpPoisson), ("konst", _FKonst),
                ("ng", NGDraw), ("quad", Quadform), ("copy", _FCopy)]


class FOp(C.Structure):
    """omc_fop_t"""

    _fields_ = [("kind", C.c_int), ("u", _FUnion)]


FUSED_MAX_OPS = 12
FOP_LOGP_NORMAL_SS, FOP_LOGP_GAMMA, FOP_LOGP_POISSON, FOP_LOGP_CONST, FOP_NG_DRAW, FOP_QUADFORM, FOP_STORE_COPY = range(1, 8)


class FusedSmall(C.Structure):
    """omc_fused_small_t"""

    _fields_ = [("n_chains", C.c_int), ("n_ops", C.c_int), ("ops", FOp * FUSED_MAX_OPS)]


EXTRA_STRUCTS = {"omc_tridiag_nn_t": TridiagNN, "omc_dense_factor_t": DenseFactor, "omc_fop_t": FOp,
                 "omc_fused_small_t": FusedSmall}

# name -> (restype, argtypes); every symbol include/omc.h declares must be listed here (tests check both ways)
PROTOTYPES = {
    "omc_abi_version": (C.c_int, []),
    "omc_last_error": (C.c_char_p, []),
    "omc_device_init": (C.c_int, [C.c_int]),
    "omc_device_sm_count": (C.c_int, []),
    "omc_counter_add": (C.c_int, [C.c_void_p, C.c_ulonglong, C.c_void_p]),
    "omc_counter_add2": (C.c_int, [C.c_void_p, C.c_ulonglong, C.c_void_p, C.c_ulonglong, C.c_void_p]),
    "omc_graph_capture_begin": (C.c_int, [C.c_void_p]),
    "omc_graph_capture_end": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "omc_graph_launch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong]),
    "omc_graph_destroy": (C.c_int, [C.c_void_p]),
    "omc_graph_num_kernel_nodes": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong)]),
    "omc_run_schedule": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong]),
    "omc_store_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p]),
    "omc_store_copy_ring": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p]),
    "omc_reg_pass_workspace": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_longlong)]),
    "omc_reg_pass": (
        C.c_int,
        [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong,
         C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p],
    ),
    "omc_reg_rss": (
        C.c_int,
        [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong,
         C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p],
    ),
    "omc_nn_dense_draw": (C.c_int, [C.POINTER(NNDense), C.c_void_p]),
    "omc_nn_dense_workspace": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_longlong)]),
    "omc_dense_factor": (C.c_int, [C.POINTER(DenseFactor), C.c_void_p]),
    "omc_quadform": (C.c_int, [C.POINTER(Quadform), C.c_void_p]),
    "omc_fused_small": (C.c_int, [C.POINTER(FusedSmall), C.c_void_p]),
    "omc_ng_draw": (C.c_int, [C.POINTER(NGDraw), C.c_void_p]),
    "omc_logp_normal_ss": (C.c_int, [C.POINTER(LogpNormalSS), C.c_void_p]),
    "omc_logp_gamma": (C.c_int, [C.POINTER(LogpGamma), C.c_void_p]),
    "omc_logp_poisson": (C.c_int, [C.POINTER(LogpPoisson), C.c_void_p]),
    "omc_logp_const": (C.c_int, [C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "omc_mixture_allocation": (C.c_int, [C.POINTER(MixtureAlloc), C.c_void_p]),
    "omc_mixture_stats": (C.c_int, [C.POINTER(MixtureStats), C.c_void_p]),
    "omc_logp_categorical": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, Vec, C.c_int, C.c_void_p, C.c_int,
                                       C.c_void_p]),
    "omc_logp_domain": (C.c_int, [C.c_int, C.c_int, Vec, Vec, C.c_int, Vec, C.c_int, C.c_void_p, C.c_void_p]),
    "omc_linear_predictor": (C.c_int, [C.POINTER(LinearPredictor), C.c_void_p]),
    "omc_combine": (C.c_int, [C.c_int, C.c_longlong, C.c_int, C.POINTER(Vec), C.POINTER(Vec), C.c_void_p, C.c_void_p]),
    "omc_rank_normalize": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_longlong, C.c_longlong, C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "omc_sum_log": (C.c_int, [C.c_void_p, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p]),
    "omc_log_elements": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]),
    "omc_logdet_dense": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "omc_tridiag_workspace": (C.c_int, [C.c_int, C.c_longlong, C.POINTER(C.c_longlong)]),
    "omc_tridiag_workspace_init": (C.c_int, [C.c_void_p, C.c_int, C.c_longlong, C.c_void_p]),
    "omc_tridiag_nn_draw": (C.c_int, [C.POINTER(TridiagNN), C.c_void_p]),
    "omc_tridiag_quadforms": (C.c_int, [C.POINTER(TridiagNN), C.c_void_p]),
    "omc_bidiag_gram": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p]),
    "omc_tridiag_matvec": (C.c_int, [C.c_void_p, C.c_void_p, Vec, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p]),
    "omc_mh_logp": (C.c_int, [C.POINTER(MHModel), C.c_void_p, C.c_void_p, C.c_void_p]),
    "omc_mh_logp_acc": (C.c_int, [C.POINTER(MHModel), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "omc_mh_grad_hess": (C.c_int, [C.POINTER(MHModel), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "omc_random_walk": (C.c_int, [C.POINTER(RandomWalkArgs), C.c_void_p]),
    "omc_mmala": (C.c_int, [C.POINTER(MMalaArgs), C.c_void_p]),
    "omc_truncnorm_rv": (C.c_int, [C.c_void_p] * 5 + [C.c_longlong, C.c_void_p, C.c_void_p]),
    "omc_truncnorm_logpdf": (C.c_int, [C.c_void_p] * 5 + [C.c_longlong, C.c_void_p, C.c_void_p]),
}


class ChainStats(C.Structure):
    """omc_chain_stats_t"""

    _fields_ = [("samples", C.c_void_p), ("n_iter", C.c_longlong), ("n_chains", C.c_int), ("size", C.c_longlong),
                ("n_sel", C.c_longlong), ("elem_stride", C.c_longlong), ("max_lag", C.c_int), ("out", C.c_void_p)]


PROTOTYPES.update({
    "omc_chain_stats": (C.c_int, [C.POINTER(ChainStats), C.c_void_p]),
    "omc_rhat_combine": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
})
EXTRA_STRUCTS["omc_chain_stats_t"] = ChainStats


class RJArgs(C.Structure):
    """omc_rj_t"""

    _fields_ = [("n_chains", C.c_int), ("n_data", C.c_int), ("n_max", C.c_int), ("n_basis", C.c_void_p),
                ("theta", C.c_void_p), ("omega", C.c_void_p), ("beta", C.c_void_p), ("B", C.c_void_p), ("X", C.c_void_p),
                ("y", Vec), ("tau_y", Vec), ("theta_lo", C.c_double), ("theta_hi", C.c_double), ("sample_omega", C.c_int),
                ("omega_shape", Vec), ("omega_rate", Vec), ("mu_beta", Vec), ("tau_beta", Vec), ("rho", Vec),
                ("birth_probability", C.c_double), ("match_scale", C.c_double), ("match_truncated", C.c_int),
                ("match_lo", C.c_double), ("match_hi", C.c_double), ("rng", Rng), ("debug", C.c_void_p),
                ("debug_sweep_stride", C.c_longlong), ("counters", C.c_void_p), ("status", C.c_void_p),
                ("probe", C.c_void_p), ("logp_only", C.c_int), ("logp_out", C.c_void_p), ("size_class", C.c_void_p),
                ("gram", C.c_void_p), ("gram_valid", C.c_void_p)]


PROTOTYPES.update({
    "omc_rj_smem_bytes": (C.c_int, [C.c_int, C.c_int]),
    "omc_reversible_jump": (C.c_int, [C.POINTER(RJArgs), C.c_void_p]),
    "omc_rj_basis": (C.c_int, [C.POINTER(RJArgs), C.c_void_p]),
})
EXTRA_STRUCTS["omc_rj_t"] = RJArgs


class RJWalk(C.Structure):
    """omc_rj_walk_t"""

    _fields_ = [("model", RJArgs), ("which", C.c_int), ("step", C.c_double), ("lim_lo", C.c_double),
                ("lim_hi", C.c_double), ("debug_tn_u", C.c_void_p), ("debug_u", C.c_void_p),
                ("debug_sweep_stride", C.c_longlong), ("counters", C.c_void_p)]


class RJMmala(C.Structure):
    """omc_rj_mmala_t"""

    _fields_ = [("model", RJArgs), ("step", C.c_double), ("debug_z", C.c_void_p), ("debug_u", C.c_void_p),
                ("debug_sweep_stride_z", C.c_longlong), ("debug_sweep_stride_u", C.c_longlong), ("counters", C.c_void_p),
                ("probe", C.c_void_p)]


PROTOTYPES.update({
    "omc_rj_knot_walk": (C.c_int, [C.POINTER(RJWalk), C.c_void_p]),
    "omc_rj_coef_mmala": (C.c_int, [C.POINTER(RJMmala), C.c_void_p]),
})
EXTRA_STRUCTS["omc_rj_walk_t"] = RJWalk
EXTRA_STRUCTS["omc_rj_mmala_t"] = RJMmala


def lib_path() -> str:
    """In-tree libomc.so; OMC_LIB overrides it (tools/ab_dense_draw.sh times builds with it)."""
    return os.environ.get("OMC_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), _LIB_NAME)


def load():
    """Load libomc.so and attach prototypes.  Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise OmcError(
            f"{path} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()' "
            "or make -C openmcmc_b200/csrc). openmcmc_b200 has no CPU fallback."
        )
    lib = C.CDLL(path)
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().omc_last_error()
        raise OmcError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")
