"""ctypes loader for libpolee_b200.so (the C ABI in include/polee_b200.h)."""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# POLEE_B200_LIB: an experimental build (csrc/Makefile VARIANT=...) instead of the real library
LIB_PATH = os.environ.get("POLEE_B200_LIB") or os.path.join(_HERE, "libpolee_b200.so")

POLEE_OK, POLEE_EINVAL, POLEE_ECUDA, POLEE_EBADTREE, POLEE_ENONFINITE, POLEE_ENCCL, POLEE_ENOMEM = range(7)
APPROX_LSN_PTT, APPROX_OPTIMIZE_PTT = 0, 1
NOISE_PHILOX, NOISE_INJECTED = 0, 1


class PoleeError(RuntimeError):
    """Non-zero status from libpolee_b200 (the Julia glue raises error(msg) at the same points)."""

    def __init__(self, code, msg):
        super().__init__("libpolee_b200 error %d: %s" % (code, msg))
        self.code = code


class PoleeOpts(C.Structure):
    _fields_ = [("device", C.c_int32), ("approx", C.c_int32), ("num_steps", C.c_int32),
                ("num_mc_samples", C.c_int32), ("gradonly", C.c_int32), ("use_efflen_jacobian", C.c_int32),
                ("noise_mode", C.c_int32), ("exact_accumulation", C.c_int32), ("seed", C.c_uint64),
                ("max_step_mu", C.c_double), ("max_step_omega", C.c_double), ("max_step_alpha", C.c_double),
                ("max_step_z", C.c_double), ("use_cuda_graph", C.c_int32), ("reserved1", C.c_int32)]


# every symbol include/polee_b200.h declares (tests check that the built library exports them all)
EXPORTS = [
    "polee_opts_default", "polee_create", "polee_destroy", "polee_trim_memory", "polee_last_error", "polee_device_info",
    "polee_set_matrix_csc", "polee_set_matrix_csc_device", "polee_set_efflens", "polee_set_gene_groups",
    "polee_set_tree",
    "polee_set_tree_sequential", "polee_set_sample", "polee_fit", "polee_fit_optimize_ptt", "polee_init_params", "polee_run_steps",
    "polee_sync", "polee_set_progress", "polee_get_params", "polee_set_params", "polee_set_noise", "polee_get_elbo", "polee_stream",
    "polee_step_stats", "polee_layout_info", "polee_time_kernel", "polee_sample", "polee_loglik_grad", "polee_frag_prob_recip", "polee_ptt_transform",
    "polee_ptt_transform_gradients", "polee_ptt_inverse_transform", "polee_lsn_draws", "polee_hsb", "polee_inv_hsb",
    "polee_inv_hsb_grad", "polee_hsb_device", "polee_inv_hsb_device", "polee_inv_hsb_grad_device", "polee_hsb_plan_create", "polee_hsb_plan_destroy", "polee_hsb_with_plan",
    "polee_inv_hsb_with_plan", "polee_inv_hsb_grad_with_plan", "polee_approx_log_prob_with_plan",
    "polee_approx_log_prob_device", "polee_hsb_grad", "polee_hsb_grad_with_plan", "polee_hsb_grad_device",
    "polee_hsb_last_error",
    "polee_make_inverse_ptt_params", "polee_exact_factorization", "polee_hclust", "polee_partition_rows", "polee_comm_unique_id", "polee_comm_init", "polee_comm_peer_export", "polee_comm_peer_import",
]


def build_library(force=False, verbose=False):
    """Compile the CUDA sources in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    src = os.path.join(_HERE, "csrc")
    if force and os.path.exists(LIB_PATH):
        os.remove(LIB_PATH)
    cmd = ["make", "-C", src, "-j8"]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout)
    if out.returncode != 0:
        raise RuntimeError("building libpolee_b200.so failed")
    return LIB_PATH


_lib = None


def load_library():
    """dlopen the library; never falls back to anything else."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(or `make -C polee_b200/csrc`). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.polee_last_error.restype = C.c_char_p
    lib.polee_last_error.argtypes = [C.c_void_p]
    lib.polee_hsb_last_error.restype = C.c_char_p
    lib.polee_stream.restype = C.c_void_p
    lib.polee_stream.argtypes = [C.c_void_p]
    _lib = lib
    return lib
