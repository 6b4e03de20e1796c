"""polee_b200 -- host-side mirror of the Polee API for the prep-sample likelihood-approximation path.

The product is the C-ABI library ``libpolee_b200.so`` (hand-written sm_100a CUDA kernels, see
``include/polee_b200.h``).  Polee's own host code is Julia and binds that library with ``ccall``
(``julia/PoleeB200.jl``); this package is the same binding written in Python -- the toolchain this
repository can execute -- with the reference's names and argument meaning
(``approximate_likelihood``, ``PolyaTreeTransform``, ``RNASeqSample`` ...), so the parity tests read
like tests of the reference.  There is no CPU fallback: every compute call goes through the library.
"""
from ._lib import LIB_PATH, PoleeError, build_library, load_library  # noqa: F401
from .api import (  # noqa: F401
    LIKAP_NUM_MC_SAMPLES,
    LIKAP_NUM_STEPS,
    ApproxLikelihoodSampler,
    Handle,
    HsbPlan,
    LogitSkewNormalPTTApprox,
    OptimizePTTApprox,
    PolyaTreeTransform,
    RNASeqSample,
    approx_log_prob,
    approx_log_prob_torch,
    approximate_likelihood,
    exact_factorization,
    hclust,
    hsb,
    hsb_grad,
    hsb_torch,
    inv_hsb,
    inv_hsb_grad,
    inv_hsb_torch,
    log_likelihood,
    make_inverse_ptt_params,
    optimize_likelihood,
    partition_rows,
    prep_many,
    trim_memory,
)
