"""prmf_b200 -- B200-native PRMF alternating factorisation (hot path of gitter-lab/prmf).

    from prmf_b200 import nmf_pathway          # drop-in for script/prmf_runner.py:nmf_pathway

Arithmetic runs in hand-written sm_100a CUDA kernels behind a C ABI (include/prmf_b200.h,
prmf_b200/libprmf_b200.so); there is no CPU execution path.
"""
from .solver import (find_mins, latent_pathway_tables, nmf_manifold_vec_obj, nmf_manifold_vec_update,  # noqa: F401
                     nmf_pathway, restrict)
from .pathways import PackedPathways, pack_pathways  # noqa: F401
from .engine import CudaEngine  # noqa: F401
from .preprocess import quantile_transform  # noqa: F401
from .cv import measure_cv_performance, nnls_rows  # noqa: F401
from .manifold_init import nnls_x, pathway_init  # noqa: F401

__version__ = "0.1.0"
