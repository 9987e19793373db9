"""optimobo_b200 -- B200-native acquisition hot path of aje220/OptiMOBO.

Batched GP posterior (Matern-5/2 / RBF ARD) + multi-objective acquisition + arg-max over very
large candidate pools as hand-written sm_100a CUDA behind a C ABI (include/optimobo_b200.h),
dropped in under the reference's Python surface.  See DESIGN.md / INTEGRATION.md.
"""
from . import _cabi, device_prep, host_prep, scalarisations  # noqa: F401
from .gp import GPModel, refresh_models  # noqa: F401
from .acquisition import (  # noqa: F401
    AcquisitionSpec, CandidatePool, EHVI, EHVI_3D, EHVI_box, EHVI_box_feasible, acquire_from_posterior, consraint_ei,
    evaluate, expected_decomposition,
    expected_improvement, hypervolume_based_PoI, hypervolume_based_PoI_box, pareto_expected_improvement, polish, posterior, propose,
    top_candidates, score_topk, propose_batch,
    propose_host, resolve_precision, scalarise_on_device, score, spec_constrained_ei, spec_ehvi, spec_ehvi3d, spec_ehvi_box,
    spec_ehvi_box_feasible, spec_ei, spec_expected_decomposition, spec_hv_poi, spec_hv_poi_box, spec_pareto_ei,
)

from . import fit, algorithms  # noqa: F401,E402

__version__ = "0.1.0"
