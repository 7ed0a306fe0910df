"""waveforminversionust_b200 -- B200-native (sm_100a) Helmholtz forward/adjoint solves and
adjoint-state gradient for ring-array ultrasound FWI, behind the reference's own Python surface.
See DESIGN.md and include/ustfwi.h."""
from .api import (  # noqa: F401
    OneHotSources,
    channel_data,
    clear_plans,
    continuation_stages,
    frequency_continuation,
    fwi_gauss_newton_product,
    fwi_joint_gauss_newton_product,
    fwi_joint_loss_function,
    fwi_loss_function,
    gauss_newton_fwi,
    gauss_newton_joint_fwi,
    hanning,
    idtft,
    joint_frequency_continuation,
    nonlinear_conjugate_gradient,
    nonlinear_conjugate_gradient_joint,
    nonlinear_conjugate_gradient_vectorized,
    run_lbfgs_fwi,
    run_lbfgs_joint_fwi,
    solve_helmholtz,
    time_domain_simulation,
)
from .geometry import attenuation_blob_model, db_cm_mhz_to_kappa, kappa_to_db_cm_mhz  # noqa: F401
from .plan import HelmholtzPlan  # noqa: F401
