"""tuna_b200 — B200-native (sm_100a) provider for the SCF two-electron hot path of h-brough/TUNA:
ERI evaluation (tuna_integrals) + Coulomb/exchange contraction (tuna_scf), behind the reference's own
Python call signatures.  See DESIGN.md and INTEGRATION.md."""
from . import workloads  # noqa: F401
from ._lib import Context, DeviceGroup, TunaError  # noqa: F401
from .basis import Basis  # noqa: F401
from .provider import (  # noqa: F401
    ERIHandle, calculate_coulomb_matrix, calculate_cross_basis_overlap_matrix, calculate_one_electron_integrals, calculate_electron_repulsion_integral, calculate_electron_repulsion_integrals,
    calculate_exchange_matrix, calculate_two_electron_integrals, configure, coulomb_and_exchange, install,
    transform_ERI_AO_to_MO, transform_ERI_AO_to_SO, transform_to_spherical_harmonics, uninstall)

__version__ = "0.1.0"
