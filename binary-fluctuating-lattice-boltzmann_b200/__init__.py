"""bflbm-b200: B200-native fluctuating binary-fluid D3Q19 lattice-Boltzmann step.

Only the hot path of MDProject/Binary-Fluctuating-Lattice-Boltzmann (LBM_binary.H / LBM_d3q19.H) lives
here: csrc/ (CUDA kernels + C ABI, include/bflbm.h) and this thin host mirror of the reference interface.
"""
from ._build import build, build_sf, LIB, SF_LIB  # noqa: F401
from .structure_factor import StructureFactor, SlabStructureFactor, REFERENCE_PAIRS  # noqa: F401
from .lattice import (  # noqa: F401
    BflbmError, Lattice, MultiLattice, Params, VARIABLE_NAMES, NVEL, NHYDRO, NHYDRO_BAR, NNORMALS, load_library, philox4x32_10,
    LBM_init, LBM_init_droplet, LBM_init_mixture, LBM_init_stripe, LBM_timestep, LBM_hydrovars,
    LBM_hydrovars_density, thermal_noise, update_com,
)
