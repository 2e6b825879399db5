"""ocean_b200 -- host-side mirror (Python stand-in for the Julia shim, see INTEGRATION.md) of the
Oceananigans NonhydrostaticModel operator interface on the new `B200()` architecture.  All
arithmetic runs in libocean_b200.so (hand-written sm_100a CUDA); importing this package fails
if that library has not been built, and nothing here falls back to the CPU."""
from ._lib import lib, B200Error, LIB_PATH, SYMBOLS, last_error  # noqa: F401
from .grids import B200, RectilinearGrid, Periodic, Bounded, Flat, FullyConnected, Center, Face  # noqa: F401
from .distributed import MultiArch  # noqa: F401
from .model import (Field, CenterField, XFaceField, YFaceField, ZFaceField, fill_halo_regions,  # noqa: F401
                    FFTBasedPoissonSolver, FourierTridiagonalPoissonSolver, BatchedTridiagonalSolver,
                    solve, solve_for_pressure, NonhydrostaticModel, WENO5, CenteredSecondOrder,
                    CenteredFourthOrder, UpwindBiasedFirstOrder, UpwindBiasedThirdOrder,
                    UpwindBiasedFifthOrder, ScalarDiffusivity, SmagorinskyLilly, AnisotropicMinimumDissipation,
                    VerticalScalarDiffusivity,
                    HorizontalScalarDiffusivity, FPlane, BuoyancyTracer, Buoyancy, SeawaterBuoyancy,
                    LinearEquationOfState, BoundaryCondition, Relaxation, GaussianMask, LinearTarget,
                    FluxBoundaryCondition, ValueBoundaryCondition, GradientBoundaryCondition,
                    boundary_values, set_boundary_condition_values, BackgroundField, background_table, set_background,
                    update_state, calculate_tendencies, set_model, time_step, sync)
from .output_writers import FieldSlicer, fetch_output, horizontal_average, Checkpointer  # noqa: F401
from .simulations import (Simulation, run, TimeStepWizard, cell_advection_timescale,  # noqa: F401
                          cell_diffusion_timescale, max_abs_velocities)


def launch_count():
    """kernels launched by libocean_b200 so far in this process"""
    return int(lib.ob200_launch_count())
