"""bluerov2_dynamics_b200 — B200-native (sm_100a) batched BlueROV2 Fossen-dynamics rollout engine.

Drop-in for the hot path of ViktorNfa/bluerov2_dynamics (state derivative -> RK4/Euler step -> open-loop rollout ->
multi-step endpoint RMSE) behind the reference's own `fossen/` model API:

    from bluerov2_dynamics_b200.fossen.BlueROV2 import BlueROV2          # 8-thruster model (stateful 3rd-order lag)
    from bluerov2_dynamics_b200.fossen.BlueROV2_thrust import BlueROV2   # wrench input, 12-state
    from bluerov2_dynamics_b200.fossen.BlueROV2_wrench import BlueROV2   # wrench input, 13-state quaternion
    from bluerov2_dynamics_b200.fossen.bluerov_torch import bluerov_compute, ssa
    from bluerov2_dynamics_b200.evaluators import simulate_physics, multistep_rmse_endpoint_physics

or `bluerov2_dynamics_b200.install_as_fossen()` to serve `import fossen...` / `import Koopman...` from this package.  Batched entry points
live on `Engine`.  All compute runs in libbrov.so (hand-written CUDA behind the C ABI of include/brov.h); there is no
CPU fallback — importing this package without the built library raises.
"""
import importlib as _importlib

__all__ = ["Engine", "RolloutResult", "InputGenerator", "BrovError", "default_physical", "derive_params", "derive_params_torch", "default_allocation",
           "lag_discretize", "with_minv", "coefficient_directions", "parameter_indices", "GradResult", "LinearizeResult", "ClosedLoopResult", "EkfResult",
           "VjpResult", "ClosedLoopVjpResult",
           "reduced9_rhs",
           "fma_peak", "pinned_empty", "install_as_fossen", "LIB_PATH"]

_FROM_LIB = ("BrovError", "LIB_PATH")


def __getattr__(name):
    """Public names resolve on first use, so that `python -m bluerov2_dynamics_b200.build` can run before the library
    exists.  Any use of the package without a loadable libbrov.so raises ImportError (there is no CPU fallback)."""
    if name in _FROM_LIB:
        return getattr(_importlib.import_module(__name__ + "._lib"), name)
    if name in __all__:
        return getattr(_importlib.import_module(__name__ + ".engine"), name)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")


def install_as_fossen() -> None:
    """Register this package's model mirror as top-level `fossen` so unmodified reference scripts
    (`from fossen.BlueROV2 import BlueROV2`, `from fossen.bluerov_torch import bluerov_compute`) run on the engine."""
    import importlib
    import sys
    pkg = importlib.import_module(__name__ + ".fossen")
    sys.modules["fossen"] = pkg
    for sub in ("BlueROV2", "BlueROV2_thrust", "BlueROV2_wrench", "bluerov_torch", "parameters"):
        sys.modules["fossen." + sub] = importlib.import_module(f"{__name__}.fossen.{sub}")
    # the training scripts also do `from Koopman.koopmanEDMDc import KoopmanEDMDc`
    sys.modules["Koopman"] = importlib.import_module(__name__ + ".Koopman")
    sys.modules["Koopman.koopmanEDMDc"] = importlib.import_module(__name__ + ".Koopman.koopmanEDMDc")
