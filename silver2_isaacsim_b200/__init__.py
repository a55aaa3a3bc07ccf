"""B200-native hydrodynamics force engine (drop-in for SILVER2's per-body force path).

Light imports only: ``params`` / ``workloads`` / ``waves`` / ``currents`` are NumPy-only; the engine classes are
imported lazily because they load the CUDA library (and fail loudly if it is missing).
"""
from . import currents, params, waves, workloads  # noqa: F401

__all__ = ["currents", "params", "waves", "workloads", "HydroEngine", "WarpHydrodynamicsWrapper",
           "NumbaHydrodynamicsWrapper", "H2OError"]


def __getattr__(name):
    if name == "HydroEngine":
        from .engine import HydroEngine
        return HydroEngine
    if name in ("WarpHydrodynamicsWrapper", "NumbaHydrodynamicsWrapper"):
        from . import wrapper
        return getattr(wrapper, name)
    if name == "H2OError":
        from ._lib import H2OError
        return H2OError
    raise AttributeError(name)
