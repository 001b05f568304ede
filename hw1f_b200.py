"""Importable alias of the package directory, whose contractual name
(`monte-carlo-simulation-of-hull-white-model-and-sensitivities-computation_b200`) contains hyphens and
therefore cannot appear in an `import` statement."""
import importlib
import os
import sys

PACKAGE_NAME = "monte-carlo-simulation-of-hull-white-model-and-sensitivities-computation_b200"
_root = os.path.dirname(os.path.abspath(__file__))
if _root not in sys.path:
    sys.path.insert(0, _root)
_pkg = importlib.import_module(PACKAGE_NAME)

Engine = _pkg.Engine
Rng = _pkg.Rng
HW1FError = _pkg.HW1FError
default_params = _pkg.default_params
caplet_schedule = _pkg.caplet_schedule
swaption_schedule = _pkg.swaption_schedule
Params = _pkg.Params
LIB_PATH = _pkg.LIB_PATH
_ffi = _pkg._ffi
package = _pkg
