"""Import the reference's UNMODIFIED kernels from an xgcm source checkout.

xarray and dask need not be installed: ``xgcm.gridops`` and ``xgcm.transform``
only need those packages for def-time type annotations.  We register empty
stand-in modules exposing the referenced type names and import the two kernel
modules as they lie on disk.  Nothing is copied.  Used by ``oracle/make_golden.py``
to record the golden vectors under ``tests/golden/``.

TEST INFRASTRUCTURE ONLY.
"""

from __future__ import annotations

import importlib
import sys
import types
from pathlib import Path


def _stub(name: str, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    mod.__xgcm_b200_stub__ = True
    return mod


def load(root):
    """Return ``(gridops, transform)`` modules of the reference checkout at ``root``."""
    root = Path(root)
    if not (root / "xgcm" / "gridops.py").is_file():
        raise RuntimeError(f"{root} is not an xgcm source checkout (no xgcm/gridops.py)")
    added = []
    if "xarray" not in sys.modules:
        sys.modules["xarray"] = _stub(
            "xarray", DataArray=type("DataArray", (), {}), Dataset=type("Dataset", (), {})
        )
        added.append("xarray")
    if "dask" not in sys.modules:
        dask = _stub("dask")
        dask_array = _stub("dask.array", Array=type("Array", (), {}))
        dask.array = dask_array
        sys.modules["dask"] = dask
        sys.modules["dask.array"] = dask_array
        added += ["dask", "dask.array"]
    # import xgcm's submodules without running xgcm/__init__.py (which needs xarray for real)
    pkg = types.ModuleType("xgcm")
    pkg.__path__ = [str(root / "xgcm")]
    prev = sys.modules.get("xgcm")
    sys.modules["xgcm"] = pkg
    try:
        gridops = importlib.import_module("xgcm.gridops")
        transform = importlib.import_module("xgcm.transform")
    finally:
        for name in list(sys.modules):
            if name == "xgcm" or name.startswith("xgcm."):
                del sys.modules[name]
        if prev is not None:
            sys.modules["xgcm"] = prev
        for name in added:
            sys.modules.pop(name, None)
    return gridops, transform
