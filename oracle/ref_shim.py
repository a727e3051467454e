"""TEST INFRASTRUCTURE ONLY -- import the *unmodified* reference from its checkout (REF_ROOT below).

Only usable where that checkout exists.  Used by tests/golden/make_golden.py and
tests/golden/make_reference_checks.py to generate the committed golden vectors that
pin oracle/planner_oracle.py.  Nothing here is imported by the product package.

Why a shim is needed (SURVEY.md section 8c):
  * /root/reference/utils/__init__.py and graphs/__init__.py eagerly import every
    sibling module (matplotlib, easydict, tensorboardX ... absent here), so the
    packages are pre-registered as bare namespace modules whose __path__ points
    into the reference tree and whose __init__ therefore never runs.
  * graphs/models/decentralplanner.py:11 imports the unused `torchsummaryX`.
"""
import importlib
import os
import sys
import types

REF_ROOT = os.environ.get("GNNPP_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "utils", "graphUtils", "graphML.py"))


class _Saved:
    def __init__(self):
        self.mods = {}


def _ns(name, relpath):
    m = types.ModuleType(name)
    m.__path__ = [os.path.join(REF_ROOT, relpath)]
    m.__package__ = name
    return m


_PKGS = {
    "utils": "utils",
    "utils.graphUtils": "utils/graphUtils",
    "graphs": "graphs",
    "graphs.models": "graphs/models",
    "dataloader": "dataloader",
}


def load():
    """Returns (graphML module, decentralplanner module, statetransformer module) of
    the real reference.  The modules are registered under private names so the
    product's own drop-in `graphs.*` / `utils.*` packages are never shadowed."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)
    saved = {k: sys.modules.get(k) for k in list(sys.modules)
             if k.split(".")[0] in ("utils", "graphs", "dataloader", "torchsummaryX")}
    for k in saved:
        sys.modules.pop(k, None)
    try:
        for name, rel in _PKGS.items():
            sys.modules[name] = _ns(name, rel)
        stub = types.ModuleType("torchsummaryX")
        stub.summary = lambda *a, **k: None
        sys.modules["torchsummaryX"] = stub
        gml = importlib.import_module("utils.graphUtils.graphML")
        dcp = importlib.import_module("graphs.models.decentralplanner")
        st = importlib.import_module("dataloader.statetransformer")
    finally:
        for k in [k for k in list(sys.modules)
                  if k.split(".")[0] in ("utils", "graphs", "dataloader", "torchsummaryX")]:
            sys.modules.pop(k, None)
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
    return gml, dcp, st


def load_sim():
    """Returns the reference's rollout-simulator module
    (utils/multirobotsim_dcenlocal.py) with its matplotlib-only visualiser import
    (:6) stubbed; used to pin the GSO construction (:320-365)."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REF_ROOT)
    saved = {k: sys.modules.get(k) for k in list(sys.modules)
             if k.split(".")[0] in ("utils", "graphs", "dataloader")}
    for k in saved:
        sys.modules.pop(k, None)
    try:
        for name, rel in _PKGS.items():
            sys.modules[name] = _ns(name, rel)
        viz = types.ModuleType("utils.multipathvisualizerCombine")
        viz.DrawpathCombine = object
        sys.modules["utils.multipathvisualizerCombine"] = viz
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            sim = importlib.import_module("utils.multirobotsim_dcenlocal")
    finally:
        for k in [k for k in list(sys.modules) if k.split(".")[0] in ("utils", "graphs", "dataloader")]:
            sys.modules.pop(k, None)
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
    return sim


class Config:
    """Minimal stand-in for the reference's EasyDict config (utils/config.py:60-212):
    the model only reads num_agents, nGraphFilterTaps and (lazily) device."""

    def __init__(self, num_agents, nGraphFilterTaps, device="cpu"):
        self.num_agents = num_agents
        self.nGraphFilterTaps = nGraphFilterTaps
        self.device = device
