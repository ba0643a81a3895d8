"""Loads the LIVE reference (babbu3682/MTD-GAN) from the checkout named by $MTDGAN_REFERENCE, for regenerating
the golden vectors under tests/golden/.  The tests never import the reference: they compare against those vectors."""
import os
import sys
import types
import importlib

REF_ROOT = os.environ.get("MTDGAN_REFERENCE", "")


def reference_available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "arch", "Ours", "networks.py"))


def load_reference():
    """Returns a namespace with the reference's hot-path modules.  The reference's top-level module
    names (losses, arch, module) collide with this repo's drop-in mirrors, so the reference is
    imported under a temporarily swapped sys.path / sys.modules and handed back as objects."""
    assert reference_available(), "set MTDGAN_REFERENCE to a checkout of babbu3682/MTD-GAN"
    try:                       # the reference's losses.py imports torchvision; its op registration inspects sys.modules
        import torchvision  # noqa: F401   and must not run while the reference's namespace packages are half-imported
    except Exception:
        pass
    saved_path = list(sys.path)
    saved_mods = {k: sys.modules.pop(k) for k in list(sys.modules)
                  if k in ("losses", "arch", "module") or k.startswith(("arch.", "module."))}
    had_cvxpy = "cvxpy" in sys.modules
    try:
        sys.path[:] = [REF_ROOT] + [p for p in saved_path if os.path.abspath(p or ".") != os.path.abspath(
            os.path.join(os.path.dirname(__file__), ".."))]
        if not had_cvxpy:
            sys.modules["cvxpy"] = types.ModuleType("cvxpy")      # only NashMTL uses it (SURVEY §8c)
        ns = types.SimpleNamespace()
        ns.networks = importlib.import_module("arch.Ours.networks")
        ns.losses = importlib.import_module("losses")
        ns.pcgrad = importlib.import_module("module.pcgrad")
        ns.weight_methods = importlib.import_module("module.weight_methods")
        return ns
    finally:
        for k in list(sys.modules):
            if k in ("losses", "arch", "module") or k.startswith(("arch.", "module.")):
                del sys.modules[k]
        sys.modules.update(saved_mods)
        if not had_cvxpy:
            sys.modules.pop("cvxpy", None)
        sys.path[:] = saved_path
