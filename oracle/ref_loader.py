"""TEST INFRASTRUCTURE ONLY -- imports the *real* reference (pure Python/PyTorch)
from a checkout of the original Fireflies project named by ``FIREFLIES_REF``
(the directory that holds its ``fireflies/`` package) with empty stub modules for
its absent third-party imports (mitsuba, drjit, kornia, geomdl, pywavefront),
following SURVEY.md Appendix C.  The reference is not part of this repository,
so nothing in the ``-m gpu`` tests, ``smoke()`` or ``bench.py`` may call this.
It is used by ``oracle/make_golden.py`` (to write ``tests/golden/*.npz``) and by
the ``not gpu`` tests that cross-check the restatement in ``oracle/ff_oracle.py``
against the reference when ``FIREFLIES_REF`` is set; they skip without it.
"""
import os
import sys
import types

REF_ROOT = os.environ.get("FIREFLIES_REF", "")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "fireflies", "__init__.py"))


def api(root: str) -> dict:
    """AST walk of a package tree: ``names`` maps each file (relative path) to its top-level functions, classes, class methods
    (``Class.method``) and assigned names; ``signatures`` maps ``file::function`` / ``file::Class.method`` to
    ``[positional parameter names, number of them without a default]``.  Plain data, so it can be stored as JSON."""
    import ast
    names, sigs = {}, {}
    for dp, _, files in os.walk(root):
        for f in sorted(files):
            if not f.endswith(".py"):
                continue
            rel = os.path.relpath(os.path.join(dp, f), root)
            with open(os.path.join(dp, f)) as fh:
                tree = ast.parse(fh.read())
            defined = set()
            for node in tree.body:
                if isinstance(node, ast.FunctionDef):
                    defined.add(node.name)
                elif isinstance(node, ast.ClassDef):
                    defined.add(node.name)
                    defined.update(f"{node.name}.{m.name}" for m in node.body if isinstance(m, ast.FunctionDef))
                elif isinstance(node, ast.Assign):
                    defined.update(t.id for t in node.targets if isinstance(t, ast.Name))
                fns = [("", node)] if isinstance(node, ast.FunctionDef) else (
                    [(node.name + ".", m) for m in node.body if isinstance(m, ast.FunctionDef)] if isinstance(node, ast.ClassDef) else [])
                for prefix, fn in fns:
                    params = [a.arg for a in fn.args.posonlyargs + fn.args.args]
                    sigs[f"{rel}::{prefix}{fn.name}"] = [params, len(params) - len(fn.args.defaults)]
            names[rel] = sorted(defined)
    return {"names": names, "signatures": sigs}


def load():
    """Return the reference ``fireflies`` package (imported once, cached)."""
    if "fireflies" in sys.modules and getattr(sys.modules["fireflies"], "_ffb_ref", False):
        return sys.modules["fireflies"]
    if not available():
        raise RuntimeError(f"reference not found under FIREFLIES_REF={REF_ROOT!r}")
    for name in ("mitsuba", "drjit", "kornia", "geomdl", "pywavefront"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["geomdl"].NURBS = types.SimpleNamespace(Curve=object)
    sys.modules["drjit"].wrap_ad = lambda **kw: (lambda f: f)
    kf = types.ModuleType("kornia.filters")
    sys.modules["kornia"].filters = kf
    sys.modules["kornia.filters"] = kf
    # mitsuba types touched by scene.py (fakes; see tests/fake_mitsuba.py for the params object)
    mi = sys.modules["mitsuba"]
    for tname in ("Float", "Float32", "Transform4f", "ScalarTransform3f", "TensorXf"):
        if not hasattr(mi, tname):
            setattr(mi, tname, type(tname, (), {}))
    sys.path.insert(0, REF_ROOT)
    try:
        import fireflies  # noqa: F401
        import fireflies.graphics.rasterization  # noqa: F401
        import fireflies.projection  # noqa: F401
        import fireflies.postprocessing  # noqa: F401
        import fireflies.utils.math  # noqa: F401
    finally:
        sys.path.remove(REF_ROOT)
    ff = sys.modules["fireflies"]
    # intent shims for reference bugs (fireflies/utils/transforms.py is an empty file)
    tr = sys.modules["fireflies.utils.transforms"]
    m = sys.modules["fireflies.utils.math"]
    for fn in ("transform_points", "transform_directions", "toMat4x4"):
        setattr(tr, fn, getattr(m, fn))
    ff._ffb_ref = True
    return ff
