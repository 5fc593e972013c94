"""Import the unmodified reference package from oracle/_ref/ (installed there by build(), see
oracle/ref_install.py).

pykg2vec imports hyperopt (common.py:8-9), seaborn, matplotlib, networkx and scikit-learn
(utils/visualization.py:7-15) at module scope; none of them is on the scored path, so empty stub modules
are registered first for those that are not installed (SURVEY.md Appendix A).  Nothing of the reference
is modified."""
import importlib.util
import os
import sys
import types

REF_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")


def available():
    return os.path.isdir(os.path.join(REF_DIR, "pykg2vec"))


def _missing(name):
    return name not in sys.modules and importlib.util.find_spec(name) is None


def install_stubs():
    if "hyperopt" not in sys.modules:
        ho = types.ModuleType("hyperopt")
        ho.hp = types.SimpleNamespace()
        for n in ("fmin", "tpe", "Trials", "STATUS_OK", "space_eval"):
            setattr(ho, n, None)
        pyll = types.ModuleType("hyperopt.pyll")
        base = types.ModuleType("hyperopt.pyll.base")
        base.scope = types.SimpleNamespace()
        sys.modules.update({"hyperopt": ho, "hyperopt.pyll": pyll, "hyperopt.pyll.base": base})
    if "seaborn" not in sys.modules:
        sb = types.ModuleType("seaborn")
        sb.set_style = lambda *a, **k: None
        sys.modules["seaborn"] = sb
    if "matplotlib" not in sys.modules:
        mpl = types.ModuleType("matplotlib")
        plt = types.ModuleType("matplotlib.pyplot")
        mpl.colors = types.SimpleNamespace()
        mpl.pyplot = plt
        sys.modules.update({"matplotlib": mpl, "matplotlib.pyplot": plt})
    if _missing("networkx"):
        sys.modules["networkx"] = types.ModuleType("networkx")
    if _missing("sklearn"):
        sk = types.ModuleType("sklearn")
        manifold = types.ModuleType("sklearn.manifold")
        manifold.TSNE = None
        sk.manifold = manifold
        sys.modules.update({"sklearn": sk, "sklearn.manifold": manifold})


def load():
    """-> the imported `pykg2vec` package of oracle/_ref (raises ImportError when it is not installed)."""
    if not available():
        raise ImportError("oracle/_ref/pykg2vec not found: build() installs it from a checkout of the reference "
                          "(oracle/ref_install.py)")
    install_stubs()
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import pykg2vec
    return pykg2vec
