"""TEST INFRASTRUCTURE ONLY -- import the unmodified reference in the build container.

``/root/reference`` exists only in the build container (never on the GPU box), and four
third-party modules the reference imports at module-import time are absent here
(``tvsclib``, ``pyfaust``, ``matplotlib``, ``importlib_resources``; SURVEY.md section 8c).
Registering empty stand-ins in ``sys.modules`` lets every layer module and
``training_helpers`` import and run unmodified: the stand-ins are only touched by
constructors' from-dense paths (tvsclib / pyfaust), which the fixtures bypass via the
``initial_*`` / ``sparse_matrices`` constructor arguments.

Used by ``tests/golden/make_golden.py`` (fixture generation) and by optional local
cross-checks; nothing that runs on the GPU box may call :func:`load_reference`.
"""
import os
import sys
import types

# a checkout of MatthiasKi/structurednets, given by the same variable as in oracle/run_c.py
REFERENCE_SRC = os.path.join(os.environ["SNB200_REFERENCE"], "src") if os.environ.get("SNB200_REFERENCE") else None


def reference_available() -> bool:
    return REFERENCE_SRC is not None and os.path.isdir(os.path.join(REFERENCE_SRC, "structurednets"))


def _stub(name, **attrs):
    mod = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(mod, k, v)
    sys.modules.setdefault(name, mod)
    return sys.modules[name]


class _Missing:
    def __init__(self, *a, **k):
        raise ImportError("third-party dependency of the reference is not installed here")


def load_reference():
    """Returns the imported reference package ``structurednets`` (layers importable)."""
    if not reference_available():
        raise RuntimeError("the reference tree is not present (only exists in the build container)")
    _stub("importlib_resources", files=lambda *_a, **_k: None)
    mpl = _stub("matplotlib")
    _stub("matplotlib.pyplot")
    _stub("matplotlib.patches", Rectangle=_Missing)
    mpl.cm = types.SimpleNamespace(get_cmap=lambda *_a, **_k: None)
    _stub("pyfaust")
    _stub("pyfaust.fact", hierarchical=_Missing)
    _stub("pyfaust.proj", sp=_Missing)
    _stub("pyfaust.factparams", ParamsHierarchical=_Missing, StoppingCriterion=_Missing)
    _stub("tvsclib")
    _stub("tvsclib.mixed_system", MixedSystem=_Missing)
    _stub("tvsclib.toeplitz_operator", ToeplitzOperator=_Missing)
    _stub("tvsclib.system_identification_svd", SystemIdentificationSVD=_Missing)
    if REFERENCE_SRC not in sys.path:
        sys.path.insert(0, REFERENCE_SRC)
    import structurednets  # noqa: F401
    import structurednets.layers.sss_layer  # noqa: F401
    import structurednets.layers.psm_layer  # noqa: F401
    import structurednets.layers.lr_layer  # noqa: F401
    import structurednets.layers.ldr_layer  # noqa: F401
    import structurednets.layers.tl_layer  # noqa: F401
    import structurednets.layers.hmat_layer  # noqa: F401
    import structurednets.training_helpers  # noqa: F401
    return structurednets
