"""Import shim for the UNMODIFIED reference at /root/reference (test infrastructure only).

Used only by ``tests/golden/make_goldens.py`` and ``tools/port_vs_reference.py``: the tests compare
with what ``make_goldens.py`` stored, so no test and nothing on the product path imports this module.

The reference has four dead imports that are not installable here (SURVEY.md section 8c):
``matplotlib.pyplot`` (generators/volumetric_rendering.py:12), ``numpy.lib.type_check.imag``
(siren/siren.py:2), ``fid_evaluation.output_images`` (siren/siren.py:7) and ``kornia.filters``
(curriculums.py:1 -> generators/neural_rendering.py:4).  Each gets an empty stub module.
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("FENERF_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "generators"))


def _stub(name, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    mod = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(mod, k, v)
    sys.modules[name] = mod
    return mod


def load():
    """Returns (generators.generators, siren.siren, curriculums) of the reference."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")
    sys.dont_write_bytecode = True
    mpl = _stub("matplotlib")
    mpl.pyplot = _stub("matplotlib.pyplot")
    import numpy.lib  # noqa: F401
    tc = _stub("numpy.lib.type_check", imag=None)
    sys.modules["numpy.lib"].type_check = tc
    _stub("fid_evaluation", output_images=None)
    k = _stub("kornia")
    k.filters = _stub("kornia.filters", filter2D=None)
    # our own package may have aliased these names (fenerf_b200.install()); drop the aliases
    for name in [n for n in list(sys.modules) if n.split(".")[0] in ("generators", "siren", "curriculums")]:
        mod = sys.modules[name]
        if not getattr(mod, "__file__", "") or not str(mod.__file__).startswith(REFERENCE_ROOT):
            del sys.modules[name]
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import generators.generators as ref_generators
        import siren.siren as ref_siren
        import curriculums as ref_curriculums
    return ref_generators, ref_siren, ref_curriculums
