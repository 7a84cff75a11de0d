"""Import the reference's own Python code (read-only checkout) with its absent
third-party dependencies stubbed, so that its cg / ddim / apTweedy / DDPM /
predictors / BaseSampler / MatmulRayTrafo run verbatim on CPU.

TEST INFRASTRUCTURE ONLY, and only usable where the environment variable
SCD_REFERENCE_ROOT names a checkout of the reference project (it is not part of
this repository).  Used by tests/golden/make_golden.py to generate the
committed golden vectors and by tests marked `needs_reference`.
Recipe: SURVEY.md Appendix B.
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get('SCD_REFERENCE_ROOT', '')


def available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, 'src'))


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules.setdefault(name, m)
    return sys.modules[name]


def import_reference():
    """Returns the reference's ``src`` package."""
    if not available():
        raise RuntimeError('no reference checkout: set SCD_REFERENCE_ROOT to the directory that holds its src/ '
                           '(now %r)' % REFERENCE_ROOT)
    if 'src' in sys.modules and getattr(sys.modules['src'], '__scd_ref__', False):
        return sys.modules['src']

    def _missing(*a, **k):
        raise RuntimeError('stubbed third-party function called')

    class _OperatorModule:      # odl.contrib.torch.OperatorModule placeholder
        def __init__(self, *a, **k):
            _missing()

    odl = _stub('odl', uniform_discr=_missing, tomo=types.SimpleNamespace())
    contrib = _stub('odl.contrib')
    ctorch = _stub('odl.contrib.torch', OperatorModule=_OperatorModule)
    discr = _stub('odl.discr', uniform_partition=_missing)
    phantom = _stub('odl.phantom', ellipsoid_phantom=_missing)
    odl.contrib = contrib; contrib.torch = ctorch; odl.discr = discr; odl.phantom = phantom
    _stub('dival', get_standard_dataset=_missing)
    pyd = _stub('pydicom'); fr = _stub('pydicom.filereader', dcmread=_missing); pyd.filereader = fr
    _stub('imageio')
    sk = _stub('skimage'); skm = _stub('skimage.metrics', structural_similarity=_missing); sk.metrics = skm
    _stub('omegaconf', OmegaConf=object)

    class ConfigDict(dict):     # ml_collections.ConfigDict stand-in
        __getattr__ = dict.__getitem__
        __setattr__ = dict.__setitem__
    _stub('ml_collections', ConfigDict=ConfigDict)

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import src  # noqa
    src.__scd_ref__ = True
    return src
