"""CPU test of the drop-in boundary: `pyradiomics_b200.install()` against a package registry built like the reference's --
the feature-class dictionary, the per-module `cMatrices` rebinding (SURVEY.md 8b) and `cShape` keeping
`calculate_coefficients2D` reachable for radiomics.shape2D (reference radiomics/shape2D.py:99) -- and the feature names
against the reference classes' (tests/golden/reference_runs.json).  No CUDA call is made."""
import importlib
import json
import os
import sys

import pytest

from helpers import GOLDEN

# A package laid out like the reference's radiomics: getFeatureClasses() imports the class modules once and caches the
# dictionary it returns (radiomics/__init__.py:104-117); the extensions are package attributes that every class module
# binds by name at import time (`from radiomics import base, cMatrices` in glcm.py, `... cShape` in shape.py / shape2D.py).
STANDIN = {
    "__init__.py": '''
import importlib
import inspect
import types

cMatrices = types.ModuleType("_cmatrices")
cShape = types.ModuleType("_cshape")
cShape.calculate_coefficients = lambda *a: None
cShape.calculate_coefficients2D = lambda *a: None
_featureClasses = None


def getFeatureClasses():
    global _featureClasses
    if _featureClasses is None:
        _featureClasses = {}
        for mod in ("firstorder", "glcm", "gldm", "glrlm", "glszm", "ngtdm", "shape", "shape2D"):
            for _, cls in inspect.getmembers(importlib.import_module(__name__ + "." + mod), inspect.isclass):
                if "RadiomicsFeaturesBase" in [b.__name__ for b in cls.__mro__[1:]]:
                    _featureClasses[mod] = cls
    return _featureClasses
''',
    "base.py": "class RadiomicsFeaturesBase:\n    pass\n",
}
for _mod, _ext in (("firstorder", "cMatrices"), ("glcm", "cMatrices"), ("gldm", "cMatrices"), ("glrlm", "cMatrices"),
                   ("glszm", "cMatrices"), ("ngtdm", "cMatrices"), ("shape", "cShape"), ("shape2D", "cShape")):
    STANDIN[f"{_mod}.py"] = (f"from radiomics_standin import base, {_ext}\n\n\n"
                             f"class Radiomics{_mod}(base.RadiomicsFeaturesBase):\n    pass\n")


@pytest.fixture(scope="module")
def rad(tmp_path_factory):
    root = tmp_path_factory.mktemp("standin")
    pkg = root / "radiomics_standin"
    pkg.mkdir()
    for name, src in STANDIN.items():
        (pkg / name).write_text(src)
    sys.path.insert(0, str(root))
    try:
        yield importlib.import_module("radiomics_standin")
    finally:
        sys.path.remove(str(root))
        for m in [m for m in sys.modules if m == "radiomics_standin" or m.startswith("radiomics_standin.")]:
            del sys.modules[m]


def test_install_registers_classes_and_rebinds_cmatrices(rad):
    import pyradiomics_b200 as B
    from pyradiomics_b200 import cmatrices, cshape, featureclasses as FC
    orig_cshape = rad.cShape
    classes = B.install(rad)
    assert classes is rad.getFeatureClasses()
    for name, cls in {**FC.FEATURE_CLASSES, **FC.NEXT_CLASSES}.items():
        assert rad.getFeatureClasses()[name] is cls
        # the reference accepts a class by the NAME of a base in its MRO (radiomics/__init__.py:95-99)
        assert "RadiomicsFeaturesBase" in [k.__name__ for k in cls.__mro__]
    assert rad.cMatrices is cmatrices
    for mod in ("glcm", "glrlm", "glszm", "gldm", "ngtdm", "firstorder"):
        assert importlib.import_module(f"{rad.__name__}.{mod}").cMatrices is cmatrices
    # cShape: both entry points of the reference's _cshape are served (radiomics/src/_cshape.c:33-39), and a name the
    # replacement does not know still resolves to the reference's own extension
    assert rad.cShape is cshape
    assert rad.cShape.calculate_coefficients is cshape.calculate_coefficients
    assert rad.cShape.calculate_coefficients2D is cshape.calculate_coefficients2D
    sh2 = importlib.import_module(f"{rad.__name__}.shape2D")
    importlib.reload(sh2)                                              # a later (re)import of shape2D keeps working
    assert sh2.cShape.calculate_coefficients2D is cshape.calculate_coefficients2D
    assert cshape.__doc__ and cshape._fallback is orig_cshape
    with pytest.raises(AttributeError):
        cshape.no_such_function


def test_feature_names_and_docstrings_match_the_reference_classes():
    """reference tests/test_docstrings.py: every get<Name>FeatureValue has a docstring; names (and their deprecation flags)
    equal the reference classes' getFeatureNames()"""
    from pyradiomics_b200 import featureclasses as FC
    ref = json.load(open(os.path.join(GOLDEN, "reference_runs.json")))["feature_names"]
    for name in ("glcm", "glrlm", "glszm", "gldm", "ngtdm", "firstorder", "shape", "shape2D"):
        ours = {**FC.FEATURE_CLASSES, **FC.NEXT_CLASSES}[name]
        assert ours.getFeatureNames() == ref[name]
        for f in ours.getFeatureNames():
            assert getattr(ours, f"get{f}FeatureValue").__doc__


def test_crop_to_tumor_mask_matches_the_reference_arithmetic():
    """reference imageoperations.py:407-445: lower crop = bb_lo - pad, upper crop = size - bb_hi - pad - 1, both clipped at 0"""
    import numpy as np
    from pyradiomics_b200 import image as I, imageoperations as IO
    rng = np.random.default_rng(0)
    img = rng.integers(0, 100, (9, 11, 13)).astype(np.int16)                 # (z,y,x)
    msk = np.zeros(img.shape, np.uint8)
    msk[2:5, 0:4, 6:12] = 1
    bb = np.array([6, 11, 0, 3, 2, 4])                                        # x_lo,x_hi,y_lo,y_hi,z_lo,z_hi
    for pad in (0, 1, 3):
        size = np.array(img.shape[::-1])
        lo = np.maximum(bb[0::2] - pad, 0)
        up = np.maximum(size - bb[1::2] - pad - 1, 0)
        ref = img[lo[2]:size[2] - up[2], lo[1]:size[1] - up[1], lo[0]:size[0] - up[0]]
        ci, cm = IO.cropToTumorMask(I.ArrayImage(img, (1, 2, 3)), I.ArrayImage(msk, (1, 2, 3)), bb, padDistance=pad)
        assert np.array_equal(ci.array, ref) and cm.array.shape == ref.shape
        assert ci.GetSpacing() == (1.0, 2.0, 3.0)
        assert cm.array.sum() == msk.sum()
