"""Shape path on the GPU through the C ABI: CUDA marching cubes / all-pairs diameters / voxel moments
against the reference's outputs (committed goldens)."""
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
G = os.path.join(HERE, "golden")
pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["blob", "noise", "sparse", "touching_border", "single", "plane"])
def test_calculate_coefficients_matches_reference(name):
    from pyradiomics_b200 import cshape
    d = np.load(os.path.join(G, "shape_random.npz"))
    sa, vol, dia = cshape.calculate_coefficients(d[f"{name}_mask"], d[f"{name}_spacing"])
    ref = d[f"{name}_coeff"]
    assert sa == pytest.approx(ref[0], rel=1e-11, abs=1e-12)
    assert vol == pytest.approx(ref[1], rel=1e-11, abs=1e-9)
    assert list(dia) == list(ref[2:6])                      # bit-identical: same double operations, max is order-free


def test_single_cube_probes_on_device():
    from pyradiomics_b200 import cshape
    pr = np.load(os.path.join(G, "shape_cube_probes.npz"))
    for cfg in range(0, 256, 3):
        m = np.zeros((2, 2, 2), dtype=bool)
        for i in range(8):
            if cfg >> i & 1:
                m[i >> 2 & 1, i >> 1 & 1, i & 1] = True
        sa, vol, _ = cshape.calculate_coefficients(m, pr["spacings"][1])
        assert sa == pytest.approx(pr["probes"][cfg, 1, 0], rel=1e-12, abs=1e-13)
        assert vol == pytest.approx(pr["probes"][cfg, 1, 1], rel=1e-12, abs=1e-13)


@pytest.mark.parametrize("case", ["brain1", "brain2", "breast1", "lung1", "lung2"])
def test_shape_class_matches_reference_class(case):
    from pyradiomics_b200 import featureclasses, image
    exp = json.load(open(os.path.join(G, "shape_expect.json")))[case]
    seg = np.load(os.path.join(G, "segment_cases.npz"))
    sp = tuple(seg[f"{case}_spacing"])
    obj = featureclasses.RadiomicsShape(image.ArrayImage(seg[f"{case}_image"], sp),
                                        image.ArrayImage(seg[f"{case}_mask"].astype(np.uint8), sp))
    got = obj.execute()
    assert set(got) == set(exp["features"])
    for f, v in exp["features"].items():
        assert float(got[f]) == pytest.approx(v, rel=1e-9), f
    for f in ("Maximum3DDiameter", "Maximum2DDiameterSlice", "Maximum2DDiameterColumn", "Maximum2DDiameterRow"):
        assert float(got[f]) == exp["features"][f], f
    for f, v in exp["baseline"].items():                    # the stored CSV at the reference's own tolerance
        assert float(got[f]) == pytest.approx(v, rel=0.03), f


def test_deprecated_features_on_request_and_voxel_mode_refused():
    from pyradiomics_b200 import featureclasses, image
    seg = np.load(os.path.join(G, "segment_cases.npz"))
    sp = tuple(seg["brain2_spacing"])
    img, msk = image.ArrayImage(seg["brain2_image"], sp), image.ArrayImage(seg["brain2_mask"].astype(np.uint8), sp)
    obj = featureclasses.RadiomicsShape(img, msk)
    obj.enableFeatureByName("Compactness2")
    obj.enableFeatureByName("Sphericity")
    got = obj.execute()
    assert float(got["Compactness2"]) == pytest.approx(float(got["Sphericity"]) ** 3, rel=1e-12)
    with pytest.raises(NotImplementedError):
        featureclasses.RadiomicsShape(img, msk, voxelBased=True).execute()


def large_roi_case():
    """96^3 ellipsoid with holes (~5e4 mesh vertices, 1e9 vertex pairs) and its spacing"""
    rng = np.random.default_rng(5)
    z, y, x = np.meshgrid(np.arange(96), np.arange(96), np.arange(96), indexing="ij")
    m = (((z - 47.3) / 40) ** 2 + ((y - 48.2) / 33) ** 2 + ((x - 46.1) / 44) ** 2 < 1.0) & (rng.random(z.shape) > 0.02)
    return m, np.array((1.7, 0.9, 1.2))


def test_large_roi_against_compiled_reference():
    """large_roi_case() against the compiled reference _cshape's outputs (tests/golden/reference_runs.json)"""
    from pyradiomics_b200 import cshape
    ref = json.load(open(os.path.join(G, "reference_runs.json")))["large_roi_shape"]
    m, sp = large_roi_case()
    sa, vol, dia = cshape.calculate_coefficients(m, sp)
    assert sa == pytest.approx(ref["surface_area"], rel=1e-11)
    assert vol == pytest.approx(ref["volume"], rel=1e-11)
    assert tuple(dia) == tuple(ref["diameters"])


SHAPE2D = ["disc", "noise", "sparse", "touching_border", "single", "checker", "ring"]


@pytest.mark.parametrize("name", SHAPE2D)
def test_calculate_coefficients2d_matches_reference(name):
    """CUDA marching squares + all-pairs diameter (rb_calculate_coefficients2D) against the compiled reference's outputs"""
    from pyradiomics_b200 import cshape
    d = np.load(os.path.join(G, "shape2d_golden.npz"))
    per, sur, dia = cshape.calculate_coefficients2D(np.pad(d[name + "_mask"], 1), d[name + "_spacing"])
    ref = d[name + "_coeff"]
    assert per == pytest.approx(ref[0], rel=1e-12)
    assert sur == pytest.approx(ref[1], rel=1e-12, abs=1e-13)
    assert dia == ref[2]                                    # bit-identical: same double operations, max is order-free


def test_shape2d_class_matches_oracle_features_and_guards():
    sys.path.insert(0, os.path.join(HERE, "..", "oracle"))
    import shape_np as S
    from pyradiomics_b200 import featureclasses as FC, image as I
    d = np.load(os.path.join(G, "shape2d_golden.npz"))
    for name in ("disc", "ring", "noise"):
        m, sp = d[name + "_mask"], d[name + "_spacing"]
        ref = S.features2d(m, sp)
        img2 = I.ArrayImage(np.zeros(m.shape, np.int16), sp[::-1])
        got = FC.RadiomicsShape2D(img2, I.ArrayImage(m.astype(np.uint8), sp[::-1])).execute()
        assert set(got) == set(FC.RadiomicsShape2D.NAMES)
        for k, v in got.items():
            assert float(v) == pytest.approx(ref[k], rel=1e-10), (name, k)
        # the same slice as a 3-D image with force2D
        m3 = m[None]
        img3 = I.ArrayImage(np.zeros(m3.shape, np.int16), (sp[1], sp[0], 3.0))
        got3 = FC.RadiomicsShape2D(img3, I.ArrayImage(m3.astype(np.uint8), (sp[1], sp[0], 3.0)), force2D=True, force2Ddimension=0).execute()
        for k, v in got3.items():
            assert float(v) == pytest.approx(ref[k], rel=1e-10), (name, k)
    with pytest.raises(ValueError):
        FC.RadiomicsShape2D(img3, I.ArrayImage(m3.astype(np.uint8)), force2D=False).execute()
    with pytest.raises(NotImplementedError):
        FC.RadiomicsShape2D(img2, I.ArrayImage(m.astype(np.uint8)), voxelBased=True)
