"""The PRODUCT's plugin classes on the CPU box: everything above the device layer -- matrix post-processing
(symmetrise / weight / empty-angle drop), the scalar feature formulas of pyradiomics_b200/_matrix_features.py, feature
enabling, deprecated features -- runs unchanged; only the three calls that need a GPU (the per-image discretisation and the
two device matrix builders) are replaced, in this test, by the oracle's C port of the reference.  Checked against EVERY
column of the reference's five texture baseline CSVs that does not need resampling (160 of 185) and against the
reference's golden matrices.  (The same classes over the CUDA matrices: tests/test_plugins_gpu.py.)"""
import json
import os

import numpy as np
import pytest

import cmatrices_oracle as O
import pipeline as PL
from helpers import GOLDEN
from pyradiomics_b200 import cmatrices, featureclasses as FC, image as I

CLASSES = ("glcm", "glrlm", "glszm", "gldm", "ngtdm")


class OracleDeviceImage:
    """stands in for featureclasses.DeviceImage: numpy binning + the oracle's matrices (test only)"""

    def __init__(self, imageArray, maskRaw, label, masked, settings):
        m = np.asarray(maskRaw) == label
        lev, self.edges, levels, Ng = PL.bin_image(np.asarray(imageArray), m, settings.get("binWidth", 25), settings.get("binCount"))
        self.lev = np.ascontiguousarray(np.where(m, lev, 0), dtype=np.int32)
        self.mask = m
        self.grayLevels = np.asarray(levels, np.int64)
        self.Ng = int(Ng)
        self.levels = self                      # the "device tensor" handed to cmatrices.calculate_*_device below

    def binned_host(self):
        return self.lev.astype(np.int64)

    def segment_texture(self, distances, alpha, force2D, force2Ddimension):
        d = np.array(list(distances), np.int32)
        f2d = force2Ddimension if force2D else -1
        Pg, ang = O.calculate_glcm(self.lev, self.mask, d, self.Ng, force2D, f2d)
        return {"glcm": (Pg, ang), "gldm": O.calculate_gldm(self.lev, self.mask, d, self.Ng, int(alpha), force2D, f2d),
                "ngtdm": O.calculate_ngtdm(self.lev, self.mask, d, self.Ng, force2D, f2d)}


@pytest.fixture()
def oracle_device(monkeypatch):
    monkeypatch.setattr(FC, "device_image", lambda img, msk, label, masked, settings: OracleDeviceImage(img, msk, label, masked, settings))
    monkeypatch.setattr(cmatrices, "calculate_glrlm_device",
                        lambda dev, Ng, Nr, f2, f2d: O.calculate_glrlm(dev.lev, dev.mask, Ng, Nr, f2, f2d if f2 else -1))
    monkeypatch.setattr(cmatrices, "calculate_glszm_device",
                        lambda dev, Ng, f2, f2d: O.calculate_glszm(dev.lev, dev.mask, Ng, int(dev.mask.sum()), f2, f2d if f2 else -1))


def _columns():
    cases = np.load(os.path.join(GOLDEN, "segment_cases.npz"))
    base = json.load(open(os.path.join(GOLDEN, "segment_expect.json")))
    extra = json.load(open(os.path.join(GOLDEN, "segment_expect_extra.json")))
    masks = np.load(os.path.join(GOLDEN, "segment_extra.npz"))
    return cases, base, extra, masks


@pytest.mark.parametrize("cname", CLASSES)
def test_plugin_classes_over_oracle_matrices_match_every_baseline_column(oracle_device, cname):
    cases, base, extra, masks = _columns()
    cols = dict(base[cname])
    cols.update(extra[cname])
    assert len(cols) == (35 if cname in ("glcm", "glrlm") else 30)      # (the *_combined columns exist for GLCM / GLRLM only)
    for test, e in cols.items():
        c = e["case"]
        img = cases[c + "_image"]
        m = masks[test + "_mask"] if test + "_mask" in masks.files else cases[c + "_mask"]
        if "normalize" in e:
            n = e["normalize"]
            img = (img.astype(np.float64) - n["mean"]) / n["std"] * n["scale"]
        obj = FC.FEATURE_CLASSES[cname](I.ArrayImage(img, cases[c + "_spacing"]), I.ArrayImage(m.astype(np.uint8), cases[c + "_spacing"]),
                                        **e["settings"])
        got = obj.execute()
        assert set(got) == set(e["features"]), (test, set(got) ^ set(e["features"]))
        for f, v in e["features"].items():
            assert abs(float(got[f]) - v) <= 1e-9 * max(abs(v), 1e-12), (cname, test, f, float(got[f]), v)


@pytest.mark.parametrize("cname", CLASSES)
def test_plugin_classes_over_oracle_matrices_match_reference_runs_of_other_settings(oracle_device, cname):
    """weighting norms (featureclasses._weights), several distances, asymmetric GLCM, force2D, binCount, gldm_a"""
    cases = np.load(os.path.join(GOLDEN, "segment_cases.npz"))
    expect = json.load(open(os.path.join(GOLDEN, "segment_expect_variants.json")))[cname]
    for test, e in expect.items():
        c = e["case"]
        sp = cases[c + "_spacing"]
        got = FC.FEATURE_CLASSES[cname](I.ArrayImage(cases[c + "_image"], sp), I.ArrayImage(cases[c + "_mask"].astype(np.uint8), sp),
                                        **e["settings"]).execute()
        assert set(got) == set(e["features"]), (test, set(got) ^ set(e["features"]))
        for f, v in e["features"].items():
            assert np.isclose(float(got[f]), v, rtol=1e-9, atol=1e-12, equal_nan=True), (cname, test, e["settings"], f, float(got[f]), v)


@pytest.mark.parametrize("case", ["brain1", "brain2", "breast1", "lung1", "lung2"])
def test_plugin_processed_matrices_over_oracle_matrices_match_the_golden_matrices(oracle_device, case):
    """reference tests/test_matrices.py:35-65 through the product's _calculateMatrix post-processing"""
    cases = np.load(os.path.join(GOLDEN, "segment_cases.npz"))
    img = I.ArrayImage(cases[case + "_image"], cases[case + "_spacing"])
    msk = I.ArrayImage(cases[case + "_mask"].astype(np.uint8), cases[case + "_spacing"])
    for cname in CLASSES:
        obj = FC.FEATURE_CLASSES[cname](img, msk, binWidth=25)
        obj._initCalculation()
        P = getattr(obj, "P_" + cname)[0]
        assert P.shape == cases[f"{case}_{cname}_P"].shape
        assert np.abs(P - cases[f"{case}_{cname}_P"]).max() < 1e-12


def test_plugin_feature_enabling_and_deprecated_features(oracle_device):
    cases = np.load(os.path.join(GOLDEN, "segment_cases.npz"))
    img, msk = cases["breast1_image"], cases["breast1_mask"].astype(np.uint8)
    obj = FC.RadiomicsGLCM(img, msk, binWidth=25)
    obj.enableFeatureByName("Contrast")
    obj.enableFeatureByName("Homogeneity1")          # deprecated in the reference: enabled by name -> skipped, not an error
    got = obj.execute()
    assert set(got) == {"Contrast"}
    with pytest.raises(LookupError):
        obj.enableFeatureByName("NoSuchFeature")
    assert FC.RadiomicsGLCM.getFeatureNames()["Homogeneity1"] is True and FC.RadiomicsGLCM.getFeatureNames()["Contrast"] is False


def test_plugin_firstorder_segment_mode_matches_every_baseline_column_without_resampling(oracle_device):
    """RadiomicsFirstOrder reduces the ROI vector on the host in segment mode: base, resegmentation and normalization columns
    of baseline_firstorder.csv (15 of 20; the resampling ones need the GPU resampler, tests/test_resample_gpu.py)"""
    cases, _, extra, masks = _columns()
    cols = dict(json.load(open(os.path.join(GOLDEN, "segment_expect_firstorder.json"))))
    cols.update(extra["firstorder"])
    assert len(cols) == 15
    for test, e in cols.items():
        c = e["case"]
        img = cases[c + "_image"]
        m = masks[test + "_mask"] if test + "_mask" in masks.files else cases[c + "_mask"]
        if "normalize" in e:
            n = e["normalize"]
            img = (img.astype(np.float64) - n["mean"]) / n["std"] * n["scale"]
        sp = cases[c + "_spacing"]
        got = FC.RadiomicsFirstOrder(I.ArrayImage(img, sp), I.ArrayImage(m.astype(np.uint8), sp), **e["settings"]).execute()
        for f, v in e["features"].items():
            assert abs(float(got[f]) - v) <= 1e-9 * max(abs(v), 1e-12), (test, f, float(got[f]), v)


# ---- shape classes: the formulas above the device coefficients (reference shape.py / shape2D.py)
@pytest.fixture()
def oracle_shape(monkeypatch):
    import shape_np as S
    from pyradiomics_b200 import cshape, imageoperations as IO
    monkeypatch.setattr(IO, "_to_device", lambda a: np.asarray(a))

    def coeff(mask, spacing_zyx):
        sa, vol, dia = S.coefficients(np.asarray(mask), np.asarray(spacing_zyx))
        return sa, vol, list(dia), 0

    def moments(mask):
        z, y, x = [c.astype(object) for c in np.nonzero(np.asarray(mask))]       # Python ints: exact like the kernel's 64-bit sums
        return [len(z), int(z.sum()), int(y.sum()), int(x.sum()), int((z * z).sum()), int((z * y).sum()), int((z * x).sum()),
                int((y * y).sum()), int((y * x).sum()), int((x * x).sum())]

    monkeypatch.setattr(cshape, "coefficients_device", coeff)
    monkeypatch.setattr(cshape, "moments_device", moments)
    monkeypatch.setattr(cshape, "calculate_coefficients2D", lambda m, sp: S.coefficients2d(np.asarray(m), np.asarray(sp)))


@pytest.mark.parametrize("case", ["brain1", "brain2", "breast1", "lung1", "lung2"])
def test_plugin_shape_class_over_oracle_coefficients(oracle_shape, case):
    """RadiomicsShape's formulas (sphericity, axis lengths from exact integer moments, ...) against the reference class's own
    values (tests/golden/shape_expect.json: full precision) and the baseline CSV"""
    exp = json.load(open(os.path.join(GOLDEN, "shape_expect.json")))[case]
    seg = np.load(os.path.join(GOLDEN, "segment_cases.npz"))
    sp = seg[case + "_spacing"]
    obj = FC.RadiomicsShape(I.ArrayImage(seg[case + "_image"], sp), I.ArrayImage(seg[case + "_mask"].astype(np.uint8), sp))
    got = obj.execute()
    assert set(got) == set(FC.RadiomicsShape.NAMES)
    for f, v in exp["features"].items():
        if f in got:
            assert float(got[f]) == pytest.approx(v, rel=1e-9), f
    for f, v in exp["baseline"].items():
        assert float(got[f]) == pytest.approx(v, rel=0.03), f


def test_plugin_shape2d_class_over_oracle_coefficients(oracle_shape):
    import shape_np as S
    d = np.load(os.path.join(GOLDEN, "shape2d_golden.npz"))
    for name in ("disc", "noise", "ring"):
        m, sp = d[name + "_mask"], d[name + "_spacing"]
        ref = S.features2d(m, sp)
        obj = FC.RadiomicsShape2D(I.ArrayImage(m.astype(np.float64), tuple(sp[::-1])), I.ArrayImage(m.astype(np.uint8), tuple(sp[::-1])))
        got = obj.execute()
        assert set(got) == set(FC.RadiomicsShape2D.NAMES)
        for f in got:
            assert float(got[f]) == pytest.approx(ref[f], rel=1e-10, nan_ok=True), (name, f)
    # a 3-D mask with one slice + force2D (shape2D.py:62-84); more than one slice is refused
    m, sp = d["disc_mask"], d["disc_spacing"]
    m3 = m[None]
    obj = FC.RadiomicsShape2D(I.ArrayImage(m3.astype(np.float64), (sp[1], sp[0], 3.0)), I.ArrayImage(m3.astype(np.uint8), (sp[1], sp[0], 3.0)),
                              force2D=True, force2Ddimension=0)
    ref = S.features2d(m, sp)
    got = obj.execute()
    assert float(got["Perimeter"]) == pytest.approx(ref["Perimeter"], rel=1e-12)
    with pytest.raises(ValueError):
        FC.RadiomicsShape2D(np.zeros((2,) + m.shape), np.repeat(m3, 2, 0).astype(np.uint8), force2D=True, force2Ddimension=0).execute()


# ---- resampleImage: the geometry arithmetic of the product (grid anchored at index 0, pad, clipping, single-slice rule,
# origin of the new grid) with the GPU interpolation replaced by scipy's (test only)
@pytest.fixture()
def scipy_resampler(monkeypatch):
    import scipy.ndimage as ndi
    import torch
    from pyradiomics_b200 import imageoperations as IO

    def to_dev(a):
        a = np.ascontiguousarray(np.asarray(a))
        return torch.from_numpy(a.view(np.uint8) if a.dtype == np.bool_ else a)

    def resample_device(arr_t, out_size_zyx, start_zyx, step_zyx, interpolator=3, default_value=0.0, out_dtype=None):
        a = arr_t.numpy()
        g = [start_zyx[d] + step_zyx[d] * np.arange(out_size_zyx[d]) for d in range(3)]
        zz, yy, xx = np.meshgrid(*g, indexing="ij")
        if interpolator == 3:
            coef = ndi.spline_filter(a.astype(np.float64), order=3, mode="mirror") if min(a.shape) > 1 else None
            if coef is None:                                   # a singleton axis: filter the others only
                coef = a.astype(np.float64)
                for ax in range(3):
                    if a.shape[ax] > 1:
                        coef = ndi.spline_filter1d(coef, order=3, axis=ax, mode="mirror")
            val = ndi.map_coordinates(coef, [zz, yy, xx], order=3, mode="mirror", prefilter=False)
        elif interpolator == 1:
            val = ndi.map_coordinates(a.astype(np.float64), [zz, yy, xx], order=1, mode="nearest")
        else:
            val = ndi.map_coordinates(a.astype(np.float64), [np.floor(zz + 0.5), np.floor(yy + 0.5), np.floor(xx + 0.5)], order=0, mode="nearest")
        inside = np.ones(val.shape, bool)
        for c, n in ((zz, a.shape[0]), (yy, a.shape[1]), (xx, a.shape[2])):
            inside &= (c >= -0.5) & (c < n - 0.5)
        val = np.where(inside, val, default_value)
        if np.issubdtype(a.dtype, np.integer):
            info = np.iinfo(a.dtype)
            val = np.trunc(np.clip(val, info.min, info.max))
        return torch.from_numpy(np.ascontiguousarray(val.astype(a.dtype)))

    monkeypatch.setattr(IO, "_to_device", to_dev)
    monkeypatch.setattr(IO, "resample_device", resample_device)
    return IO


def test_plugin_resampleImage_grid_equals_the_oracle_on_the_baseline_case(scipy_resampler):
    import resample_np as RS
    IO = scipy_resampler
    z = np.load(os.path.join(GOLDEN, "resample_breast1.npz"))
    sp = tuple(float(v) for v in z["spacing"])
    for new, interp in (((2, 2, 2), "sitkBSpline"), ((1.5, 1.0, 0), "sitkBSpline"), ((3, 3, 3), "sitkLinear"), ((2, 2, 2), "sitkNearestNeighbor")):
        ri, rm = IO.resampleImage(I.ArrayImage(z["image"], sp), I.ArrayImage(z["mask"], sp), resampledPixelSpacing=list(new),
                                  interpolator=interp, padDistance=5)
        order = {"sitkBSpline": 3, "sitkLinear": 1, "sitkNearestNeighbor": 0}[interp]
        oi, om, onew = RS.resample(z["image"], z["mask"], sp, new, order=order)
        assert np.array_equal(I.as_array(rm), om), (new, interp)
        if order != 0:
            assert np.array_equal(I.as_array(ri), oi), (new, interp)
        assert np.allclose(I.spacing_xyz(ri), onew) and I.as_array(ri).dtype == z["image"].dtype
        size, start, step, _ = RS.grid(z["mask"], sp, new)
        assert np.allclose(I.origin_xyz(ri), np.array(start) * np.array(sp))        # TransformContinuousIndexToPhysicalPoint of voxel 0
    # same spacing: nothing to interpolate, the call degenerates to the crop (:517-537)
    ci, cm = IO.resampleImage(I.ArrayImage(z["image"], sp), I.ArrayImage(z["mask"], sp), resampledPixelSpacing=list(sp), padDistance=2)
    idx = np.array(np.where(z["mask"] == 1))
    want = tuple(slice(max(int(a) - 2, 0), min(int(b) + 3, n)) for a, b, n in zip(idx.min(1), idx.max(1), z["mask"].shape))
    assert np.array_equal(I.as_array(cm), z["mask"][want]) and np.array_equal(I.as_array(ci), z["image"][want])


def test_plugin_resampleImage_single_slice_roi_and_errors(scipy_resampler):
    import resample_np as RS
    IO = scipy_resampler
    rng = np.random.default_rng(5)
    img = rng.integers(0, 500, (6, 20, 22)).astype(np.int16)
    m = np.zeros(img.shape, np.uint8)
    m[3, 4:15, 5:17] = 1                                  # single-slice ROI: that axis keeps its spacing (:509-511)
    sp = (0.5, 0.5, 3.0)
    ri, rm = IO.resampleImage(I.ArrayImage(img, sp), I.ArrayImage(m, sp), resampledPixelSpacing=[1.0, 1.0, 1.0])
    oi, om, onew = RS.resample(img, m, sp, (1.0, 1.0, 1.0))
    assert np.allclose(I.spacing_xyz(ri), onew) and onew[2] == 3.0
    assert np.array_equal(I.as_array(ri), oi) and np.array_equal(I.as_array(rm), om)
    with pytest.raises(ValueError):
        IO.resampleImage(I.ArrayImage(img, sp), I.ArrayImage(np.zeros_like(m), sp), resampledPixelSpacing=[1, 1, 1])
    with pytest.raises(ValueError):
        IO.resampleImage(None, I.ArrayImage(m, sp), resampledPixelSpacing=[1, 1, 1])


# ---- getWaveletImage / _swt3: the level loop, the single wrap-padding of odd axes, cropping and the names the reference
# generates, with the device transform of one level replaced by the oracle's (test only)
@pytest.fixture()
def numpy_swt(monkeypatch):
    import torch
    import filters_np as FN
    from pyradiomics_b200 import imageoperations as IO
    monkeypatch.setattr(IO, "_to_device", lambda a: torch.from_numpy(np.ascontiguousarray(np.asarray(a))))

    def level1(x, axes, lo, hi, z_range=None):
        dec = FN.swtn_level1(x.numpy(), np.asarray(lo, float), np.asarray(hi, float), [int(a) for a in axes])
        return {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in dec.items()}

    monkeypatch.setattr(IO, "swt_level1_device", level1)
    return IO


@pytest.mark.parametrize("shape,kw", [((9, 10, 11), {}), ((8, 9, 7), dict(level=2)), ((7, 8, 9), dict(level=2, start_level=1)),
                                      ((6, 9, 8), dict(force2D=True, force2Ddimension=0)), ((11, 12), {}),
                                      ((8, 8, 9), dict(wavelet="haar")), ((9, 7, 8), dict(wavelet="db2", level=2))])
def test_plugin_wavelet_generator_equals_the_oracle_level_loop(numpy_swt, shape, kw):
    import filters_np as FN
    IO = numpy_swt
    rng = np.random.default_rng(len(shape) + sum(shape))
    img = rng.normal(100, 40, shape)
    nd = len(shape)
    axes = list(range(nd - 1, -1, -1))
    if kw.get("force2D"):
        axes.remove(kw.get("force2Ddimension", 0))
    lo, hi = IO.wavelet_filters(kw.get("wavelet", "coif1"))
    approx, levels = FN.swt3_levels(img, lo, hi, axes, kw.get("level", 1), kw.get("start_level", 0))
    want = {}
    for i, bands in enumerate(levels, start=1):
        for key, arr in bands.items():
            if set(key) == {"a"}:
                continue
            name = key.replace("a", "L").replace("d", "H")                   # imageoperations.py:954
            want[(f"wavelet-{name}" if i == 1 else f"wavelet{i}-{name}")] = arr
    want[f"wavelet-{'L' * len(axes)}" if len(levels) == 1 else f"wavelet{len(levels)}-{'L' * len(axes)}"] = approx
    got = {name: I.as_array(im) for im, name, _ in IO.getWaveletImage(img, None, **kw)}
    assert list(got) == list(want)                          # same names in the reference's order (imageoperations.py:877-896)
    assert len(got) == kw.get("level", 1) * (2 ** len(axes) - 1) + 1
    for name in want:
        assert got[name].shape == img.shape
        assert np.array_equal(got[name], want[name]), name


def test_plugin_log_generator_checks_and_names(monkeypatch):
    """getLoGImage's guards and names (reference imageoperations.py:807-836) with the device filter stubbed out"""
    import torch
    from pyradiomics_b200 import imageoperations as IO
    calls = []
    monkeypatch.setattr(IO, "_to_device", lambda a: torch.from_numpy(np.ascontiguousarray(np.asarray(a))))
    monkeypatch.setattr(IO, "log_filter_device", lambda x, sigma, spacing_zyx: calls.append((sigma, spacing_zyx)) or x.to(torch.float32))
    img = I.ArrayImage(np.zeros((8, 10, 12), np.int16), (0.5, 1.0, 2.0))
    got = [(name, I.as_array(im).dtype) for im, name, _ in IO.getLoGImage(img, None, sigma=[1.0, 2.5, 3, 0.0, -1, 30.0])]
    # sigma 30 mm / spacing 2 mm -> needs 16 planes, the image has 8: skipped; 0 and negative: skipped
    assert [n for n, _ in got] == ["log-sigma-1-0-mm-3D", "log-sigma-2-5-mm-3D", "log-sigma-3-mm-3D"]
    assert all(dt == np.float32 for _, dt in got)                      # ITK's filter returns Float32
    assert calls == [(1.0, (2.0, 1.0, 0.5)), (2.5, (2.0, 1.0, 0.5)), (3.0, (2.0, 1.0, 0.5))]
    assert list(IO.getLoGImage(I.ArrayImage(np.zeros((3, 10, 12)), (1, 1, 1)), None, sigma=[1.0])) == []      # an axis < 4
    assert list(IO.getLoGImage(np.zeros((10, 12)), None, sigma=[1.0])) == []                                   # 2-D image
    assert list(IO.getLoGImage(img, None)) == []                                                               # no sigma given


def test_bin_edges_from_min_max_equal_the_reference_arithmetic_for_every_dtype():
    """imageoperations._edges_from_minmax (the host half of binImage: the GPU only reduces min / max and digitizes) against
    the reference's getBinEdges arithmetic on the ROI vector (oracle/pipeline.bin_edges = imageoperations.py:119-149), in the
    image's own scalar type: float32 images round differently from float64 ones, integers promote in np.arange"""
    from pyradiomics_b200 import imageoperations as IO
    rng = np.random.default_rng(17)
    n = 0
    for dt in (np.int16, np.int32, np.float32, np.float64):
        for trial in range(120):
            scale = [1, 7, 300, 4000][trial % 4]
            v = rng.normal(rng.uniform(-scale, scale), scale, 50)
            if trial % 9 == 0:
                v[:] = v[0]                                        # flat region
            v = v.astype(dt)
            for kw in (dict(binWidth=25), dict(binWidth=3.5), dict(binWidth=0.1), dict(binWidth=5000), dict(binWidth=7),
                       dict(binCount=8), dict(binCount=64), dict(binCount=1)):
                if np.issubdtype(dt, np.integer) and kw.get("binWidth") == 0.1 and scale == 4000:
                    continue                                       # (tens of thousands of edges: nothing new)
                with np.errstate(over="ignore"):                   # int16 + 2 * 5000 wraps in NumPy scalar arithmetic -- in both
                    ref = PL.bin_edges(v, kw.get("binWidth", 25), kw.get("binCount"))
                    got = IO._edges_from_minmax(v.min(), v.max(), dt, **kw)
                assert np.asarray(got).shape == np.asarray(ref).shape, (dt, kw, v.min(), v.max())
                assert np.array_equal(np.asarray(got, np.float64), np.asarray(ref, np.float64)), (dt, kw, v.min(), v.max())
                # ... and digitizing with them gives the reference's levels
                assert np.array_equal(np.digitize(v, np.asarray(got, np.float64)), np.digitize(v, ref))
                n += 1
    assert n > 3500


# ---- cmatrices: argument errors are raised on the host, before anything touches the device, with the reference's exception
# types (SURVEY.md 8b "Error conventions") -- the types the compiled reference extension raises for the same calls
# (tests/golden/reference_runs.json, make_golden.py --reference-runs-only)
BAD_CALLS = {
    "ndim mismatch": lambda cm, i, m: cm.calculate_glcm(i, m[0], np.array([1]), 8, False, -1),
    "shape mismatch": lambda cm, i, m: cm.calculate_glcm(i, m[:, :4], np.array([1]), 8, False, -1),
    "voxels without kernelRadius": lambda cm, i, m: cm.calculate_glcm(i, m, np.array([1]), 8, False, -1, 0, np.zeros((3, 2), np.int32)),
    "voxels with the wrong first dimension": lambda cm, i, m: cm.calculate_glrlm(i, m, 8, 6, False, -1, 1, np.zeros((2, 4), np.int32)),
    "voxels 1-D": lambda cm, i, m: cm.calculate_ngtdm(i, m, np.array([1]), 8, False, -1, 1, np.zeros(3, np.int32)),
    "distances 2-D": lambda cm, i, m: cm.calculate_gldm(i, m, np.ones((2, 2), np.int32), 8, 0, False, -1),
    "size 2-D": lambda cm, i, m: cm.generate_angles(np.ones((2, 3), np.int32), np.array([1]), 0, False, -1),
    "no angle": lambda cm, i, m: cm.generate_angles(np.array([5, 5, 5], np.int32), np.array([9]), 0, False, -1),
}


@pytest.mark.parametrize("what", list(BAD_CALLS))
def test_cmatrices_argument_errors_have_the_reference_exception_types(what):
    want = json.load(open(os.path.join(GOLDEN, "reference_runs.json")))["argument_errors"][what]
    img = np.ones((4, 5, 6), np.int32)
    msk = np.ones((4, 5, 6), bool)
    with pytest.raises(Exception) as got:
        BAD_CALLS[what](cmatrices, img, msk)
    assert type(got.value).__name__ == want, (what, repr(got.value), want)
    assert type(got.value) in (ValueError, RuntimeError)


def test_plugin_voxel_settings_of_a_2d_image_describe_one_plane(oracle_device):
    """a 2-D image runs through the 3-D kernels as a single plane: spacing gets a leading 1, a force2D dimension moves up by
    one axis (featureclasses._voxel_settings) -- the settings the emulated kernel reproduces the reference's 2-D maps with
    (tests/test_host_emul.py, golden voxelx_image2d)"""
    z = np.load(os.path.join(GOLDEN, "voxelx_image2d.npz"))
    sp = tuple(float(v) for v in z["spacing"])
    obj = FC.RadiomicsGLCM(I.ArrayImage(z["image"], sp), I.ArrayImage(z["mask"].astype(np.uint8), sp), voxelBased=True, binWidth=1)
    s = obj._voxel_settings()
    assert (s.kernelRadius, s.force2D, s.ndist, s.distances[0], s.symmetricalGLCM) == (1, 0, 1, 1, 1)
    assert tuple(s.spacing_zyx) == (1.0, sp[1], sp[0])
    assert s.Ng == int(obj.coefficients["Ng"]) and s.n_roi_levels == len(obj.coefficients["grayLevels"])
    obj2 = FC.RadiomicsGLRLM(I.ArrayImage(z["image"], sp), I.ArrayImage(z["mask"].astype(np.uint8), sp), voxelBased=True, binWidth=1,
                             force2D=True, force2Ddimension=1, weightingNorm="euclidean", kernelRadius=2, initValue=-1.0)
    s2 = obj2._voxel_settings()
    assert (s2.force2D, s2.force2Ddimension, s2.kernelRadius, s2.initValue) == (1, 2, 2, -1.0)
    assert obj.masked is True and obj2.voxelBased is True
