"""GPU tests of the plugin layer: gray-level discretisation (bit-identical to NumPy), the feature
classes against the reference's baseline CSV values / golden matrices / voxel maps, and the
wavelet + LoG kernels against their numpy restatements and mathematical properties."""
import json
import os

import numpy as np
import pytest
import torch

import filters_np as FN
import pipeline as PL
from helpers import (GOLDEN, assert_maps_close, check_segment_baseline_columns, check_segment_variant_runs, ref_map,
                     voxel_goldens)
from pyradiomics_b200 import featureclasses as FC, image as I, imageoperations as IO

pytestmark = pytest.mark.gpu
CASES = ["brain1", "brain2", "breast1", "lung1", "lung2"]


@pytest.fixture(scope="module")
def seg():
    return np.load(os.path.join(GOLDEN, "segment_cases.npz")), json.load(open(os.path.join(GOLDEN, "segment_expect.json")))


# ------------------------------------------------------------------------------ discretisation
@pytest.mark.parametrize("kw", [dict(binWidth=25), dict(binWidth=3.5), dict(binCount=64), dict(binWidth=5000)])
@pytest.mark.parametrize("dtype", ["int16", "float64", "float32"])
def test_binning_is_bit_identical_to_numpy(kw, dtype):
    rng = np.random.default_rng(4)
    img = (rng.normal(300, 180, (9, 20, 21))).astype(dtype)
    if dtype == "int16":
        img[0, 0, :4] = [75, 100, 125, -25]            # values exactly on bin edges
    msk = rng.random(img.shape) > 0.3
    got, edges = IO.binImage(img, msk, **kw)
    ref, redges, _, _ = PL.bin_image(img, msk, kw.get("binWidth", 25), kw.get("binCount"))
    assert np.array_equal(np.asarray(edges, float), np.asarray(redges, float))
    assert np.array_equal(got, ref)
    assert np.array_equal(IO.getBinEdges(img[msk], **kw), redges)


def test_binning_flat_region():
    img = np.full((4, 5, 6), 50, np.int16)
    got, edges = IO.binImage(img, np.ones(img.shape, bool), binWidth=25)
    assert list(edges) == [50, 75, 100] or len(edges) >= 2
    assert (got == 1).all()


# ------------------------------------------------------------------------------ feature classes
@pytest.mark.parametrize("cname", list(FC.FEATURE_CLASSES))
def test_segment_features_match_reference_baseline(seg, cname):
    """reference tests/test_features.py: every baseline column whose settings touch only the hot path"""
    cases, expect = seg
    for test, e in expect[cname].items():
        c = e["case"]
        img = I.ArrayImage(cases[c + "_image"], cases[c + "_spacing"])
        msk = I.ArrayImage(cases[c + "_mask"].astype(np.uint8), cases[c + "_spacing"])
        obj = FC.FEATURE_CLASSES[cname](img, msk, **e["settings"])
        got = obj.execute()
        assert set(got) == set(e["features"]), (set(got) ^ set(e["features"]))
        for f, v in e["features"].items():
            assert abs(float(got[f]) - v) <= 1e-7 * max(abs(v), 1e-12), (cname, test, f, float(got[f]), v)


@pytest.mark.parametrize("case", CASES)
def test_processed_matrices_match_reference_golden(seg, case):
    """reference tests/test_matrices.py:35-65: P_<class> after _initCalculation()"""
    cases, _ = seg
    img = I.ArrayImage(cases[case + "_image"], cases[case + "_spacing"])
    msk = I.ArrayImage(cases[case + "_mask"].astype(np.uint8), cases[case + "_spacing"])
    for cname, cls in FC.FEATURE_CLASSES.items():
        obj = cls(img, msk, binWidth=25)
        obj._initCalculation()
        P = getattr(obj, "P_" + cname)[0]
        assert np.abs(P - cases[f"{case}_{cname}_P"]).max() < 1e-3


@pytest.mark.parametrize("cname", list(FC.FEATURE_CLASSES))
def test_segment_features_match_every_baseline_column(cname):
    """the 160 baseline columns without resampling (resegmented masks, normalisation included) over the CUDA matrices, at
    1e-9: the host logic is pinned on the oracle's matrices (test_plugin_host_logic_cpu.py), so a failure here is the kernels'"""
    check_segment_baseline_columns(cname)


@pytest.mark.parametrize("cname", list(FC.FEATURE_CLASSES))
def test_segment_features_match_reference_runs_of_other_settings(cname):
    """weighting norms, several distances, asymmetric GLCM, force2D, binCount, gldm_a over the CUDA matrices, at 1e-9"""
    check_segment_variant_runs(cname)


@pytest.mark.parametrize("name,z,kw", voxel_goldens(extra=True), ids=[g[0] for g in voxel_goldens(extra=True)])
def test_voxel_based_plugin_maps_match_reference(name, z, kw):
    sp = z["spacing"]
    img = I.ArrayImage(z["image"], sp)
    msk = I.ArrayImage(z["mask"].astype(np.uint8), sp)
    for cname, cls in FC.FEATURE_CLASSES.items():
        got = cls(img, msk, voxelBased=True, **kw).execute()
        for f, im in got.items():
            assert_maps_close(I.as_array(im), ref_map(z, cname, f), f"{name}/{cname}/{f}")


def test_unmasked_kernel_and_feature_selection():
    rng = np.random.default_rng(2)
    img = rng.integers(0, 200, (6, 7, 8)).astype(np.int16)
    msk = np.zeros(img.shape, np.uint8)
    msk[2:5, 2:6, 1:7] = 1
    obj = FC.RadiomicsGLDM(img, msk, voxelBased=True, maskedKernel=False, binWidth=25, initValue=-1)
    obj.enableFeatureByName("DependenceEntropy")
    got = obj.execute()
    assert list(got) == ["DependenceEntropy"]
    m = I.as_array(got["DependenceEntropy"])
    assert (m[msk == 0] == -1).all()
    ref = PL.extract("gldm", img, msk.astype(bool), voxelBased=True, binWidth=25, maskedKernel=False)
    assert np.allclose(m[msk == 1], ref["DependenceEntropy"], rtol=1e-9)
    with pytest.raises(LookupError):
        obj.enableFeatureByName("NoSuchFeature")


def test_every_feature_has_a_docstring():
    """reference tests/test_docstrings.py"""
    for cls in FC.FEATURE_CLASSES.values():
        for name in cls.getFeatureNames():
            assert getattr(cls, f"get{name}FeatureValue").__doc__


# ------------------------------------------------------------------------------ wavelet
@pytest.mark.parametrize("shape", [(8, 10, 12), (7, 9, 12), (5, 6)])
def test_wavelet_matches_restatement_and_is_an_isometry(shape):
    rng = np.random.default_rng(1)
    x = rng.normal(size=shape)
    lo, hi = IO.wavelet_filters("coif1")
    assert abs(lo.sum() - np.sqrt(2)) < 1e-12 and abs((lo ** 2).sum() - 1) < 1e-12 and abs(hi.sum()) < 1e-12
    got = {n: I.as_array(im) for im, n, _ in IO.getWaveletImage(I.ArrayImage(x), None)}
    nd = len(shape)
    ref = FN.swtn_level1(x, lo, hi, tuple(range(nd - 1, -1, -1)))
    assert len(got) == 2 ** nd
    for key, arr in ref.items():
        name = "wavelet-" + key.replace("a", "L").replace("d", "H")
        assert np.allclose(got[name], arr, rtol=1e-12, atol=1e-12), name
    if all(s % 2 == 0 for s in shape):
        # undecimated transform with these sqrt(2)-normalised filters: sum of band energies = 2^nd * |x|^2
        e = sum((v ** 2).sum() for v in got.values())
        assert abs(e - 2 ** nd * (x ** 2).sum()) < 1e-9 * e
    const = {n: I.as_array(im) for im, n, _ in IO.getWaveletImage(I.ArrayImage(np.full(shape, 3.0)), None)}
    for n, v in const.items():
        target = 3.0 * np.sqrt(2) ** nd if n == "wavelet-" + "L" * nd else 0.0
        assert np.allclose(v, target, atol=1e-12)


# ------------------------------------------------------------------------------ LoG
def test_log_matches_restatement_and_analytic_gaussian_laplace():
    import scipy.ndimage as ndi
    rng = np.random.default_rng(3)
    x = ndi.gaussian_filter(rng.normal(size=(40, 44, 48)), 2.0) * 100
    sp = (1.0, 1.0, 1.0)
    for sigma in (1.0, 2.0, 3.0):
        out = [I.as_array(im) for im, n, _ in IO.getLoGImage(I.ArrayImage(x.astype(np.float32), sp), None, sigma=[sigma])][0]
        assert out.dtype == np.float32
        # restatement (float64 recursion of the same coefficients)
        ref = np.zeros(x.shape)
        xf = x.astype(np.float32).astype(np.float64)
        for d in range(3):
            cur = xf
            for e in range(3):
                if e != d:
                    cur = FN.recursive_gaussian_axis(cur, IO.recursive_gaussian_coefficients(sigma, 0), e).astype(np.float32).astype(np.float64)
            ref += (FN.recursive_gaussian_axis(cur, IO.recursive_gaussian_coefficients(sigma, 2), d) * sigma ** 2).astype(np.float32)
        assert np.allclose(out, ref, rtol=2e-4, atol=2e-4 * np.abs(ref).max())
        # analytic sigma^2-normalised Gaussian Laplacian (truncated FIR), interior only
        ana = ndi.gaussian_laplace(x, sigma, mode="nearest", truncate=6.0) * sigma ** 2
        c = slice(12, -12)
        err = np.abs(out[c, c, c] - ana[c, c, c]).max() / np.abs(ana[c, c, c]).max()
        assert err < 0.03, (sigma, err)


def test_log_size_guards():
    assert list(IO.getLoGImage(I.ArrayImage(np.zeros((3, 8, 8))), None, sigma=[1.0])) == []
    names = [n for _, n, _ in IO.getLoGImage(I.ArrayImage(np.zeros((8, 8, 8), np.float32)), None, sigma=[1.5, -1])]
    assert names == ["log-sigma-1-5-mm-3D"]


# ------------------------------------------------------------------------------ pipelines
def test_filter_pipeline_equals_per_image_plugins():
    """config-4 shape: original + 8 wavelet bands + LoG sigmas, each binned then run through the
    fused kernels on the device == doing the same image by image through the plugin classes."""
    from pyradiomics_b200 import pipeline as PP
    rng = np.random.default_rng(9)
    import scipy.ndimage as ndi
    x = (ndi.gaussian_filter(rng.normal(size=(12, 14, 16)), 1.5) * 400 + 300).astype(np.float32)
    m = np.ones(x.shape, np.uint8)
    got = {}
    info = PP.voxel_suite_with_filters(torch.as_tensor(x).cuda(), torch.as_tensor(m).cuda(), classes=("gldm", "glrlm"),
                                       sigmas=(1.0,), binWidth=25,
                                       consume=lambda n, c, t: got.__setitem__((n, c), t.cpu().numpy().copy()))
    assert len(info) == 1 + 8 + 1
    names = [n for n, _, _ in info]
    assert names[0] == "original" and "wavelet-HHH" in names and "wavelet-LLL" in names and names[-1] == "log-sigma-1-0-mm-3D"
    imgs = {"original": I.ArrayImage(x)}
    for im, n, _ in IO.getWaveletImage(I.ArrayImage(x), None):
        imgs[n] = im
    for im, n, _ in IO.getLoGImage(I.ArrayImage(x), None, sigma=[1.0]):
        imgs[n] = im
    for n in names:
        for c in ("gldm", "glrlm"):
            ref = FC.FEATURE_CLASSES[c](imgs[n], I.ArrayImage(m), voxelBased=True, binWidth=25).execute()
            from pyradiomics_b200 import _lib as L
            for k, f in enumerate(L.feature_names(c)):
                assert np.allclose(got[(n, c)][k], I.as_array(ref[f]), rtol=1e-9, atol=1e-11, equal_nan=True), (n, c, f)


def test_segment_batch_shards_cases(seg):
    from pyradiomics_b200 import pipeline as PP
    cases, expect = seg
    cs = [(cases[c + "_image"], cases[c + "_mask"].astype(np.uint8)) for c in CASES]
    r0 = PP.segment_batch(cs, classes=("ngtdm",), rank=0, world=2, binWidth=25)
    r1 = PP.segment_batch(cs, classes=("ngtdm",), rank=1, world=2, binWidth=25)
    assert sorted(r0) == [0, 2, 4] and sorted(r1) == [1, 3]
    for k, c in enumerate(CASES):
        got = (r0 if k % 2 == 0 else r1)[k]["ngtdm"]
        for f, v in expect["ngtdm"][c]["features"].items():
            assert abs(got[f] - v) <= 1e-7 * abs(v)


# ------------------------------------------------------------------------------ first-order (next row)
def test_firstorder_segment_matches_reference_baseline(seg):
    cases, _ = seg
    exp = json.load(open(os.path.join(GOLDEN, "segment_expect_firstorder.json")))
    for test, e in exp.items():
        c = e["case"]
        obj = FC.RadiomicsFirstOrder(I.ArrayImage(cases[c + "_image"], cases[c + "_spacing"]),
                                     I.ArrayImage(cases[c + "_mask"].astype(np.uint8), cases[c + "_spacing"]), **e["settings"])
        got = obj.execute()
        assert set(got) == set(e["features"])
        for f, v in e["features"].items():
            assert abs(float(got[f]) - v) <= 1e-9 * max(abs(v), 1e-12), (test, f, float(got[f]), v)


@pytest.mark.parametrize("name,r", [("r1", 1), ("r2", 2)])
def test_firstorder_voxel_maps(name, r):
    """16 features against the reference's own voxel-mode run; all 18 against the oracle (Entropy /
    Uniformity of the reference use a shifted window -- firstorder.py:109 -- and are not goldens)"""
    import firstorder_np as FO
    z = np.load(os.path.join(GOLDEN, "voxel_firstorder.npz"))
    m = z[name + "_mask"]
    got = FC.RadiomicsFirstOrder(I.ArrayImage(z["image"], z["spacing"]), I.ArrayImage(m.astype(np.uint8), z["spacing"]),
                                 voxelBased=True, kernelRadius=r, binWidth=25, voxelArrayShift=100).execute()
    ref = FO.extract(z["image"], m, voxelBased=True, spacing_xyz=z["spacing"], kernelRadius=r, binWidth=25, voxelArrayShift=100)
    assert list(got) == FO.NAMES
    for f in FO.NAMES:
        arr = I.as_array(got[f])
        assert np.allclose(arr[m], ref[f], rtol=1e-9, atol=1e-9), f
        assert (arr[~m] == 0).all()
        if f not in ("Entropy", "Uniformity"):
            assert np.allclose(arr[m], z[f"{name}_{f}"][m], rtol=1e-5, atol=1e-8), f


# ------------------------------------------------------------------------------ voxel driver / output assembly (round 2)
def _raw_case(shape=(20, 22, 23), seed=3):
    rng = np.random.default_rng(seed)
    lev = rng.integers(1, 33, shape)
    raw = ((lev - 1) * 25 + 3).astype(np.int16)
    msk = (rng.random(shape) < 0.85).astype(np.uint8)
    return raw, msk


def test_plugin_voxel_path_copies_only_enabled_maps_and_matches_full_run():
    raw, msk = _raw_case()
    full = FC.RadiomicsGLCM(raw, msk, voxelBased=True, binWidth=25).execute()
    obj = FC.RadiomicsGLCM(raw, msk, voxelBased=True, binWidth=25)
    obj.enableFeatureByName("MCC")
    obj.enableFeatureByName("Contrast")
    obj.enableFeatureByName("SumSquares")
    part = obj.execute()
    assert sorted(part) == ["Contrast", "MCC", "SumSquares"]
    for k, v in part.items():
        assert np.array_equal(v.array, full[k].array, equal_nan=True)
    # the three maps are views of ONE page-locked block of exactly three maps
    base = part["MCC"].array.base
    assert base is not None and base.shape[0] == 3


def test_plugin_shares_one_discretisation_between_the_classes():
    raw, msk = _raw_case(seed=4)
    FC.clear_device_cache()
    objs = [FC.FEATURE_CLASSES[c](raw, msk, voxelBased=True, binWidth=25) for c in FC.FEATURE_CLASSES]
    assert len({id(o._device) for o in objs}) == 1                  # binned once, shared (base.py:119-125 runs it 5x)
    raw2 = raw.copy()
    raw2[3, 4, 5] += 400                                            # an edited image must not hit the cache
    assert FC.RadiomicsGLCM(raw2, msk, voxelBased=True, binWidth=25)._device is not objs[0]._device
    # the lazily downloaded discretised array equals the reference's binImage
    ref, _, levels, Ng = PL.bin_image(raw, msk.astype(bool), 25)
    assert np.array_equal(objs[0].imageArray, ref) and objs[0].coefficients["Ng"] == Ng
    assert np.array_equal(objs[0].coefficients["grayLevels"], levels)


@pytest.mark.parametrize("cname", ["glcm", "ngtdm"])
def test_plugin_zrange_and_float32_maps(cname):
    raw, msk = _raw_case(seed=5)
    cls = FC.FEATURE_CLASSES[cname]
    full = cls(raw, msk, voxelBased=True, binWidth=25, b200_zchunk=7).execute()
    slab = cls(raw, msk, voxelBased=True, binWidth=25, b200_zrange=(6, 15), b200_zchunk=4).execute()
    f32 = cls(raw, msk, voxelBased=True, binWidth=25, b200_map_dtype="float32", b200_zchunk=5).execute()
    for k in full:
        a = full[k].array
        assert slab[k].array.shape == (9,) + raw.shape[1:]
        assert np.array_equal(slab[k].array, a[6:15], equal_nan=True)       # same bits as the whole-volume run
        assert f32[k].array.dtype == np.float32
        assert np.array_equal(f32[k].array, a.astype(np.float32), equal_nan=True)


def test_plugin_progress_reporter_and_logger_names():
    import logging
    raw, msk = _raw_case(seed=6)
    seen = []

    class Rep:
        def __init__(self, iterable=None, desc="", total=None):
            seen.append(("init", total))

        def __enter__(self):
            return self

        def __exit__(self, *a):
            seen.append(("exit",))

        def update(self, n=1):
            seen.append(("update", n))

    FC.setProgressReporter(Rep)
    lg = logging.getLogger("radiomics")
    old = lg.level
    lg.setLevel(logging.INFO)
    try:
        obj = FC.RadiomicsGLDM(raw, msk, voxelBased=True, binWidth=25, b200_zchunk=8)
        assert obj.logger.name == "radiomics.gldm"                   # reference base.py:61: the class's module logger
        obj.execute()
    finally:
        FC.setProgressReporter(None)
        lg.setLevel(old)
    assert seen[0] == ("init", raw.shape[0]) and seen[-1] == ("exit",)
    assert sum(s[1] for s in seen if s[0] == "update") == raw.shape[0]


def test_host_extractor_float32_and_float64_agree():
    from pyradiomics_b200 import voxel
    rng = np.random.default_rng(8)
    lev = rng.integers(1, 33, (18, 19, 20)).astype(np.int32)
    msk = np.ones(lev.shape, np.uint8)
    a = voxel.HostExtractor(lev.shape, zchunk=5).run(lev, msk, 32, 32)
    a = {c: t.clone() for c, t in a.items()}
    b = voxel.HostExtractor(lev.shape, zchunk=7, out_dtype=torch.float32).run(lev, msk, 32, 32)
    for c in a:
        assert torch.equal(a[c].to(torch.float32), b[c]) or torch.allclose(a[c].to(torch.float32), b[c], equal_nan=True, rtol=0, atol=0)


# ------------------------------------------------------------------------------ wavelet: phase, levels, odd sizes (round 2)
@pytest.mark.parametrize("shape", [(12, 10, 16), (9, 11, 13)])
def test_wavelet_impulse_response_is_the_filter_taps_at_the_documented_phase(shape):
    """out[n] = sum_j h[j] x[(n + F/2 - j) mod N]  =>  an impulse at p puts tap h[j] at p - F/2 + j (periodic), separably
    for all 8 bands; first band letter <-> x (the LAST numpy axis: the reference passes axes = (2,1,0))"""
    lo, hi = IO.wavelet_filters("coif1")
    F = lo.size
    p = (4, 5, 6)
    x = np.zeros(shape)
    x[p] = 1.0
    got = {n: I.as_array(im) for im, n, _ in IO.getWaveletImage(I.ArrayImage(x), None)}
    pads = [s + (s % 2) for s in shape]

    def line(h, n_axis, n_pad, pos):
        v = np.zeros(n_pad)
        for j in range(F):
            v[(pos - F // 2 + j) % n_pad] += h[j]
        return v[:n_axis]

    for name, arr in got.items():
        letters = name.split("-")[1]                       # x, y, z
        fx, fy, fz = [(hi if c == "H" else lo) for c in letters]
        ref = np.einsum("i,j,k->ijk", line(fz, shape[0], pads[0], p[0]), line(fy, shape[1], pads[1], p[1]),
                        line(fx, shape[2], pads[2], p[2]))
        assert np.allclose(arr, ref, rtol=0, atol=1e-15), name


@pytest.mark.parametrize("shape,kw", [((9, 11, 13), dict(level=2)), ((8, 9, 10), dict(level=2, start_level=1)),
                                      ((10, 12, 14), dict(level=3)), ((7, 9), dict(level=2))])
def test_wavelet_levels_keep_the_padded_approximation_like_the_reference(shape, kw):
    """_swt3 pads ONCE and feeds the padded approximation to the next level (imageoperations.py:917-937): for odd sizes
    level >= 2 differs from re-wrapping a cropped approximation (round 1 did the latter)"""
    rng = np.random.default_rng(2)
    x = rng.normal(size=shape)
    lo, hi = IO.wavelet_filters("coif1")
    nd = len(shape)
    axes = tuple(range(nd - 1, -1, -1))
    approx, levels = FN.swt3_levels(x, lo, hi, axes, kw.get("level", 1), kw.get("start_level", 0))
    got = {n: I.as_array(im) for im, n, _ in IO.getWaveletImage(I.ArrayImage(x), None, **kw)}
    assert len(got) == len(levels) * (2 ** nd - 1) + 1
    for idx, dec in enumerate(levels, start=1):
        for key, arr in dec.items():
            band = key.replace("a", "L").replace("d", "H")
            name = f"wavelet-{band}" if idx == 1 else f"wavelet{idx}-{band}"
            assert np.allclose(got[name], arr, rtol=1e-12, atol=1e-12), name
    last = f"wavelet-{'L' * nd}" if len(levels) == 1 else f"wavelet{len(levels)}-{'L' * nd}"
    assert np.allclose(got[last], approx, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("wavelet", ["haar", "db2", "coif1"])
def test_fused_3d_wavelet_kernel_equals_axis_by_axis_kernel(wavelet):
    lo, hi = IO.wavelet_filters(wavelet)
    x = torch.randn((20, 37, 70), dtype=torch.float64, device="cuda")           # tiles with ragged edges in y and x
    fused = IO.swt_level1_device(x, (2, 1, 0), lo, hi)
    cur = {"": x}
    for ax in (2, 1, 0):
        nxt = {}
        for k, t in cur.items():
            a, d = torch.empty_like(t), torch.empty_like(t)
            import ctypes as C
            from pyradiomics_b200._lib import check, lib
            check(lib().rb_swt_axis_dev(C.c_void_p(t.data_ptr()), 20, 37, 70, ax, lo.ctypes.data_as(C.c_void_p),
                                        hi.ctypes.data_as(C.c_void_p), int(lo.size), C.c_void_p(a.data_ptr()), C.c_void_p(d.data_ptr()),
                                        None), "swt")
            nxt[k + "a"], nxt[k + "d"] = a, d
        cur = nxt
    # (37 is odd: the axis kernel wrap-pads by index mapping, the fused kernel is purely periodic -> compare on an even copy too)
    xe = x[:, :36].contiguous()
    fe = IO.swt_level1_device(xe, (2, 1, 0), lo, hi)
    ref = FN.swtn_level1(xe.cpu().numpy(), lo, hi, (2, 1, 0))
    for k in ref:
        assert np.allclose(fe[k].cpu().numpy(), ref[k], rtol=1e-12, atol=1e-12), k
    assert set(fused) == set(cur)


def test_log_x_axis_tiles_match_restatement_on_ragged_sizes():
    """the shared-memory-transposed x pass: line counts and lengths that are not multiples of 32"""
    rng = np.random.default_rng(5)
    x = rng.normal(size=(5, 7, 45)).astype(np.float32) * 50
    out = [I.as_array(im) for im, n, _ in IO.getLoGImage(I.ArrayImage(x, (1.0, 1.0, 1.0)), None, sigma=[1.5])][0]
    ref = np.zeros(x.shape)
    xf = x.astype(np.float64)
    for d in range(3):
        cur = xf
        for e in range(3):
            if e != d:
                cur = FN.recursive_gaussian_axis(cur, IO.recursive_gaussian_coefficients(1.5, 0), e).astype(np.float32).astype(np.float64)
        ref += (FN.recursive_gaussian_axis(cur, IO.recursive_gaussian_coefficients(1.5, 2), d) * 1.5 ** 2).astype(np.float32)
    assert np.allclose(out, ref, rtol=2e-4, atol=2e-4 * np.abs(ref).max())


@pytest.mark.gpu
def test_staged_upload_of_large_host_arrays_is_exact():
    """imageoperations._to_device stages big pageable arrays through page-locked blocks with copy threads"""
    from pyradiomics_b200 import imageoperations as IO
    rng = np.random.default_rng(3)
    for dt, shape in ((np.int16, (97, 613, 611)), (np.uint8, (70 * (1 << 20) + 13,)), (np.float64, (9, 1031, 1033))):
        a = rng.integers(0, 200, shape).astype(dt)
        assert a.nbytes >= IO._STAGE_MIN
        t = IO._to_device(a)
        assert tuple(t.shape) == a.shape
        np.testing.assert_array_equal(t.cpu().numpy(), a)
    b = rng.random((64, 64, 64))                        # small arrays take the plain path
    np.testing.assert_array_equal(IO._to_device(b).cpu().numpy(), b)
