"""CPU tests of the ORACLE itself (no GPU): the C port against the compiled reference, against the
reference's golden matrices / feature CSV columns, and against the reference's voxel-mode runs."""
import json
import os

import numpy as np
import pytest

import cmatrices_oracle as O
import pipeline as PL
from helpers import GOLDEN, assert_maps_close, digest, port_trial_outputs, port_trials, ref_map, voxel_goldens

CASES = ["brain1", "brain2", "breast1", "lung1", "lung2"]


@pytest.fixture(scope="module")
def seg():
    return np.load(os.path.join(GOLDEN, "segment_cases.npz")), json.load(open(os.path.join(GOLDEN, "segment_expect.json")))


def test_port_equals_compiled_reference():
    """bit-exact agreement of oracle/cmatrices_port.c with the gcc-built reference _cmatrices on
    random 2-D/3-D inputs, segment and voxel mode, several distances / force2D: every matrix and angle table
    against the digest of the reference's (tests/golden/reference_runs.json)."""
    ref = json.load(open(os.path.join(GOLDEN, "reference_runs.json")))["port_trials"]
    n = 0
    for trial, *args in port_trials():
        if ref[trial] is None:                       # empty ROI, or angles the reference refuses
            continue
        got = [digest(a) for a in port_trial_outputs(O, *args)]
        assert len(got) == len(ref[trial])
        for k, (g, r) in enumerate(zip(got, ref[trial])):
            assert g == r, (trial, k)
        n += len(got) == 12
    assert n > 20


def _processed(cname, img, msk, levels, Ng):
    """P_<class> as the reference feature classes expose it (what data/baseline/*.npy hold)."""
    import features_np as F
    if cname == "glcm":
        P, _ = O.calculate_glcm(img, msk, np.array([1]), Ng, False, 0)
        return F.glcm_matrix(P, levels)[0]
    if cname == "glrlm":
        P, _ = O.calculate_glrlm(img, msk, Ng, max(img.shape), False, 0)
        P = P[0, levels - 1]
        return P[:, P.sum((0, 2)) != 0]
    if cname == "glszm":
        P = O.calculate_glszm(img, msk, Ng, int(msk.sum()), False, 0)[0, levels - 1]
        return P[:, P.sum(0) != 0]
    if cname == "gldm":
        P = O.calculate_gldm(img, msk, np.array([1]), Ng, 0, False, 0)[0, levels - 1]
        return P[:, P.sum(0) != 0]
    P = O.calculate_ngtdm(img, msk, np.array([1]), Ng, False, 0)[0]
    return P[P[:, 0] != 0]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("cname", PL.CLASS_NAMES)
def test_port_reproduces_reference_golden_matrices(seg, case, cname):
    """reference tests/test_matrices.py:35-65 against data/baseline/<case>_<class>.npy"""
    cases, _ = seg
    img, levels_edges, levels, Ng = PL.bin_image(cases[f"{case}_image"], cases[f"{case}_mask"], 25)
    got = _processed(cname, img, cases[f"{case}_mask"], levels, Ng)
    ref = cases[f"{case}_{cname}_P"]
    assert got.shape == ref.shape
    if cname == "glcm":
        assert np.abs(got - ref).max() < 1e-12
    elif cname == "ngtdm":
        assert np.array_equal(got[:, [0, 2]], ref[:, [0, 2]]) and np.allclose(got[:, 1], ref[:, 1], rtol=1e-12)
    else:
        assert np.array_equal(got, ref)


@pytest.mark.parametrize("cname", PL.CLASS_NAMES)
def test_pipeline_reproduces_reference_feature_baseline(seg, cname):
    """reference tests/test_features.py against data/baseline/baseline_<class>.csv (columns whose
    settings only touch the hot path)."""
    cases, expect = seg
    for test, e in expect[cname].items():
        c = e["case"]
        got = PL.extract(cname, cases[c + "_image"], cases[c + "_mask"], spacing_zyx=cases[c + "_spacing"][::-1], **e["settings"])
        for f, v in e["features"].items():
            assert abs(got[f] - v) <= 1e-9 * max(abs(v), 1e-12), (cname, test, f, got[f], v)


@pytest.mark.parametrize("cname", PL.CLASS_NAMES)
def test_pipeline_reproduces_reference_runs_of_settings_the_baselines_do_not_cover(seg, cname):
    """weighting norms, several distances, asymmetric GLCM, force2D, binCount, gldm_a in SEGMENT mode: runs of the reference's
    classes on three bundled cases (tests/golden/segment_expect_variants.json, make_golden.py --segment-variants-only)"""
    cases, _ = seg
    expect = json.load(open(os.path.join(GOLDEN, "segment_expect_variants.json")))[cname]
    assert len(expect) >= 9
    for test, e in expect.items():
        c = e["case"]
        got = PL.extract(cname, cases[c + "_image"], cases[c + "_mask"], spacing_zyx=cases[c + "_spacing"][::-1], **e["settings"])
        for f, v in e["features"].items():
            assert np.isclose(got[f], v, rtol=1e-9, atol=1e-12, equal_nan=True), (cname, test, e["settings"], f, got[f], v)


@pytest.mark.parametrize("cname", PL.CLASS_NAMES)
def test_pipeline_reproduces_the_resegmented_baseline_columns(seg, cname):
    """`<case>_flatRegion` (one gray level: the single-edge branch of getBinEdges, every class on a flat ROI),
    `<case>_resegmentation` (masks resegmented by the reference's own resegmentMask) and `<case>_normalization` (float image,
    binWidth 5) columns (tests/golden/make_golden.py --segment-extra-only): with these and the resampling columns
    (test_resample_cpu.py) the oracle reproduces EVERY column of the five texture baseline CSVs (185)"""
    cases, _ = seg
    masks = np.load(os.path.join(GOLDEN, "segment_extra.npz"))
    expect = json.load(open(os.path.join(GOLDEN, "segment_expect_extra.json")))
    assert len(expect[cname]) == 15
    for test, e in expect[cname].items():
        c = e["case"]
        img, m = cases[c + "_image"], (masks[test + "_mask"] if test + "_mask" in masks.files else cases[c + "_mask"])
        if "normalize" in e:                 # `<case>_normalization`: (x - mean) / std of the WHOLE image, times normalizeScale
            n = e["normalize"]
            img = (img.astype(np.float64) - n["mean"]) / n["std"] * n["scale"]
        got = PL.extract(cname, img, m, spacing_zyx=cases[c + "_spacing"][::-1], **e["settings"])
        for f, v in e["features"].items():
            assert abs(got[f] - v) <= 1e-9 * max(abs(v), 1e-12), (cname, test, f, got[f], v)


@pytest.mark.parametrize("name,z,kw", voxel_goldens(extra=True), ids=[g[0] for g in voxel_goldens(extra=True)])
def test_pipeline_reproduces_reference_voxel_maps(name, z, kw):
    m = z["mask"]
    for cname in PL.CLASS_NAMES:
        got = PL.extract(cname, z["image"], m, voxelBased=True, spacing_zyx=z["spacing"][::-1], **kw)
        for f, arr in got.items():
            assert_maps_close(arr, ref_map(z, cname, f)[m], f"{name}/{cname}/{f}", rtol=1e-8, atol=1e-10)


def test_firstorder_oracle_reproduces_the_resegmented_and_normalised_columns(seg):
    """`<case>_resegmentation` / `<case>_normalization` of baseline_firstorder.csv (with the base and the resampling columns:
    all 20)"""
    import firstorder_np as FO
    cases, _ = seg
    masks = np.load(os.path.join(GOLDEN, "segment_extra.npz"))
    expect = json.load(open(os.path.join(GOLDEN, "segment_expect_extra.json")))["firstorder"]
    assert len(expect) == 10
    for test, e in expect.items():
        c = e["case"]
        img, m = cases[c + "_image"], (masks[test + "_mask"] if test + "_mask" in masks.files else cases[c + "_mask"])
        if "normalize" in e:
            n = e["normalize"]
            img = (img.astype(np.float64) - n["mean"]) / n["std"] * n["scale"]
        got = FO.extract(img, m, spacing_xyz=cases[c + "_spacing"], **e["settings"])
        for f, v in e["features"].items():
            assert abs(got[f] - v) <= 1e-9 * max(abs(v), 1e-12), (test, f, got[f], v)


def test_firstorder_oracle_reproduces_reference():
    """oracle/firstorder_np.py against data/baseline/baseline_firstorder.csv and the reference's voxel run"""
    import firstorder_np as FO
    cases = np.load(os.path.join(GOLDEN, "segment_cases.npz"))
    exp = json.load(open(os.path.join(GOLDEN, "segment_expect_firstorder.json")))
    for test, e in exp.items():
        c = e["case"]
        got = FO.extract(cases[c + "_image"], cases[c + "_mask"], spacing_xyz=cases[c + "_spacing"], **e["settings"])
        for f, v in e["features"].items():
            assert abs(got[f] - v) <= 1e-10 * max(abs(v), 1e-12), (test, f)
    z = np.load(os.path.join(GOLDEN, "voxel_firstorder.npz"))
    for name, r in (("r1", 1), ("r2", 2)):
        m = z[name + "_mask"]
        got = FO.extract(z["image"], m, voxelBased=True, spacing_xyz=z["spacing"], kernelRadius=r, binWidth=25, voxelArrayShift=100)
        for f in FO.NAMES:
            if f not in ("Entropy", "Uniformity"):
                assert np.allclose(got[f], z[f"{name}_{f}"][m], rtol=1e-10, atol=1e-9), (name, f)
