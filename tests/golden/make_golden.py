"""Generates the committed golden fixtures in tests/golden/ FROM THE REFERENCE ITSELF.

Run in the build container only (needs /root/reference):  python tests/golden/make_golden.py

* segment_cases.npz / segment_expect.json -- the five bundled reference cases cropped to the
  ROI bbox (raw intensities + mask), the reference's own golden matrices
  data/baseline/<case>_<class>.npy (what reference tests/test_matrices.py:35-65 checks) and
  the feature columns of data/baseline/baseline_<class>.csv that depend only on hot-path
  settings (what reference tests/test_features.py checks).
* voxel_*.npz -- feature maps produced by the (patched, see oracle/ref_harness.py) reference
  feature classes in voxel-based mode on small seeded volumes; no reference test pins voxel
  mode (SURVEY.md section 4), so these runs of the reference are the pin.
* voxmat_*.npz -- dense per-voxel matrices from the reference `_cmatrices` (voxel mode).
"""
from __future__ import annotations

import ast
import csv
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))
import ref_harness as rh  # noqa: E402

rad = rh.load_reference()
import SimpleITK as sitk  # noqa: E402  (stub)
from radiomics import glcm, gldm, glrlm, glszm, ngtdm  # noqa: E402

CLASSES = {
    "glcm": glcm.RadiomicsGLCM, "glrlm": glrlm.RadiomicsGLRLM, "glszm": glszm.RadiomicsGLSZM,
    "gldm": gldm.RadiomicsGLDM, "ngtdm": ngtdm.RadiomicsNGTDM,
}
CASES = ["brain1", "brain2", "breast1", "lung1", "lung2"]
HOT_KEYS = {"binWidth", "binCount", "label", "distances", "force2D", "force2Ddimension",
            "symmetricalGLCM", "weightingNorm", "gldm_a"}
# settings that alter the image/mask before the hot path (need SimpleITK) -> column skipped
PRE_KEYS = {"normalize", "resampledPixelSpacing", "resegmentRange", "preCrop", "correctMask"}


def segment_goldens():
    arrays, expect = {}, {}
    for case in CASES:
        img, m, sp = rh.load_case(case)
        arrays[f"{case}_image"] = img
        arrays[f"{case}_mask"] = m
        arrays[f"{case}_spacing"] = np.array(sp)
        for cname in CLASSES:
            arrays[f"{case}_{cname}_P"] = np.load(
                os.path.join(rh.REF_ROOT, "data", "baseline", f"{case}_{cname}.npy"))
    for cname, cls in CLASSES.items():
        rows = list(csv.reader(open(os.path.join(rh.REF_ROOT, "data", "baseline", f"baseline_{cname}.csv"))))
        header = rows[0]
        byname = {r[0]: r for r in rows}
        for col in range(1, len(header)):
            test = header[col]
            case = byname["diagnostics_Configuration_TestCase"][col]
            settings = ast.literal_eval(byname["diagnostics_Configuration_Settings"][col])
            if any(settings.get(k) not in (None, False, [], 0) for k in PRE_KEYS):
                continue
            kw = {k: v for k, v in settings.items() if k in HOT_KEYS and v is not None}
            feats = {}
            for r in rows:
                if r[0].startswith(f"original_{cname}_"):
                    feats[r[0].split("_", 2)[2]] = float(r[col])
            # cross-check: the reference run here must reproduce its own baseline
            img, m, sp = rh.load_case(case)
            obj = cls(sitk.Image(img, sp), sitk.Image(m.astype(np.uint8), sp), **kw)
            got = obj.execute()
            worst = max(abs(float(got[f]) - v) / max(abs(v), 1e-300) for f, v in feats.items())
            assert worst < 1e-9, (cname, test, worst)
            expect.setdefault(cname, {})[test] = {"case": case, "settings": kw, "features": feats}
            print("segment", cname, test, "ok rel", worst)
    np.savez_compressed(os.path.join(HERE, "segment_cases.npz"), **arrays)
    json.dump(expect, open(os.path.join(HERE, "segment_expect.json"), "w"), indent=0, sort_keys=True)


def segment_goldens_resegmented():
    """the `_flatRegion` (resegmentRange [0], binWidth 5000: one gray level) and `_resegmentation` (sigma mode, [-3, 3])
    columns of the five texture baselines.  The mask is resegmented by the REFERENCE's own imageoperations.resegmentMask
    (plain NumPy, runs through the harness) on the ROI crop; mask + expected values -> segment_extra.npz / segment_expect_extra.json
    (oracle pins on the CPU box; the flat region is the single-level edge case of getBinEdges and of every class)."""
    from radiomics import firstorder, imageoperations as rio
    arrays, expect = {}, {}
    for cname, cls in list(CLASSES.items()) + [("firstorder", firstorder.RadiomicsFirstOrder)]:
        rows = list(csv.reader(open(os.path.join(rh.REF_ROOT, "data", "baseline", f"baseline_{cname}.csv"))))
        header = rows[0]
        byname = {r[0]: r for r in rows}
        for col in range(1, len(header)):
            test = header[col]
            if not (test.endswith("_flatRegion") or test.endswith("_resegmentation") or test.endswith("_normalization")):
                continue
            case = byname["diagnostics_Configuration_TestCase"][col]
            settings = ast.literal_eval(byname["diagnostics_Configuration_Settings"][col])
            assert not settings.get("resampledPixelSpacing")
            kw = {k: v for k, v in settings.items() if k in HOT_KEYS | {"voxelArrayShift"} and v is not None}
            img, m, sp = rh.load_case(case)
            if test.endswith("_normalization"):
                # normalizeImage (imageoperations.py:615-654) = sitk.Normalize over the WHOLE image, times normalizeScale.
                # SimpleITK is absent: restated as (x - mean) / std (N-1), checked against the baseline through the
                # reference's own feature class below; mean / std of the whole image travel with the fixture
                full, _ = rh.read_nrrd(os.path.join(rh.REF_ROOT, "data", f"{case}_image.nrrd"))
                mu, sd = float(full.astype(np.float64).mean()), float(full.astype(np.float64).std(ddof=1))
                scale = float(settings.get("normalizeScale", 1))
                nimg = (img.astype(np.float64) - mu) / sd * scale
                feats = {r[0].split("_", 2)[2]: float(r[col]) for r in rows if r[0].startswith(f"original_{cname}_")}
                got = cls(sitk.Image(nimg, sp), sitk.Image(m.astype(np.uint8), sp), **kw).execute()
                worst = max(abs(float(got[f]) - v) / max(abs(v), 1e-300) for f, v in feats.items())
                assert worst < 1e-9, (cname, test, worst)
                expect.setdefault(cname, {})[test] = {"case": case, "settings": kw, "features": feats,
                                                      "normalize": {"mean": mu, "std": sd, "scale": scale}}
                print("segment extra", cname, test, "normalised, ok rel", worst)
                continue
            im_s, ma_s = sitk.Image(img, sp), sitk.Image(m.astype(np.uint8), sp)
            ma_r = rio.resegmentMask(im_s, ma_s, resegmentRange=settings["resegmentRange"],
                                     resegmentMode=settings.get("resegmentMode", "absolute"), label=1)
            mr = sitk.GetArrayFromImage(ma_r) == 1
            feats = {r[0].split("_", 2)[2]: float(r[col]) for r in rows if r[0].startswith(f"original_{cname}_")}
            got = cls(im_s, sitk.Image(mr.astype(np.uint8), sp), **kw).execute()
            worst = max(abs(float(got[f]) - v) / max(abs(v), 1e-300) for f, v in feats.items())
            assert worst < 1e-9, (cname, test, worst)
            arrays[f"{test}_mask"] = mr
            expect.setdefault(cname, {})[test] = {"case": case, "settings": kw, "features": feats}
            print("segment extra", cname, test, "roi", int(mr.sum()), "of", int(m.sum()), "ok rel", worst)
    np.savez_compressed(os.path.join(HERE, "segment_extra.npz"), **arrays)
    json.dump(expect, open(os.path.join(HERE, "segment_expect_extra.json"), "w"), indent=0, sort_keys=True)


def segment_goldens_variants():
    """settings the baseline CSVs do not exercise in segment mode, run through the reference's classes on three bundled
    cases -> segment_expect_variants.json (same layout as segment_expect.json; oracle + plugin host-logic pins on the CPU box)"""
    variants = {
        "glcm": [dict(weightingNorm="manhattan"), dict(weightingNorm="euclidean"), dict(weightingNorm="infinity"),
                 dict(distances=[1, 2, 3]), dict(symmetricalGLCM=False), dict(force2D=True, force2Ddimension=0), dict(binCount=16),
                 dict(distances=[2], weightingNorm="euclidean", symmetricalGLCM=False)],
        "glrlm": [dict(weightingNorm="manhattan"), dict(weightingNorm="euclidean"), dict(weightingNorm="infinity"),
                  dict(force2D=True, force2Ddimension=0), dict(binCount=16)],
        "glszm": [dict(force2D=True, force2Ddimension=0), dict(binCount=16), dict(binWidth=10)],
        "gldm": [dict(gldm_a=2), dict(distances=[2]), dict(force2D=True, force2Ddimension=0), dict(gldm_a=1, distances=[1, 2])],
        "ngtdm": [dict(distances=[1, 2]), dict(force2D=True, force2Ddimension=0), dict(binCount=16)],
    }
    expect = {}
    for cname, cls in CLASSES.items():
        for case in ("brain2", "breast1", "lung1"):
            img, m, sp = rh.load_case(case)
            for k, var in enumerate(variants[cname]):
                kw = dict(binWidth=25)
                kw.update(var)
                if "binCount" in var:
                    kw.pop("binWidth")
                got = cls(sitk.Image(img, sp), sitk.Image(m.astype(np.uint8), sp), **kw).execute()
                feats = {f: float(v) for f, v in got.items()}
                expect.setdefault(cname, {})[f"{case}_x{k}"] = {"case": case, "settings": kw, "features": feats}
                print("segment variant", cname, case, var, len(feats))
    json.dump(expect, open(os.path.join(HERE, "segment_expect_variants.json"), "w"), indent=0, sort_keys=True)


def voxel_volumes():
    vols = {}
    rng = np.random.default_rng(0)
    # (a) BASELINE.json config-2 generator at toy size: iid uniform levels 1..32, full mask
    vols["uniform32"] = dict(image=rng.integers(1, 33, (7, 8, 9)).astype(np.int32),
                             mask=np.ones((7, 8, 9), bool), kw=dict(binWidth=1))
    # (b) smooth field, few levels per window, ragged mask (holes + border cut)
    z, y, x = np.meshgrid(np.arange(8), np.arange(9), np.arange(10), indexing="ij")
    sm = 40 * np.sin(z / 3.0) + 30 * np.cos(y / 4.0) + 25 * np.sin(x / 2.5) + rng.normal(0, 4, z.shape)
    msk = ((z - 3.5) ** 2 / 16 + (y - 4) ** 2 / 20 + (x - 4.5) ** 2 / 26) <= 1.0
    msk &= rng.random(z.shape) > 0.07
    vols["smooth_ragged"] = dict(image=np.round(sm * 4).astype(np.int32), mask=msk, kw=dict(binWidth=25))
    # (c) 8 levels, kernelRadius 2, distances [1,2]
    vols["r2_d12"] = dict(image=rng.integers(1, 9, (6, 7, 6)).astype(np.int32),
                          mask=rng.random((6, 7, 6)) > 0.1,
                          kw=dict(binWidth=1, kernelRadius=2, distances=[1, 2]))
    # (d) force2D + asymmetric GLCM + gldm_a=1
    vols["force2d_asym"] = dict(image=rng.integers(1, 6, (4, 8, 8)).astype(np.int32),
                                mask=rng.random((4, 8, 8)) > 0.05,
                                kw=dict(binWidth=1, force2D=True, force2Ddimension=0,
                                        symmetricalGLCM=False, gldm_a=1))
    # (e) weighted GLCM/GLRLM (anisotropic spacing)
    vols["weighted"] = dict(image=rng.integers(1, 7, (5, 6, 7)).astype(np.int32),
                            mask=np.ones((5, 6, 7), bool), spacing=(0.8, 0.8, 2.5),
                            kw=dict(binWidth=1, weightingNorm="euclidean"))
    return vols


def voxel_volumes_extra():
    """more settings variants, added at the end of round 2 (`--voxel-extra-only` -> voxelx_*.npz).  They pin the oracle and
    the host-compiled device math (tests/test_oracle.py, tests/test_host_emul.py); the GPU tests still run on voxel_*.npz."""
    vols = {}
    rng = np.random.default_rng(7)
    z, y, x = np.meshgrid(np.arange(7), np.arange(8), np.arange(7), indexing="ij")
    blob = ((z - 3) ** 2 / 9.5 + (y - 3.5) ** 2 / 13 + (x - 3) ** 2 / 10) <= 1.0
    # (f) kernelRadius 3 (343-voxel windows), 5 levels, ragged ROI
    vols["r3"] = dict(image=rng.integers(1, 6, (7, 8, 7)).astype(np.int32), mask=blob & (rng.random(blob.shape) > 0.08),
                      kw=dict(binWidth=1, kernelRadius=3))
    # (g) the other weighting norms on anisotropic spacing
    for norm in ("manhattan", "infinity", "no_weighting"):
        vols[f"w_{norm}"] = dict(image=rng.integers(1, 6, (5, 6, 6)).astype(np.int32), mask=rng.random((5, 6, 6)) > 0.1,
                                 spacing=(0.7, 1.3, 2.0), kw=dict(binWidth=1, weightingNorm=norm))
    # (h) binCount on a float image
    f = 300 * np.sin(z / 2.0) * np.cos(y / 3.0) + 40 * rng.normal(size=z.shape)
    vols["bincount8"] = dict(image=f.astype(np.float64), mask=blob, kw=dict(binCount=8))
    # (i) distance 2 only, kernelRadius 2
    vols["d2_r2"] = dict(image=rng.integers(1, 7, (6, 6, 7)).astype(np.int32), mask=rng.random((6, 6, 7)) > 0.12,
                         kw=dict(binWidth=1, kernelRadius=2, distances=[2]))
    # (j) many levels (60) at kernelRadius 1: every window is all-distinct or nearly so
    vols["ng60"] = dict(image=rng.integers(1, 61, (6, 7, 7)).astype(np.int32), mask=np.ones((6, 7, 7), bool), kw=dict(binWidth=1))
    # (k) force2D along x, gldm_a = 2
    vols["force2d_x_a2"] = dict(image=rng.integers(1, 7, (6, 7, 4)).astype(np.int32), mask=rng.random((6, 7, 4)) > 0.06,
                                kw=dict(binWidth=1, force2D=True, force2Ddimension=2, gldm_a=2))
    # (l) binWidth on negative intensities (lower bound below zero)
    vols["negative"] = dict(image=(rng.integers(-260, 190, (6, 6, 6))).astype(np.int32), mask=rng.random((6, 6, 6)) > 0.1,
                            kw=dict(binWidth=50))
    # (m) unmasked kernel: the windows see every voxel of the image, only ROI voxels get a value (base.py:100-104)
    vols["unmasked_kernel"] = dict(image=rng.integers(1, 9, (6, 7, 8)).astype(np.int32),
                                   mask=blob[:6, :7, :7].repeat(2, 2)[:, :, :8] & (rng.random((6, 7, 8)) > 0.2),
                                   kw=dict(binWidth=1, maskedKernel=False))
    # (n) a 2-D image (Nd = 2: 4 / 8 angles, 3 x 3 windows)
    vols["image2d"] = dict(image=rng.integers(1, 7, (9, 10)).astype(np.int32), mask=rng.random((9, 10)) > 0.12, spacing=(0.8, 1.1),
                           kw=dict(binWidth=1))
    return vols


def voxel_goldens(extra=False):
    for name, v in (voxel_volumes_extra() if extra else voxel_volumes()).items():
        sp = v.get("spacing", (1.0, 1.0, 1.0))
        out = {"image": v["image"], "mask": v["mask"], "spacing": np.array(sp),
               "settings": np.array(json.dumps(v["kw"]))}
        for cname, cls in CLASSES.items():
            obj = cls(sitk.Image(v["image"], sp), sitk.Image(v["mask"].astype(np.uint8), sp),
                      voxelBased=True, **v["kw"])
            res = obj.execute()
            for f, im in res.items():
                out[f"{cname}_{f}"] = sitk.GetArrayFromImage(im)
            print("voxel", name, cname, len(res))
            if cname == "glcm":
                # Reference defect (SURVEY.md App. A #6): one voxel with an empty angle makes
                # eigvals raise and the WHOLE batch's MCC map stays at initValue.  Pin the
                # per-voxel meaning with voxelBatch=1 (each voxel its own batch -> empty angles
                # are dropped per voxel, failures stay local).
                o1 = cls(sitk.Image(v["image"], sp), sitk.Image(v["mask"].astype(np.uint8), sp),
                         voxelBased=True, voxelBatch=1, **v["kw"])
                o1.enableFeatureByName("MCC")
                import logging
                logging.getLogger("radiomics").setLevel(logging.CRITICAL)
                out["glcm_MCC_voxelBatch1"] = sitk.GetArrayFromImage(o1.execute()["MCC"])
                logging.getLogger("radiomics").setLevel(logging.INFO)
        np.savez_compressed(os.path.join(HERE, f"voxel{'x' if extra else ''}_{name}.npz"), **out)


def voxmat_goldens():
    """dense per-voxel matrices straight from the reference C extension (integer parity)."""
    cm = rad.cMatrices
    rng = np.random.default_rng(1)
    img = rng.integers(1, 7, (5, 6, 7)).astype(np.int32)
    msk = rng.random((5, 6, 7)) > 0.15
    vox = np.array(np.where(msk)).astype(np.int32)
    out = {"image": img, "mask": msk, "voxels": vox}
    out["glcm"], out["glcm_angles"] = cm.calculate_glcm(img, msk, np.array([1]), 6, False, 0, 1, vox)
    out["glrlm"], out["glrlm_angles"] = cm.calculate_glrlm(img, msk, 6, 7, False, 0, 1, vox)
    out["glszm"] = cm.calculate_glszm(img, msk, 6, int(msk.sum()), False, 0, 1, vox)
    out["gldm"] = cm.calculate_gldm(img, msk, np.array([1]), 6, 0, False, 0, 1, vox)
    out["ngtdm"] = cm.calculate_ngtdm(img, msk, np.array([1]), 6, False, 0, 1, vox)
    np.savez_compressed(os.path.join(HERE, "voxmat_small.npz"), **out)


def firstorder_goldens():
    """first-order class (SURVEY.md section 8f rank 2): baseline CSV columns (segment mode) and a
    voxel-mode run of the reference.  The voxel volume keeps the ROI >= 2*kernelRadius away from the
    far border because the reference indexes its unpadded discretised array with padded coordinates
    (firstorder.py:109) and raises IndexError otherwise; for the same reason its voxel-mode Entropy /
    Uniformity (shifted histogram window) are NOT stored as goldens."""
    from radiomics import firstorder
    rows = list(csv.reader(open(os.path.join(rh.REF_ROOT, "data", "baseline", "baseline_firstorder.csv"))))
    header = rows[0]
    byname = {r[0]: r for r in rows}
    expect = {}
    for col in range(1, len(header)):
        test = header[col]
        case = byname["diagnostics_Configuration_TestCase"][col]
        settings = ast.literal_eval(byname["diagnostics_Configuration_Settings"][col])
        if any(settings.get(k) not in (None, False, [], 0) for k in PRE_KEYS):
            continue
        kw = {k: v for k, v in settings.items() if k in HOT_KEYS | {"voxelArrayShift"} and v is not None}
        feats = {r[0].split("_", 2)[2]: float(r[col]) for r in rows if r[0].startswith("original_firstorder_")}
        img, m, sp = rh.load_case(case)
        got = firstorder.RadiomicsFirstOrder(sitk.Image(img, sp), sitk.Image(m.astype(np.uint8), sp), **kw).execute()
        worst = max(abs(float(got[f]) - v) / max(abs(v), 1e-300) for f, v in feats.items())
        assert worst < 1e-9, (test, worst)
        expect[test] = {"case": case, "settings": kw, "features": feats}
        print("segment firstorder", test, "ok rel", worst)
    json.dump(expect, open(os.path.join(HERE, "segment_expect_firstorder.json"), "w"), indent=0, sort_keys=True)
    rng = np.random.default_rng(21)
    z, y, x = np.meshgrid(np.arange(10), np.arange(11), np.arange(12), indexing="ij")
    img = (300 + 120 * np.sin(z / 2.0) + 90 * np.cos(y / 3.0) + 60 * np.sin(x / 2.5) + rng.normal(0, 25, z.shape)).astype(np.int16)
    out = {"image": img}
    for name, r, msk in (("r1", 1, (rng.random(z.shape) > 0.2) & (z < 8) & (y < 9) & (x < 10)),
                         ("r2", 2, (rng.random(z.shape) > 0.3) & (z < 6) & (y < 7) & (x < 8))):
        sp = (0.8, 0.9, 2.0)
        obj = firstorder.RadiomicsFirstOrder(sitk.Image(img, sp), sitk.Image(msk.astype(np.uint8), sp), voxelBased=True,
                                             kernelRadius=r, binWidth=25, voxelArrayShift=100)
        res = obj.execute()
        out[f"{name}_mask"] = msk
        for f, im in res.items():
            if f not in ("Entropy", "Uniformity"):
                out[f"{name}_{f}"] = sitk.GetArrayFromImage(im)
        print("voxel firstorder", name, len(res))
    out["spacing"] = np.array((0.8, 0.9, 2.0))
    np.savez_compressed(os.path.join(HERE, "voxel_firstorder.npz"), **out)


def shape_goldens():
    """segment-mode shape class (SURVEY.md section 8f rank 4).
    (a) shape_cube_probes.npz: the reference's (surface area, volume) of every single-cube mask
        (256 corner configurations, bit i <-> corner (z, y, x) = (i>>2 & 1, i>>1 & 1, i & 1)) under three
        spacings -- the black-box behaviour the marching-cubes table of the product is derived from and
        checked against (csrc/gen_mc_table.py);
    (b) shape_expect.json: baseline_shape.csv columns without resampling, re-verified against a run of the
        reference class here;
    (c) shape_random.npz: random / structured masks with the reference's coefficients."""
    import build_ref
    from radiomics import shape
    cs = build_ref.load("_cshape")
    spacings = np.array([(1.0, 1.0, 1.0), (1.0, 1.3, 1.7), (2.1, 0.7, 1.1)])
    probes = np.zeros((256, 3, 2))
    for cfg in range(256):
        m = np.zeros((2, 2, 2), dtype=bool)
        for i in range(8):
            if cfg >> i & 1:
                m[i >> 2 & 1, i >> 1 & 1, i & 1] = True
        for k, sp in enumerate(spacings):
            sa, vol, _ = cs.calculate_coefficients(m, sp)
            probes[cfg, k] = (sa, vol)
    np.savez_compressed(os.path.join(HERE, "shape_cube_probes.npz"), spacings=spacings, probes=probes)
    rows = list(csv.reader(open(os.path.join(rh.REF_ROOT, "data", "baseline", "baseline_shape.csv"))))
    header = rows[0]
    byname = {r[0]: r for r in rows}
    expect = {}
    for col in range(1, len(header)):
        test = header[col]
        case = byname["diagnostics_Configuration_TestCase"][col]
        settings = ast.literal_eval(byname["diagnostics_Configuration_Settings"][col])
        if any(settings.get(k) not in (None, False, [], 0) for k in PRE_KEYS):
            continue
        feats = {r[0].split("_", 2)[2]: float(r[col]) for r in rows if r[0].startswith("original_shape_")}
        img, m, sp = rh.load_case(case)
        obj = shape.RadiomicsShape(sitk.Image(img, sp), sitk.Image(m.astype(np.uint8), sp))
        obj.enableAllFeatures()
        got = obj.execute()
        worst = max(abs(float(got[f]) - v) / max(abs(v), 1e-300) for f, v in feats.items())
        # the stored CSV predates the reference's current mesh table (SurfaceArea differs by 8e-4 on brain1); the
        # reference's own test accepts 3 % (tests/testUtils.py:266-275).  The tight goldens are the values computed here.
        assert worst < 0.03, (test, worst)
        expect[test] = {"case": case, "features": {f: float(got[f]) for f in got}, "baseline": feats}
        print("segment shape", test, "ok rel", worst, len(got), "features")
    json.dump(expect, open(os.path.join(HERE, "shape_expect.json"), "w"), indent=0, sort_keys=True)
    rng = np.random.default_rng(33)
    out = {}
    z, y, x = np.meshgrid(np.arange(14), np.arange(17), np.arange(19), indexing="ij")
    masks = {
        "blob": ((z - 6.3) ** 2 / 20 + (y - 8.1) ** 2 / 40 + (x - 9.2) ** 2 / 60) < 1.0,
        "noise": rng.random(z.shape) > 0.5,
        "sparse": rng.random(z.shape) > 0.93,
        "touching_border": np.ones((5, 6, 7), dtype=bool),
        "single": np.pad(np.ones((1, 1, 1), dtype=bool), 2),
        "plane": np.pad(np.ones((1, 6, 7), dtype=bool), 1),
    }
    for name, m in masks.items():
        sp = np.array((2.5, 0.8, 1.1))
        sa, vol, dia = cs.calculate_coefficients(np.ascontiguousarray(m), sp)
        out[f"{name}_mask"] = m
        out[f"{name}_coeff"] = np.array([sa, vol, *dia])
        out[f"{name}_spacing"] = sp
        print("shape coeff", name, sa, vol, dia)
    np.savez_compressed(os.path.join(HERE, "shape_random.npz"), **out)


def shape2d_goldens():
    """2-D shape coefficients of the compiled reference _cshape (calculate_coefficients2D, cshape.c:420-595) on padded
    random / structured single-slice masks -> shape2d_golden.npz"""
    import build_ref
    cs = build_ref.load("_cshape")
    rng = np.random.default_rng(7)
    yy, xx = np.mgrid[0:40, 0:48]
    masks = {
        "disc": ((yy - 20) ** 2 / 1.0 + (xx - 22) ** 2 / 1.7) < 150,
        "noise": rng.random((30, 33)) < 0.5,
        "sparse": rng.random((25, 25)) < 0.08,
        "touching_border": np.zeros((12, 14), bool),
        "single": np.zeros((5, 5), bool),
        "checker": (yy[:10, :11] + xx[:10, :11]) % 2 == 0,
        "ring": (((yy - 20) ** 2 + (xx - 24) ** 2) < 300) & (((yy - 20) ** 2 + (xx - 24) ** 2) > 90),
    }
    masks["touching_border"][0:5, 9:14] = True
    masks["single"][2, 2] = True
    out = {}
    for name, m in masks.items():
        sp = np.array([1.0 + 0.37 * (len(name) % 3), 0.8 + 0.11 * (len(name) % 4)])
        ref = cs.calculate_coefficients2D(np.pad(m.astype(np.int8), 1), sp)
        out[name + "_mask"], out[name + "_spacing"], out[name + "_coeff"] = m, sp, np.array(ref)
        print("shape2D coeff", name, ref)
    np.savez_compressed(os.path.join(HERE, "shape2d_golden.npz"), **out)


def resample_goldens():
    """the reference's bundled breast1 case (small enough to commit whole) + every `original_*` value of the
    `breast1_resampling` column of data/baseline/baseline_<class>.csv (resampledPixelSpacing [2,2,2], sitkBSpline):
    the pin of the resampling step -> resample_breast1.npz"""
    import csv
    import ref_harness as rh
    img, sp = rh.read_nrrd(os.path.join(rh.REF_ROOT, "data", "breast1_image.nrrd"))
    msk, _ = rh.read_nrrd(os.path.join(rh.REF_ROOT, "data", "breast1_label.nrrd"))
    exp = {}
    for cls in ("firstorder", "glcm", "glrlm", "glszm", "gldm", "ngtdm", "shape"):
        rows = list(csv.reader(open(os.path.join(rh.REF_ROOT, "data", "baseline", f"baseline_{cls}.csv"))))
        i = rows[0].index("breast1_resampling")
        for r in rows[1:]:
            if r[0].startswith("original_"):
                exp[r[0]] = float(r[i])
    np.savez_compressed(os.path.join(HERE, "resample_breast1.npz"), image=img, mask=msk.astype(np.uint8), spacing=np.array(sp),
                        names=np.array(sorted(exp)), values=np.array([exp[k] for k in sorted(exp)]))
    print("resample golden", img.shape, sp, len(exp), "values")
    # the other four bundled cases, cropped: ROI box + the pad distance + 16 voxels (the cubic B-spline decomposition forgets
    # a mirrored edge after ~16 samples), with the index the crop started at and the full size -- the output grid is
    # anchored at the full image's index 0.  The crop resamples to exactly the arrays of the whole image (checked here).
    import resample_np as RS
    out = {}
    for case in ("brain1", "brain2", "lung1", "lung2"):
        img, sp = rh.read_nrrd(os.path.join(rh.REF_ROOT, "data", f"{case}_image.nrrd"))
        msk, _ = rh.read_nrrd(os.path.join(rh.REF_ROOT, "data", f"{case}_label.nrrd"))
        msk = msk.astype(np.uint8)
        exp = {}
        for cls in ("firstorder", "glcm", "glrlm", "glszm", "gldm", "ngtdm", "shape"):
            rows = list(csv.reader(open(os.path.join(rh.REF_ROOT, "data", "baseline", f"baseline_{cls}.csv"))))
            i = rows[0].index(f"{case}_resampling")
            for r in rows[1:]:
                if r[0].startswith("original_"):
                    exp[r[0]] = float(r[i])
        idx = np.array(np.where(msk == 1))
        marg = np.ceil((5 * 2.0 + 2.0) / np.array(sp)[::-1]).astype(int) + 16
        a = np.maximum(idx.min(1) - marg, 0)
        b = np.minimum(idx.max(1) + marg + 1, np.array(img.shape))
        sl = tuple(slice(x, y) for x, y in zip(a, b))
        ci, cm = np.ascontiguousarray(img[sl]), np.ascontiguousarray(msk[sl])
        off, full = tuple(int(v) for v in a[::-1]), img.shape[::-1]
        whole = RS.resample(img, msk, sp, (2, 2, 2))
        crop = RS.resample(ci, cm, sp, (2, 2, 2), offset_xyz=off, full_size_xyz=full)
        assert np.array_equal(whole[0], crop[0]) and np.array_equal(whole[1], crop[1]), case
        out.update({f"{case}_image": ci, f"{case}_mask": cm, f"{case}_spacing": np.array(sp), f"{case}_offset_xyz": np.array(off),
                    f"{case}_full_size_xyz": np.array(full), f"{case}_names": np.array(sorted(exp)),
                    f"{case}_values": np.array([exp[k] for k in sorted(exp)])})
        print("resample golden", case, ci.shape, "of", img.shape, len(exp), "values")
    np.savez_compressed(os.path.join(HERE, "resample_cases.npz"), **out)


def reference_runs():
    """what the tests compare with the compiled reference extensions and classes, so that they need neither ->
    reference_runs.json:
    (a) port_trials: sha256 digests (helpers.digest) of every matrix the reference _cmatrices returns on the seeded
        trials of helpers.port_trials (null where the reference refuses the trial's angles);
    (b) argument_errors: the exception type the reference _cmatrices raises for each malformed call of
        test_plugin_host_logic_cpu.BAD_CALLS;
    (c) large_roi_shape: the reference _cshape's (surface area, volume, diameters) of test_shape_gpu's 96^3 ellipsoid;
    (d) feature_names: getFeatureNames() of the reference's feature classes."""
    import importlib

    import build_ref
    sys.path[:0] = [os.path.join(HERE, ".."), os.path.join(HERE, "..", "..")]
    import helpers
    from test_plugin_host_logic_cpu import BAD_CALLS
    from test_shape_gpu import large_roi_case

    cm = build_ref.load()
    trials = []
    for trial, *args in helpers.port_trials():
        if args[1].sum() == 0:
            trials.append(None)
            continue
        try:
            trials.append([helpers.digest(a) for a in helpers.port_trial_outputs(cm, *args)])
        except RuntimeError:
            trials.append(None)
    errors = {}
    img, msk = np.ones((4, 5, 6), np.int32), np.ones((4, 5, 6), bool)
    for what, call in BAD_CALLS.items():
        try:
            call(cm, img, msk)
        except Exception as e:
            errors[what] = type(e).__name__
    m, sp = large_roi_case()
    sa, vol, dia = build_ref.load("_cshape").calculate_coefficients(m, sp)
    names = {}
    for mod, cls in (("glcm", "RadiomicsGLCM"), ("glrlm", "RadiomicsGLRLM"), ("glszm", "RadiomicsGLSZM"), ("gldm", "RadiomicsGLDM"),
                     ("ngtdm", "RadiomicsNGTDM"), ("firstorder", "RadiomicsFirstOrder"), ("shape", "RadiomicsShape"),
                     ("shape2D", "RadiomicsShape2D")):
        names[mod] = getattr(importlib.import_module(f"radiomics.{mod}"), cls).getFeatureNames()
    out = {"port_trials": trials, "argument_errors": errors,
           "large_roi_shape": {"surface_area": float(sa), "volume": float(vol), "diameters": [float(v) for v in dia]},
           "feature_names": names}
    json.dump(out, open(os.path.join(HERE, "reference_runs.json"), "w"), indent=0, sort_keys=True)
    print("reference runs:", sum(t is not None for t in trials), "port trials,", len(errors), "argument errors")


if __name__ == "__main__":
    if "--reference-runs-only" in sys.argv:
        reference_runs()
        sys.exit(0)
    if "--segment-variants-only" in sys.argv:
        segment_goldens_variants()
        sys.exit(0)
    if "--segment-extra-only" in sys.argv:
        segment_goldens_resegmented()
        sys.exit(0)
    if "--voxel-extra-only" in sys.argv:
        voxel_goldens(extra=True)
        sys.exit(0)
    if "--resample-only" in sys.argv:
        resample_goldens()
        sys.exit(0)
    if "--shape2d-only" in sys.argv:
        shape2d_goldens()
        sys.exit(0)
    if "--shape-only" in sys.argv:
        shape_goldens()
        sys.exit(0)
    if "--firstorder-only" in sys.argv:
        firstorder_goldens()
        sys.exit(0)
    segment_goldens()
    firstorder_goldens()
    voxmat_goldens()
    voxel_goldens()
