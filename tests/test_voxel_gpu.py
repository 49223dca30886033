"""GPU parity tests of the fused voxel-based feature kernels (through the C ABI)."""
import ctypes as C

import numpy as np
import pytest
import torch

import pipeline as PL
from helpers import RTOL, assert_maps_close, binned, ref_map, voxel_goldens
from pyradiomics_b200 import _lib, voxel

pytestmark = pytest.mark.gpu


def _maps_host(cname, lev, Ng, nlev, spacing=(1, 1, 1), **kw):
    """all maps of one class through the HOST-buffer C-ABI entry point"""
    L = _lib.lib()
    img = np.ascontiguousarray(lev, dtype=np.int32)
    msk = np.ascontiguousarray(lev != 0, dtype=np.uint8)
    s = _lib.make_settings(Ng, nlev, spacing_zyx=spacing, **kw)
    nf = L.rb_num_features(_lib.CLASS_ID[cname])
    out = np.empty((nf,) + img.shape)
    _lib.check(L.rb_voxel_features_host(_lib.CLASS_ID[cname], img.ctypes.data_as(C.c_void_p), msk.ctypes.data_as(C.c_void_p),
                                        *img.shape, C.byref(s), out.ctypes.data_as(C.c_void_p)), cname)
    return dict(zip(_lib.feature_names(cname), out))


# voxelx_image2d is left to test_plugins_gpu.py: how a 2-D image maps onto one plane (spacing, force2D axis) is decided in
# featureclasses, not in the kernels' C ABI
GOLDENS = [g for g in voxel_goldens(extra=True) if g[0] != "image2d"]


@pytest.mark.parametrize("name,z,kw", GOLDENS, ids=[g[0] for g in GOLDENS])
def test_golden_maps_from_the_reference(name, z, kw):
    kw2 = {k: v for k, v in kw.items() if k not in ("binWidth", "binCount", "maskedKernel")}
    sp = z["spacing"][::-1]
    if kw.get("maskedKernel", True):
        lev, levels, Ng = binned(z, kw)
        lev = np.where(z["mask"], lev, 0)
        for cname in _lib.CLASSES:
            got = _maps_host(cname, lev, Ng, len(levels), spacing=sp, **kw2)
            for f, arr in got.items():
                assert_maps_close(arr, ref_map(z, cname, f), f"{name}/{cname}/{f}")
        return
    # unmasked kernel (maskedKernel=False): the whole image is binned and seen by the windows, the ROI only selects the
    # centre voxels -- the device API's `centers`
    lev, _, levels, Ng = PL.bin_image(z["image"], np.ones(z["mask"].shape, bool), kw.get("binWidth", 25), kw.get("binCount"))
    img = torch.as_tensor(np.ascontiguousarray(lev, dtype=np.int32)).cuda()
    packed, _ = voxel.pack_levels(img, torch.ones_like(img), Ng)
    centers = torch.as_tensor(np.ascontiguousarray(z["mask"], dtype=np.uint8)).cuda()
    s = _lib.make_settings(Ng, len(levels), spacing_zyx=sp, **kw2)
    m = z["mask"].astype(bool)
    for cname in _lib.CLASSES:
        out = voxel.voxel_features(cname, packed, s, centers=centers).cpu().numpy()
        for k, f in enumerate(_lib.feature_names(cname)):
            assert (out[k][~m] == 0).all(), f"{name}/{cname}/{f}: initValue outside the ROI"
            assert_maps_close(out[k][m], ref_map(z, cname, f).reshape(m.shape)[m], f"{name}/{cname}/{f}")


def _random_volume(kind, shape, seed):
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        return rng.integers(1, 33, shape).astype(np.int32)
    zz, yy, xx = np.meshgrid(*[np.arange(s) for s in shape], indexing="ij")
    f = np.sin(zz / 2.7) + np.cos(yy / 3.1) + np.sin(xx / 2.3 + 1) + 0.25 * rng.normal(size=shape)
    q = np.quantile(f, np.linspace(0, 1, 33)[1:-1])
    return (np.digitize(f, q) + 1).astype(np.int32)


@pytest.mark.parametrize("kind", ["uniform", "smooth"])
def test_against_oracle_on_seeded_volume(kind):
    """BASELINE.json config-2/3 generators at a size the oracle finishes in seconds"""
    shape = (10, 11, 12)
    lev = _random_volume(kind, shape, 0)
    msk = np.ones(shape, bool)
    levels = np.unique(lev)
    for cname in _lib.CLASSES:
        got = _maps_host(cname, lev, int(levels.max()), len(levels))
        ref = PL.extract(cname, lev, msk, voxelBased=True, binWidth=1)
        for f, arr in ref.items():
            assert_maps_close(got[f][msk], arr, f"{kind}/{cname}/{f}")


def test_level_range_error_is_loud():
    lev = np.ones((4, 4, 4), np.int32)
    lev[1, 1, 1] = 9
    with pytest.raises(IndexError):
        _maps_host("gldm", lev, 3, 2)


@pytest.mark.parametrize("cname", _lib.CLASSES)
def test_slab_and_reflection_properties_at_scale(cname):
    """size-independent properties on a 96^3 volume: (i) computing z-slabs separately equals the
    whole-volume maps bit for bit (the multi-GPU decomposition), (ii) reflecting the volume along
    x reflects every map (texture matrices are reflection-invariant)."""
    torch.manual_seed(0)
    dev = torch.device("cuda")
    N = 96 if cname != "glcm" else 64
    lev = torch.randint(1, 33, (N, N, N), device=dev, dtype=torch.uint8)
    s = _lib.make_settings(32, 32)
    whole = voxel.voxel_features(cname, lev, s)
    parts = [voxel.voxel_features(cname, lev, s, z0=a, z1=b) for a, b in ((0, N // 3), (N // 3, N - 5), (N - 5, N))]
    assert torch.equal(torch.cat(parts, 1), whole)
    flipped = voxel.voxel_features(cname, lev.flip(2).contiguous(), s).flip(3)
    a, b = whole.cpu().numpy(), flipped.cpu().numpy()
    assert np.isfinite(a).all()
    # a reflection reorders the level-graph nodes of the fp64 eigen-solves (and their floating-point sums): MCC moves in
    # the last bits only
    assert np.allclose(a, b, rtol=1e-9, atol=1e-11 if cname == "glcm" else 1e-12)


def test_tensor_api_matches_host_api():
    lev = _random_volume("smooth", (9, 9, 9), 5)
    res = voxel.extract_maps(lev, np.ones_like(lev, bool), classes=("ngtdm", "gldm"))
    for cname in ("ngtdm", "gldm"):
        host = _maps_host(cname, lev, int(lev.max()), len(np.unique(lev)))
        for f, t in res[cname].items():
            assert np.array_equal(t.cpu().numpy(), host[f])


@pytest.mark.parametrize("kind", ["uniform", "smooth"])
def test_glcm_fast_path_equals_generic_kernel(kind, monkeypatch):
    """the r=1 GLCM fast kernel against the generic kernel (same C ABI, env switch) on 40^3"""
    lev = torch.as_tensor(_random_volume(kind, (40, 40, 40), 2).astype(np.uint8)).cuda()
    if kind == "smooth":
        lev[5:9, 3:30, 7] = 0  # holes in the mask
    s = _lib.make_settings(32, 32)
    fast = voxel.voxel_features("glcm", lev, s).cpu().numpy()
    monkeypatch.setenv("B200_RADIOMICS_FORCE_GENERIC", "1")
    gen = voxel.voxel_features("glcm", lev, s).cpu().numpy()
    monkeypatch.delenv("B200_RADIOMICS_FORCE_GENERIC")
    names = _lib.feature_names("glcm")
    for k, f in enumerate(names):
        # the generic kernel's MCC is a bisection on the eigenvalues of M M^T followed by a square root near 0, good to
        # ~1e-7 absolute (the fast path's MCC is held to 1e-9 against LAPACK in test_voxel_fastpath_edges_gpu.py); Imc1 / Imc2
        # of near-independent margins are rounding noise in every implementation
        atol = 1e-6 if f in ("MCC", "Imc2", "Imc1") else 1e-9
        assert np.allclose(fast[k], gen[k], rtol=1e-7, atol=atol, equal_nan=True), f


@pytest.mark.parametrize("kind", ["uniform", "smooth"])
def test_glrlm_fast_path_equals_generic_kernel(kind, monkeypatch):
    lev = torch.as_tensor(_random_volume(kind, (40, 40, 40), 3).astype(np.uint8)).cuda()
    lev[5:9, 3:30, 7] = 0
    lev[20, :, :] = 0
    s = _lib.make_settings(32, 32)
    fast = voxel.voxel_features("glrlm", lev, s).cpu().numpy()
    monkeypatch.setenv("B200_RADIOMICS_FORCE_GENERIC", "1")
    gen = voxel.voxel_features("glrlm", lev, s).cpu().numpy()
    monkeypatch.delenv("B200_RADIOMICS_FORCE_GENERIC")
    assert np.allclose(fast, gen, rtol=1e-10, atol=1e-12, equal_nan=True)


@pytest.mark.parametrize("cname", ["glszm", "gldm", "ngtdm"])
@pytest.mark.parametrize("kind,alpha", [("uniform", 0), ("smooth", 0), ("smooth", 2)])
def test_small_class_fast_paths_equal_generic_kernel(cname, kind, alpha, monkeypatch):
    lev = torch.as_tensor(_random_volume(kind, (36, 40, 44), 4).astype(np.uint8)).cuda()
    lev[5:9, 3:30, 7] = 0
    lev[20, :, :] = 0
    s = _lib.make_settings(32, 32, gldm_a=alpha)
    fast = voxel.voxel_features(cname, lev, s).cpu().numpy()
    monkeypatch.setenv("B200_RADIOMICS_FORCE_GENERIC", "1")
    gen = voxel.voxel_features(cname, lev, s).cpu().numpy()
    monkeypatch.delenv("B200_RADIOMICS_FORCE_GENERIC")
    assert np.allclose(fast, gen, rtol=1e-10, atol=1e-12, equal_nan=True)


def test_host_extractor_chunks_and_halo_block():
    """the e2e host-buffer path: z-chunked kernels + per-map D2H copies == the device API; the
    z0:z1 interior of a block with halo planes == the same planes of the whole volume"""
    lev = _random_volume("smooth", (11, 10, 9), 6)
    msk = np.ones(lev.shape, np.uint8)
    dev = torch.as_tensor(lev.astype(np.uint8)).cuda()
    s = _lib.make_settings(32, 32)
    hx = voxel.HostExtractor(lev.shape, zchunk=3)
    res = hx.run(lev, msk, 32, 32)
    for c in _lib.CLASSES:
        assert np.array_equal(res[c].numpy(), voxel.voxel_features(c, dev, s).cpu().numpy()), c
    hx2 = voxel.HostExtractor((7, 10, 9), classes=("glrlm", "ngtdm"), z0=1, z1=6, zchunk=2)
    full_alive = None
    res2 = hx2.run(lev[3:10], msk[3:10], 32, 32)
    for c in ("glrlm", "ngtdm"):
        assert np.array_equal(res2[c].numpy(), voxel.voxel_features(c, dev, s, z0=4, z1=9).cpu().numpy()), c


def test_sixteen_bit_levels_take_the_generic_kernels():
    """Ng > 255 -> uint16 level volume -> generic kernels; against the oracle"""
    rng = np.random.default_rng(8)
    lev = rng.integers(250, 301, (7, 8, 9)).astype(np.int32)
    lev[0, 0, 0] = 1            # keeps binWidth=1 discretisation of the oracle the identity
    lev[2, 3, 4] = 0
    msk = lev != 0
    levels = np.unique(lev[msk])
    for cname in _lib.CLASSES:
        got = _maps_host(cname, lev, int(levels.max()), len(levels))
        ref = PL.extract(cname, lev, msk, voxelBased=True, binWidth=1)
        for f, arr in ref.items():
            assert_maps_close(got[f][msk], arr, f"u16/{cname}/{f}")


def test_extract_to_nrrd_streams_device_maps_to_files(tmp_path):
    """voxel driver + output assembly (SURVEY.md 8f rank 3): kernels -> page-locked chunks -> gzip NRRD per map, checked
    through a minimal NRRD reader against the device maps"""
    import gzip
    rng = np.random.default_rng(21)
    lev = torch.as_tensor(rng.integers(1, 17, (12, 14, 15)).astype(np.uint8)).cuda()
    s = _lib.make_settings(16, 16)
    paths = voxel.extract_to_nrrd(lev, s, str(tmp_path), classes=("gldm", "glcm"), spacing_xyz=(0.5, 0.5, 2.0), zchunk=5,
                                  features={"glcm": ["MCC", "Contrast"]})
    assert set(paths) == {f"original_gldm_{n}" for n in _lib.feature_names("gldm")} | {"original_glcm_MCC", "original_glcm_Contrast"}
    ref = voxel.voxel_features("glcm", lev, s)
    for name in ("MCC", "Contrast"):
        raw = open(paths[f"original_glcm_{name}"], "rb").read()
        head, body = raw.split(b"\n\n", 1)
        assert b"sizes: 15 14 12" in head and b"type: double" in head and b"encoding: gzip" in head
        arr = np.frombuffer(gzip.decompress(body), dtype="<f8").reshape(12, 14, 15)
        assert np.array_equal(arr, ref[_lib.feature_names("glcm").index(name)].cpu().numpy(), equal_nan=True)
