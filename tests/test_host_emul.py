"""CPU check of the DEVICE arithmetic: pyradiomics_b200/csrc/vox_features.cuh is __host__
__device__, so tests/host_emul/emul.cpp compiles it with g++ and the per-voxel feature math the
CUDA kernels run is compared with the reference's voxel-mode golden maps without a GPU.
(Test-only build; the product never runs this code on the CPU.)"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cmatrices_oracle as O
import pipeline as PL
from helpers import (adversarial_windows, assert_maps_close, binned, mcc_angle_numpy, random_window, ref_map, slot_angles,
                     voxel_goldens)
from pyradiomics_b200 import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
NAMES = {
    "glcm": ["Autocorrelation", "ClusterProminence", "ClusterShade", "ClusterTendency", "Contrast", "Correlation",
             "DifferenceAverage", "DifferenceEntropy", "DifferenceVariance", "Id", "Idm", "Idmn", "Idn", "Imc1", "Imc2",
             "InverseVariance", "JointAverage", "JointEnergy", "JointEntropy", "MCC", "MaximumProbability", "SumAverage",
             "SumEntropy", "SumSquares"],
    "glrlm": ["GrayLevelNonUniformity", "GrayLevelNonUniformityNormalized", "GrayLevelVariance", "HighGrayLevelRunEmphasis",
              "LongRunEmphasis", "LongRunHighGrayLevelEmphasis", "LongRunLowGrayLevelEmphasis", "LowGrayLevelRunEmphasis",
              "RunEntropy", "RunLengthNonUniformity", "RunLengthNonUniformityNormalized", "RunPercentage", "RunVariance",
              "ShortRunEmphasis", "ShortRunHighGrayLevelEmphasis", "ShortRunLowGrayLevelEmphasis"],
    "glszm": ["GrayLevelNonUniformity", "GrayLevelNonUniformityNormalized", "GrayLevelVariance", "HighGrayLevelZoneEmphasis",
              "LargeAreaEmphasis", "LargeAreaHighGrayLevelEmphasis", "LargeAreaLowGrayLevelEmphasis", "LowGrayLevelZoneEmphasis",
              "SizeZoneNonUniformity", "SizeZoneNonUniformityNormalized", "SmallAreaEmphasis", "SmallAreaHighGrayLevelEmphasis",
              "SmallAreaLowGrayLevelEmphasis", "ZoneEntropy", "ZonePercentage", "ZoneVariance"],
    "gldm": ["DependenceEntropy", "DependenceNonUniformity", "DependenceNonUniformityNormalized", "DependenceVariance",
             "GrayLevelNonUniformity", "GrayLevelVariance", "HighGrayLevelEmphasis", "LargeDependenceEmphasis",
             "LargeDependenceHighGrayLevelEmphasis", "LargeDependenceLowGrayLevelEmphasis", "LowGrayLevelEmphasis",
             "SmallDependenceEmphasis", "SmallDependenceHighGrayLevelEmphasis", "SmallDependenceLowGrayLevelEmphasis"],
    "ngtdm": ["Busyness", "Coarseness", "Complexity", "Contrast", "Strength"],
}


@pytest.fixture(scope="module")
def emul():
    so = os.path.join(HERE, "host_emul", "libemul.so")
    src = os.path.join(HERE, "host_emul", "emul.cpp")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", so + ".%d" % os.getpid(), src])
    os.replace(so + ".%d" % os.getpid(), so)
    return C.CDLL(so)


def alive_mask_bruteforce(lev, centers, ang, r3):
    """which GLCM angles have a co-occurrence inside at least one kernel window (numpy restatement
    of the reference's 'delete empty angles', radiomics/glcm.py:187-196)."""
    m = lev != 0
    out = np.zeros(_lib.ALIVE_WORDS, np.uint32)
    for ai, a in enumerate(ang):
        pm = np.zeros_like(m)
        src = tuple(slice(max(0, -a[d]), lev.shape[d] - max(0, a[d])) for d in range(3))
        dst = tuple(slice(max(0, a[d]), lev.shape[d] + min(0, a[d])) for d in range(3))
        pm[src] = m[src] & m[dst]
        for c in zip(*np.where(centers)):
            lo = [max(c[d] - r3[d], c[d] - r3[d] - a[d], 0) for d in range(3)]
            hi = [min(c[d] + r3[d], c[d] + r3[d] - a[d], lev.shape[d] - 1) for d in range(3)]
            if all(lo[d] <= hi[d] for d in range(3)) and pm[lo[0]:hi[0] + 1, lo[1]:hi[1] + 1, lo[2]:hi[2] + 1].any():
                out[ai >> 5] |= np.uint32(1 << (ai & 31))
                break
    return out


def test_feature_name_tables_match_library_order():
    for cls, names in NAMES.items():
        assert names == sorted(names, key=lambda s: s) or cls == "glcm"  # 'MCC' < 'Ma...' in ASCII
        assert len(names) == {"glcm": 24, "glrlm": 16, "glszm": 16, "gldm": 14, "ngtdm": 5}[cls]


@pytest.mark.parametrize("name,z,kw", voxel_goldens(extra=True), ids=[g[0] for g in voxel_goldens(extra=True)])
def test_device_math_on_host_matches_reference_maps(emul, name, z, kw):
    centers = None
    if kw.get("maskedKernel", True):
        lev, levels, Ng = binned(z, kw)
    else:
        # unmasked kernel (base.py:100-104): every voxel of the image is binned and seen by the windows, the ROI only
        # selects the centre voxels (the kernel's `centers` argument, what the plugin passes for maskedKernel=False)
        lev, _, levels, Ng = PL.bin_image(z["image"], np.ones(z["mask"].shape, bool), kw.get("binWidth", 25), kw.get("binCount"))
        centers = np.ascontiguousarray(z["mask"], dtype=np.uint8)
    mask, sp_zyx = z["mask"], tuple(z["spacing"][::-1])
    if lev.ndim == 2:                        # a 2-D image runs as one plane, like featureclasses.levels3d / _voxel_settings
        lev, mask, sp_zyx = lev[None], mask[None], (1.0,) + sp_zyx
        centers = None if centers is None else centers[None]
    lev16 = np.ascontiguousarray(lev, dtype=np.uint16)
    kws = {k: v for k, v in kw.items() if k != "maskedKernel"}
    s = _lib.make_settings(Ng, len(levels), spacing_zyx=sp_zyx, **kws)
    Zs, Ys, Xs = lev.shape
    ang = O.generate_angles(lev.shape, kw.get("distances", [1]), 0, s.force2D, s.force2Ddimension)
    r3 = [0 if (s.force2D and s.force2Ddimension == k) else s.kernelRadius for k in range(3)]
    alive = alive_mask_bruteforce(lev, mask, ang, r3)
    for cid, cname in enumerate(_lib.CLASSES):
        out = np.zeros((len(NAMES[cname]), Zs, Ys, Xs))
        rc = emul.emul_voxel_features(cid, lev16.ctypes.data_as(C.c_void_p), None if centers is None else centers.ctypes.data_as(C.c_void_p),
                                      Zs, Ys, Xs, C.byref(s), alive.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
        assert rc == 0
        for k, f in enumerate(NAMES[cname]):
            ref = ref_map(z, cname, f).reshape(out[k].shape)
            got = out[k] if centers is None else np.where(mask, out[k], ref)      # (outside the ROI: initValue)
            assert_maps_close(got, ref, f"{name}/{cname}/{f}", rtol=1e-7, atol=1e-9)


@pytest.mark.parametrize("name,r", [("r1", 1), ("r2", 2)])
def test_firstorder_device_math_on_host(emul, name, r):
    """first-order window statistics (csrc/firstorder.cuh) against the reference's voxel-mode run"""
    import firstorder_np as FO
    import pipeline as PL
    z = np.load(os.path.join(HERE, "golden", "voxel_firstorder.npz"))
    img, m = z["image"], z[name + "_mask"]
    lev, _, _, _ = PL.bin_image(img, m, 25)
    lev16 = np.ascontiguousarray(np.where(m, lev, 0), dtype=np.uint16)
    imgd = np.ascontiguousarray(img, dtype=np.float64)
    mk = np.ascontiguousarray(m, dtype=np.uint8)
    Zs, Ys, Xs = img.shape
    out = np.zeros((18, Zs, Ys, Xs))
    emul.emul_firstorder(imgd.ctypes.data_as(C.c_void_p), mk.ctypes.data_as(C.c_void_p), lev16.ctypes.data_as(C.c_void_p),
                         Zs, Ys, Xs, r, r, r, C.c_double(100.0), C.c_double(float(np.prod(z["spacing"]))),
                         out.ctypes.data_as(C.c_void_p))
    ref = FO.extract(img, m, voxelBased=True, spacing_xyz=z["spacing"], kernelRadius=r, binWidth=25, voxelArrayShift=100)
    for k, f in enumerate(FO.NAMES):
        assert np.allclose(out[k][m], ref[f], rtol=1e-10, atol=1e-9), f
        if f not in ("Entropy", "Uniformity"):
            assert np.allclose(out[k][m], z[f"{name}_{f}"][m], rtol=1e-9, atol=1e-8), f


@pytest.mark.parametrize("kind", ["uniform", "smooth", "uniform60"])
def test_glcm_fast_math_equals_generic_math_on_host(emul, kind):
    """the r=1 GLCM fast path (sorting networks, bipartite filter, dense / Lanczos eigen-tasks) against the
    generic entry-list / Householder path on a 24^3 volume with holes -- catches solver regressions without a GPU."""
    rng = np.random.default_rng(2)
    shape = (24, 24, 24)
    Ng = 60 if kind == "uniform60" else 32
    if kind.startswith("uniform"):
        lev = rng.integers(1, Ng + 1, shape)            # 60 levels: nearly every window is all-distinct (trees, n = 19)
    else:
        zz, yy, xx = np.meshgrid(*[np.arange(s) for s in shape], indexing="ij")
        f = np.sin(zz / 2.7) + np.cos(yy / 3.1) + np.sin(xx / 2.3 + 1) + 0.25 * rng.normal(size=shape)
        lev = np.digitize(f, np.quantile(f, np.linspace(0, 1, 33)[1:-1])) + 1
        lev[5:9, 3:20, 7] = 0
    lev = np.ascontiguousarray(lev, dtype=np.uint16)
    s = _lib.make_settings(Ng, Ng)
    Zs, Ys, Xs = shape
    fast = np.zeros((24, Zs, Ys, Xs))
    gen = np.zeros((24, Zs, Ys, Xs))
    assert emul.emul_glcm_fast(lev.ctypes.data_as(C.c_void_p), Zs, Ys, Xs, C.byref(s), None, fast.ctypes.data_as(C.c_void_p)) == 0
    assert emul.emul_voxel_features(0, lev.ctypes.data_as(C.c_void_p), None, Zs, Ys, Xs, C.byref(s), None, gen.ctypes.data_as(C.c_void_p)) == 0
    for k, f in enumerate(NAMES["glcm"]):
        atol = 1e-6 if f in ("Imc2", "Imc1") else 1e-9
        assert np.allclose(fast[k], gen[k], rtol=1e-7, atol=atol, equal_nan=True), f


@pytest.fixture(scope="module")
def emul_dyn():
    """the same device math with the task-sized eigenvalue search (LZ_EIG_EXACT_STATIC=0)"""
    so = os.path.join(HERE, "host_emul", "libemul_dyn.so")
    src = os.path.join(HERE, "host_emul", "emul.cpp")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-DLZ_EIG_EXACT_STATIC=0", "-o", so + ".%d" % os.getpid(), src])
    os.replace(so + ".%d" % os.getpid(), so)
    lib = C.CDLL(so)
    lib.emul_glcm_lanczos_axis.restype = C.c_double
    return lib


def test_eigen_task_solvers_against_lapack(emul, emul_dyn):
    """the dense register solve (n <= 12 levels) and the register Lanczos solve (13..18 levels, per-thread shared vectors)
    on random / structured / holed / adversarial windows, against numpy's eigvalsh -- both in fp64 throughout: 1e-9"""
    emul.emul_glcm_solve_window_cls.restype = C.c_double
    emul.emul_glcm_lanczos_axis.restype = C.c_double
    slots = slot_angles()
    rng = np.random.default_rng(11)
    worst = {"dense": 0.0, "lanczos": 0.0, "lanczos_small": 0.0}
    count = {"dense": 0, "lanczos": 0, "lanczos_small": 0}
    wins = [random_window(rng, it) for it in range(1500)] + adversarial_windows()
    for w in wins:
        p = w.ctypes.data_as(C.c_void_p)
        for s, a in enumerate(slots):
            ref, n = mcc_angle_numpy(w, a)
            if ref is None:
                continue
            d = emul.emul_glcm_solve_window_cls(p, s, 32, -1)
            if n > 12 and s > 2:
                assert d == 1.0 and abs(ref - 1.0) < 1e-12            # a tree: bipartite
                continue
            if n == 19:
                assert d == 1.0 and abs(ref - 1.0) < 1e-12
                continue
            key = "dense" if n <= 12 else "lanczos"
            worst[key] = max(worst[key], abs(d - ref)); count[key] += 1
            if s <= 2 and n <= 18:
                # the Lanczos solver itself on ANY size (padded nodes, breakdowns), with the strided shared-memory layout
                perm = {2: (0, 1, 2), 1: (0, 2, 1), 0: (1, 2, 0)}[s]        # window axes (z,y,x) -> canonical (a,b,c)
                wp = np.ascontiguousarray(w.reshape(3, 3, 3).transpose(perm).reshape(27))
                nout = C.c_int(0)
                N = 14 if n <= 14 else 16 if n <= 16 else 18
                lz = emul.emul_glcm_lanczos_axis(wp.ctypes.data_as(C.c_void_p), N, 128, 77, C.byref(nout))
                assert nout.value == n
                if n > 12:
                    assert lz == d                                          # layout-independent, same code as the dispatcher
                for N2 in (16, 18):                                         # a larger size template: same value (a task's size
                    if N2 > N:                                              # class fixes its template on the device: no top-up)
                        assert abs(emul.emul_glcm_lanczos_axis(wp.ctypes.data_as(C.c_void_p), N2, 1, 0, C.byref(nout)) - lz) < 1e-12
                        # ... and the SAME BITS in the task-sized build that topped-up batches would need
                        assert emul_dyn.emul_glcm_lanczos_axis(wp.ctypes.data_as(C.c_void_p), N2, 1, 0, C.byref(nout)) == \
                            emul_dyn.emul_glcm_lanczos_axis(wp.ctypes.data_as(C.c_void_p), N, 128, 77, C.byref(nout))
                worst["lanczos_small"] = max(worst["lanczos_small"], abs(lz - ref)); count["lanczos_small"] += 1
    assert count["dense"] > 3000 and count["lanczos"] > 150 and count["lanczos_small"] > 1000, count
    assert worst["dense"] < 1e-9, worst
    assert worst["lanczos"] < 1e-9, worst
    assert worst["lanczos_small"] < 1e-9, worst


def test_phaseA_graph_scan_against_bruteforce(emul):
    """glcm_graph_scan (one breadth-first sweep over class masks: connected? bipartite?) on the level graphs of random /
    structured / holed windows, all 13 angles"""
    slots = slot_angles()
    rng = np.random.default_rng(5)
    seen = {(c, b): 0 for c in (0, 1) for b in (0, 1)}
    for it in range(8000):
        w = random_window(rng, it)
        a = slots[it % 13]
        prs = [(i * 9 + j * 3 + k, (i + a[0]) * 9 + (j + a[1]) * 3 + k + a[2]) for i in range(3) for j in range(3) for k in range(3)
               if 0 <= i + a[0] < 3 and 0 <= j + a[1] < 3 and 0 <= k + a[2] < 3]
        dsh = prs[0][1] - prs[0][0]
        adj = {}
        for pa, pb in prs:
            if w[pa] and w[pb]:
                adj.setdefault(int(w[pa]), set()).add(int(w[pb])); adj.setdefault(int(w[pb]), set()).add(int(w[pa]))
        if not adj:
            continue
        selfpair = any(u in vs for u, vs in adj.items())
        start = int(w[min(pa for pa, pb in prs if w[pa] and w[pb])])          # the sweep starts at the lowest pair end
        col = {start: 0}; st = [start]; bip = not selfpair
        while st:
            u = st.pop()
            for v in adj[u]:
                if v not in col:
                    col[v] = 1 - col[u]; st.append(v)
                elif col[v] == col[u]:
                    bip = False
        conn = len(col) == len(adj)
        lo = sum(1 << pa for pa, _ in prs)
        r = emul.emul_glcm_graph_scan(w.ctypes.data_as(C.c_void_p), dsh, C.c_uint32(lo), int(selfpair))
        assert bool(r & 2) == conn, (w, a)
        if conn:
            assert bool(r & 1) == bip, (w, a)
        seen[(int(conn), int(bip and conn))] += 1
    assert seen[(1, 1)] > 100 and seen[(1, 0)] > 500 and seen[(0, 0)] > 500, seen


@pytest.mark.parametrize("kind", ["uniform", "smooth", "uniform200", "twolevel"])
def test_glrlm_glszm_gldm_ngtdm_fast_math_equals_generic_math_on_host(emul, kind):
    """the r=1 bitmask fast paths (csrc/glrlm_fast.cuh, small_fast.cuh) against the generic entry-list kernels' math on a
    22^3 volume with holes (ragged windows, dropped GLRLM angles)"""
    rng = np.random.default_rng(3)
    shape = (22, 22, 22)
    Ng = 32
    if kind == "uniform":
        lev = rng.integers(1, 33, shape)
        lev[rng.random(shape) < 0.1] = 0
    elif kind == "uniform200":                        # every window all-singleton levels (the bulk path of GLRLM / GLSZM)
        Ng = 200
        lev = rng.integers(1, 201, shape)
        lev[rng.random(shape) < 0.05] = 0
    elif kind == "twolevel":                          # no singleton at all: two levels in big zones / long runs, sparse holes
        zz, yy, xx = np.meshgrid(*[np.arange(s) for s in shape], indexing="ij")
        lev = 1 + ((zz // 3 + yy // 2 + xx // 4) % 2) * 6
        lev[rng.random(shape) < 0.03] = 0
    else:
        zz, yy, xx = np.meshgrid(*[np.arange(s) for s in shape], indexing="ij")
        f = np.sin(zz / 2.7) + np.cos(yy / 3.1) + np.sin(xx / 2.3 + 1) + 0.25 * rng.normal(size=shape)
        lev = np.digitize(f, np.quantile(f, np.linspace(0, 1, 33)[1:-1])) + 1
        lev[5:9, 3:20, 7] = 0
        lev[12, :, :] = 0                         # a plane of holes: windows that lose whole GLRLM angles
    lev = np.ascontiguousarray(lev, dtype=np.uint16)
    s = _lib.make_settings(Ng, Ng)
    Zs, Ys, Xs = shape
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for cid, cname in enumerate(_lib.CLASSES):
        if cname == "glcm":
            continue
        nf = len(NAMES[cname])
        fast, gen = np.zeros((nf, Zs, Ys, Xs)), np.zeros((nf, Zs, Ys, Xs))
        if cname == "glrlm":
            assert emul.emul_glrlm_fast(p(lev), Zs, Ys, Xs, C.byref(s), p(fast)) == 0
        else:
            assert emul.emul_small_fast(cid, p(lev), Zs, Ys, Xs, C.byref(s), p(fast)) == 0
        assert emul.emul_voxel_features(cid, p(lev), None, Zs, Ys, Xs, C.byref(s), None, p(gen)) == 0
        for k, f in enumerate(NAMES[cname]):
            assert np.allclose(fast[k], gen[k], rtol=1e-10, atol=1e-12, equal_nan=True), (cname, f, np.nanmax(np.abs(fast[k] - gen[k])))
