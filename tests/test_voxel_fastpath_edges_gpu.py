"""The fused kernelRadius-1 voxel kernels (csrc/voxel_fast.cu: GLCM phase A -> eigen-task solves -> finish, glrlm_fast_kernel,
small_fast_kernel<GLSZM|GLDM|NGTDM>) at their internal boundaries, against the float64 oracle (oracle/ C port + numpy).

With r = 1 a voxel's maps depend only on its 3x3x3 window, on Ng, on the ROI's gray levels and on the alive GLCM angles.
So the oracle runs on windows gathered from the device's input and tiled at stride 3 (helpers.oracle_at_windows); it
never touches the large volumes.  Every comparison starts at rtol 1e-9 / atol 1e-12."""
from collections import Counter

import numpy as np
import pytest
import scipy.ndimage as ndi
import torch

import cmatrices_oracle as O
from helpers import (adversarial_windows, gather_windows, mcc_angle_numpy, oracle_at_windows, random_window, slot_angles,
                     tile_windows)
from pyradiomics_b200 import _lib, voxel

pytestmark = pytest.mark.gpu
RTOL, ATOL = 1e-9, 1e-12
# The oracle's MCC is the square root of the second eigenvalue of the non-symmetric Q = M^2 (np.linalg.eigvals), good to
# a few 1e-9 absolute (measured on a B200: at most 4.0e-9, test B at Ng = 2); the device MCC is held to 1e-9 against the
# symmetric LAPACK restatement in test A instead.
LOOSE = {"glcm.MCC": (0.0, 1e-7)}


def device_maps(lev, Ng, n_levels, centers=None):
    """maps of all classes of the level volume (0 = outside the ROI) through the device API, and the GLCM angles
    (dz, dy, dx) the device keeps alive"""
    t = torch.as_tensor(np.ascontiguousarray(lev, dtype=np.uint8), device="cuda")
    c = None if centers is None else torch.as_tensor(np.ascontiguousarray(centers, dtype=np.uint8), device="cuda")
    s = _lib.make_settings(Ng, n_levels)
    bits = voxel.glcm_alive_angles(t, s, c)
    ang = O.generate_angles(lev.shape, [1], 0, False, 0)
    alive = {tuple(int(v) for v in a) for k, a in enumerate(ang) if bits[k >> 5] >> (k & 31) & 1}
    maps = {cn: voxel.voxel_features(cn, t, s, centers=c).cpu().numpy() for cn in _lib.CLASSES}
    return maps, alive


def compare(got, ref, what):
    """got {class: [F, N]} against the oracle {class: {feature: [N]}}; returns {class.feature: max abs error}"""
    worst = {}
    for cn, g in got.items():
        for k, f in enumerate(_lib.feature_names(cn)):
            rtol, atol = LOOSE.get(f"{cn}.{f}", (RTOL, ATOL))
            a, b = g[k], ref[cn][f]
            ok = np.isclose(a, b, rtol=rtol, atol=atol, equal_nan=True)
            assert ok.all(), f"{what} {cn}.{f}: {int((~ok).sum())} of {ok.size} differ; first {np.argwhere(~ok)[0]}: " \
                             f"got {a[~ok][0]!r} ref {b[~ok][0]!r}"
            with np.errstate(invalid="ignore"):
                d = np.abs(a - b)
            worst[f"{cn}.{f}"] = float(np.nanmax(d)) if np.isfinite(d).any() else 0.0
    return worst


def at(maps, vox):
    z, y, x = (np.asarray(v) for v in vox)
    return {cn: m[:, z, y, x] for cn, m in maps.items()}


# ---------------------------------------------------------------------------------------------------- A
def test_A_solver_windows_against_oracle_and_lapack():
    """the 1563 windows of the host-emulated eigen-solver test, tiled into one volume, through the device kernels:
    every graph size n = 2..19, more than one tile of 4096 eigen-tasks, every per-size-group solve launch"""
    rng = np.random.default_rng(11)
    wins = np.array([random_window(rng, it) for it in range(1500)] + adversarial_windows())
    lev, cen = tile_windows(wins)
    maps, alive = device_maps(lev, 32, 32)
    got = at(maps, cen)
    roi = wins[:, 13] != 0
    for cn, g in got.items():                    # a block centre outside the ROI is no centre: initValue
        assert (g[:, ~roi] == 0).all(), cn
    wins, got = wins[roi], {cn: g[:, roi] for cn, g in got.items()}
    ref, oracle_alive = oracle_at_windows(wins, 32, np.arange(1, 33))
    assert all(a == alive for a in oracle_alive) and len(alive) == 13
    worst = compare(got, ref, "solver windows")

    # MCC against a LAPACK restatement: the mean over the voxel's non-empty angles of the second largest |eigenvalue| of
    # P / sqrt(px py) (disconnected level graph -> 1, one node -> 0)
    sizes, tasks = Counter(), Counter()
    lapack = np.empty(len(wins))
    for i, w in enumerate(wins):
        vals = []
        for a in slot_angles():
            m, n = mcc_angle_numpy(w, a)
            if n == 0:
                continue
            sizes[n] += 1
            if m is not None and m < 1 - 1e-9:      # connected, not bipartite: an eigen-task of phase B
                tasks[n] += 1
            vals.append(0.0 if n == 1 else 1.0 if m is None else m)
        lapack[i] = np.mean(vals)
    mcc = got["glcm"][_lib.feature_names("glcm").index("MCC")]
    err = np.abs(mcc - lapack)
    assert err.max() < 1e-9, (err.max(), int(err.argmax()))
    # ... and the restatement is the oracle's (np.linalg.eigvals of the non-symmetric Q = M^2 is the less accurate one)
    assert np.abs(ref["glcm"]["MCC"] - lapack).max() < 1e-7
    assert all(sizes[n] > 0 for n in range(2, 20)), sizes
    assert all(tasks[n] > 0 for n in range(3, 19)), tasks            # every dense / Lanczos template gets tasks
    assert min(tasks[n] for n in range(13, 19)) >= 25, tasks
    assert sum(tasks.values()) > 4096, sum(tasks.values())            # several solve tiles
    print(f"\nA: {len(wins)} windows, {sum(tasks.values())} eigen-tasks, MCC vs LAPACK max {err.max():.2e}, "
          f"max abs error {max(worst.values()):.2e} ({max(worst, key=worst.get)})")


# ---------------------------------------------------------------------------------------------------- B
def _ng_volume(Ng, kind):
    rng = np.random.default_rng(Ng)
    shape = (12, 13, 14)
    if kind == "uniform":
        lev = rng.integers(1, Ng + 1, shape)
    else:                                       # levels in [Ng-40, Ng] and one voxel at 1: Ng far above the ROI's level count
        lev = rng.integers(Ng - 40, Ng + 1, shape)
        lev[5, 6, 7] = 1
    lev[0, 0, 0] = Ng
    return lev


@pytest.mark.parametrize("Ng,kind", [(1, "uniform"), (2, "uniform"), (3, "uniform")] +
                         [(n, k) for n in (127, 128, 200, 255) for k in ("uniform", "high")])
def test_B_level_count_extremes(Ng, kind):
    """the per-Ng tables (csrc/glcm_fast.cuh: idmn / idn by |i-j|, pair keys with a+b >= 256) up to the 8-bit limit;
    Ng = 200 / 255 uniform make every level a singleton in every window"""
    lev = _ng_volume(Ng, kind)
    levels = np.unique(lev)
    maps, alive = device_maps(lev, Ng, len(levels))
    vox = np.array(np.where(lev != 0))
    if len(levels) > 32:
        # the oracle's MCC is one dense eigvals of an n x n matrix per (voxel, angle): the 8 corners and a random sample
        rng = np.random.default_rng(1)
        corners = np.array(np.meshgrid(*[[0, s - 1] for s in lev.shape], indexing="ij")).reshape(3, -1)
        vox = np.concatenate([corners, vox[:, rng.choice(vox.shape[1], 32 if len(levels) > 64 else 392, replace=False)]], 1)
    ref, oracle_alive = oracle_at_windows(gather_windows(lev, vox), Ng, levels, batch=min(200, max(8, (256 << 20) // (Ng * Ng * 13 * 8))))
    assert all(a == alive for a in oracle_alive)
    worst = compare(at(maps, vox), ref, f"Ng={Ng} {kind}")
    print(f"\nB Ng={Ng} {kind}: {vox.shape[1]} voxels, max abs error {max(worst.values()):.2e} ({max(worst, key=worst.get)})")


# ---------------------------------------------------------------------------------------------------- C
def _degenerate_cases():
    rng = np.random.default_rng(5)
    out = []
    # (15, 17, 1): windows of one level in the generic NGTDM kernel, where i*p_i - j*p_j must be an exact 0 (regression)
    for shape in [(1, 17, 19), (15, 1, 19), (15, 17, 1), (1, 1, 23), (2, 2, 2)]:
        img = rng.integers(1, 7, shape)
        centers = rng.random(shape) < 0.5
        centers.flat[0] = True
        out.append((f"extent{shape}", img, np.ones(shape, bool), centers))
    zz, yy, xx = np.indices((9, 10, 11))
    img = rng.integers(1, 7, (9, 10, 11))
    one = np.zeros(img.shape, bool)
    one[4, 0, 7] = True
    out.append(("one-voxel ROI", img, one, one))          # a flat ROI without any pair: MCC is 1, not NaN (regression)
    cb = (zz + yy + xx) % 2 == 0
    out.append(("checkerboard", img, cb, cb))                         # no face-neighbour pair in the ROI
    isolated = (zz % 2 == 0) & (yy % 2 == 0) & (xx % 2 == 0)          # no neighbour pair at all: every GLCM angle empty
    isolated[3:6, 4:7, 4:7] = True                                    # ... except in one 3x3x3 blob
    out.append(("isolated voxels", img, isolated, isolated))
    return out


@pytest.mark.parametrize("pad", [0, 1], ids=["as-is", "zero-padded"])
@pytest.mark.parametrize("masked", [True, False], ids=["masked-kernel", "centers"])
@pytest.mark.parametrize("name,img,roi,centers", _degenerate_cases(), ids=[c[0] for c in _degenerate_cases()])
def test_C_degenerate_extents_and_masks(name, img, roi, centers, masked, pad):
    """single planes / rows / 2^3 volumes (whole image as ROI) and broken masks, either with the ROI as level volume
    (centers=None) or with the whole image as levels and a separate `centers` mask (maskedKernel=False: for the masks the ROI
    itself, for the extents a random half).  zero-padded: one empty plane on every face, so all 13 / 26 angles exist and the
    fast paths run (an unpadded plane or row has fewer offsets and takes the generic kernel)."""
    if masked:
        lev, centers = np.where(roi, img, 0), None
    else:
        lev, roi = img, centers
    if pad:
        lev, roi = np.pad(lev, 1), np.pad(roi, 1)
        centers = None if centers is None else np.pad(centers, 1)
    levels = np.unique(lev[lev != 0])
    Ng = int(levels.max())
    maps, alive = device_maps(lev, Ng, len(levels), centers)
    vox = np.array(np.where(roi))
    ref, oracle_alive = oracle_at_windows(gather_windows(lev, vox), Ng, levels, batch=vox.shape[1])
    # one oracle call over every centre: its empty-angle drop is the reference's, and the device's alive mask must match
    assert oracle_alive == [alive], (oracle_alive, alive)
    compare(at(maps, vox), ref, name)
    for cn, m in maps.items():                  # outside the ROI: initValue
        assert (m[:, ~roi] == 0).all(), cn


def test_C_single_voxel_volume_has_no_angles():
    """a 1x1x1 volume has no neighbour offset at all: an argument error, like the oracle's (and the reference's)"""
    with pytest.raises(RuntimeError):
        O.generate_angles((1, 1, 1), [1], 0, False, 0)
    t = torch.ones((1, 1, 1), dtype=torch.uint8, device="cuda")
    for cn in _lib.CLASSES:
        with pytest.raises(ValueError):
            voxel.voxel_features(cn, t, _lib.make_settings(1, 1))


# ---------------------------------------------------------------------------------------------------- D + E
SHAPE = (4, 1024, 1024)
HOLES = [(slice(0, 2), slice(100, 140), slice(200, 260)),        # across planes 0 / 1
         (slice(2, 4), slice(300, 340), slice(700, 760)),        # across the chunk seam, planes 2 / 3
         (slice(3, 4), slice(500, 520), slice(0, 30)),           # on the x = 0 face
         (slice(1, 4), slice(1000, 1024), slice(1000, 1024))]    # in the far corner


@pytest.fixture(scope="module")
def big():
    """smooth levels 1..32 (Gaussian-filtered noise, as bench.synth_volume) with zeroed boxes, on the device"""
    rng = np.random.default_rng(0)
    f = ndi.gaussian_filter(rng.standard_normal(SHAPE, dtype=np.float32), 3.0)
    q = np.quantile(f.ravel()[::97], np.linspace(0, 1, 33)[1:-1])
    lev = (np.digitize(f, q) + 1).astype(np.uint8)
    for h in HOLES:
        lev[h] = 0
    vox = _sample(lev, np.random.default_rng(3))
    ref, oracle_alive = oracle_at_windows(gather_windows(lev, vox), 32, np.arange(1, 33))
    yield lev, torch.as_tensor(lev, device="cuda"), vox, ref, oracle_alive
    torch.cuda.synchronize()
    _lib.check(_lib.lib().rb_release_device_caches(), "release")    # the eigen-task queue of this shape is about 1 GB


def test_D_eigen_task_queue_grown_then_reused(big):
    """a small GLCM call, a call that grows the stream's queue, the small call again: bit-identical results"""
    lev40 = torch.as_tensor(np.random.default_rng(2).integers(1, 33, (40, 40, 40)).astype(np.uint8), device="cuda")
    s = _lib.make_settings(32, 32)
    first = voxel.voxel_features("glcm", lev40, s)
    voxel.voxel_features("glcm", big[1], s)
    last = voxel.voxel_features("glcm", lev40, s)
    assert torch.equal(first.view(torch.int64), last.view(torch.int64))


def _sample(lev, rng):
    """>= 3000 ROI voxels: every plane, the x / y faces, edges and corners, the neighbours of the holes"""
    Z, Y, X = lev.shape
    roi = lev != 0
    picks = [np.array(np.where(roi)).T[rng.choice(int(roi.sum()), 2000, replace=False)]]
    for z in range(Z):                          # (planes 0 and 3 are the z faces: their y / x faces are volume edges)
        face = rng.integers(0, [Y, X], (140, 2))
        face[:70, 0] = rng.choice([0, Y - 1], 70)
        face[70:, 1] = rng.choice([0, X - 1], 70)
        corners = np.array([[0, 0], [0, X - 1], [Y - 1, 0], [Y - 1, X - 1]])
        yx = np.concatenate([face, corners])
        picks.append(np.column_stack([np.full(len(yx), z), yx]))
    ring = np.array(np.where(ndi.binary_dilation(~roi, np.ones((3, 3, 3), bool)) & roi)).T
    picks.append(ring[rng.choice(len(ring), 600, replace=False)])
    vox = np.unique(np.concatenate(picks), axis=0)
    vox = vox[roi[tuple(vox.T)]]
    return vox.T


@pytest.mark.parametrize("cname", _lib.CLASSES)
def test_E_chunk_and_grid_stride_boundaries(big, cname):
    """4 x 1024 x 1024: the GLCM call runs plane chunks [0,3) and [3,4), and every chunk is larger than every grid cap of
    the fast kernels (grid-stride loops, phase A, solve tiles).  The whole-volume maps equal the slab calls [0,1), [1,3),
    [3,4) bit for bit, and a sample of >= 3000 voxels (every plane, faces, edges, corners, hole neighbours) equals the
    oracle."""
    lev, dev, vox, ref, oracle_alive = big
    assert (48 << 20) // (SHAPE[1] * SHAPE[2] * 13) == 3                # voxel_fast.cu: glcm_fast_launch's plane chunk
    s = _lib.make_settings(32, 32)
    alive = None
    if cname == "glcm":
        alive = voxel.glcm_alive_angles(dev, s)
        assert all(a == {tuple(int(v) for v in a) for a in O.generate_angles(SHAPE, [1], 0, False, 0)} for a in oracle_alive)
        assert alive[0] == (1 << 13) - 1
    whole = voxel.voxel_features(cname, dev, s, alive=alive)
    parts = torch.cat([voxel.voxel_features(cname, dev, s, z0=a, z1=b, alive=alive) for a, b in ((0, 1), (1, 3), (3, 4))], 1)
    assert torch.equal(whole.view(torch.int64), parts.view(torch.int64))
    del parts
    maps = whole.cpu().numpy()
    del whole
    assert (maps[:, lev == 0] == 0).all()
    assert vox.shape[1] >= 3000 and set(vox[0]) == {0, 1, 2, 3}
    worst = compare({cname: maps[:, vox[0], vox[1], vox[2]]}, ref, f"4x1024x1024 {cname}")
    print(f"\nE {cname}: {vox.shape[1]} voxels, max abs error {max(worst.values()):.2e} ({max(worst, key=worst.get)})")
