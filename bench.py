#!/usr/bin/env python
"""bench.py -- voxels/s of full-texture-suite voxel-based extraction (BASELINE.json metric, config 3).

A "step" is one pass of the hot path over the whole synthetic 512^3 volume: GLCM + GLRLM + GLSZM + GLDM + NGTDM fused
kernels -> 75 float64 feature maps (reference dtypes), kernelRadius 1, Ng 32.
  value  : device-resident (levels in HBM -> maps in HBM), CUDA events, max over ranks
  e2e    : the same through the reference-facing PLUGIN call with HOST buffers: raw int16 image + mask ->
           Radiomics{GLCM,GLRLM,GLSZM,GLDM,NGTDM}(image, mask, voxelBased=True, binWidth=25).execute() -> 75 float64
           host maps (H2D, discretisation, kernels, D2H inside the timed region)
  N > 1  : the volume is split into z-slabs, one per GPU ("strong" scaling); the device-timed step exchanges the halo
           planes with NCCL send/recv and all-reduces the GLCM alive-angle mask; the e2e step hands every rank the whole
           host image (bin edges / gray levels of the whole ROI) and each rank returns its slab of the maps
  parity_sample : OUTSIDE the timed region, >= 20 000 random centre voxels (a quarter of them on the volume's faces, edges
           and corners) of the produced maps against the CPU oracle (oracle/: the compiled reference `_cmatrices` +
           the numpy feature restatement) at the north-star tolerance 1e-5; `deterministic`: the step is run twice more
           and every map compared bit for bit
  secondary : the smooth volume (same metric), config 2 (GLCM-only 256^3), config 4 (wavelet + LoG -> bin -> suite,
           12 images at 512^3) and config 5(ii) (batch of 64 independent 256^3 cases, segment-based suite, sharded by case)
  --impl reference : the reference's own CPU path (compiled `_cmatrices` from oracle/_ref for the matrices + the numpy
           feature restatement) on the host cores, bounded voxel sample per step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

# algorithmic bytes per voxel with the reference dtypes (SURVEY.md 8d): int32 image + bool mask in, 8 B per map out.
# (The timed device-resident path reads a 1-byte packed level volume instead of the 5 B: < 1 % of the figure.)
ALG_BYTES = {"glcm": 5 + 8 * 24, "glrlm": 5 + 8 * 16, "glszm": 5 + 8 * 16, "gldm": 5 + 8 * 14, "ngtdm": 5 + 8 * 5}
CLASSES = ("glcm", "glrlm", "glszm", "gldm", "ngtdm")
METRIC = "voxels/s full-texture voxel-based"
RTOL, ATOL = 1e-5, 1e-9
# --dump-outputs: 75 float64 maps at 100 000 sampled voxels = 60 MB, within the 64 MB a dump may take
DUMP_VOXELS, DUMP_SEED = 100_000, 7


def synth_volume(n, kind):
    """SURVEY.md section 8(d): iid uniform levels 1..32 (seed 0), or the smooth variant."""
    rng = np.random.default_rng(0)
    if kind == "uniform":
        return rng.integers(1, 33, (n, n, n), dtype=np.int32)
    import scipy.ndimage as ndi
    f = ndi.gaussian_filter(rng.standard_normal((n, n, n), dtype=np.float32), 3.0)
    q = np.quantile(f.ravel()[:: max(1, f.size // 2000000)], np.linspace(0, 1, 33)[1:-1])
    return (np.digitize(f, q) + 1).astype(np.int32)


def raw_from_levels(lev):
    """what a scanner would hand over: int16 intensities that binWidth=25 discretises back to `lev` (SURVEY.md 8d)"""
    return ((lev.astype(np.int32) - 1) * 25 + 3).astype(np.int16)


def sample_voxels(n, count, seed):
    """random centre voxels [3, count]; every fourth one is pushed onto a face / edge / corner of the volume"""
    rng = np.random.default_rng(seed)
    vox = rng.integers(0, n, (3, count)).astype(np.int32)
    b = np.arange(count) % 4 == 0
    for d in range(3):
        on = b & (rng.random(count) < 0.6)
        vox[d, on] = np.where(rng.random(int(on.sum())) < 0.5, 0, n - 1)
    return vox


# ----------------------------------------------------------------------------------- CPU arm
_CPU = {}
# the CPU arm is the reference's compiled C for the matrices but the numpy RESTATEMENT for the features (the reference's
# Python feature classes need SimpleITK / pywt, absent here and on the GPU box): labelled "port", the weaker claim
CPU_ARM_DETAIL = {"reference": "matrices: the unmodified reference _cmatrices compiled from /root/reference (oracle/_ref); "
                               "features: numpy restatement oracle/features_np.py",
                  "port": "matrices: C restatement oracle/cmatrices_port.c; features: numpy restatement oracle/features_np.py"}


def _cpu_worker(args):
    """full suite (matrices + features) for a list of centre voxels, reference-style dense path"""
    import features_np as F
    vox, Ng, levels, keep = args
    img, msk, cm = _CPU["img"], _CPU["msk"], _CPU["cm"]
    d1 = np.array([1])
    t0 = time.perf_counter()
    res = {}
    P, _ = cm.calculate_glcm(img, msk, d1, Ng, False, 0, 1, vox)
    res["glcm"] = F.glcm_features(F.glcm_matrix(P, levels), levels, Ng)
    del P
    P, _ = cm.calculate_glrlm(img, msk, Ng, int(max(img.shape)), False, 0, 1, vox)
    res["glrlm"] = F.glrlm_features(P, levels)
    del P
    res["glszm"] = F.glszm_features(cm.calculate_glszm(img, msk, Ng, int(msk.size), False, 0, 1, vox), levels)
    res["gldm"] = F.gldm_features(cm.calculate_gldm(img, msk, d1, Ng, 0, False, 0, 1, vox), levels)
    res["ngtdm"] = F.ngtdm_features(cm.calculate_ngtdm(img, msk, d1, Ng, False, 0, 1, vox))
    dt = time.perf_counter() - t0
    if not keep:
        return dt, None
    return dt, {c: {k: np.asarray(v, dtype=np.float64) for k, v in r.items()} for c, r in res.items()}


def cpu_arm_setup(vol):
    import build_ref
    try:
        cm, kind = build_ref.load(), "reference"
    except ImportError:
        import cmatrices_oracle as cm
        kind = "port"
    _CPU.update(img=vol, msk=np.ones(vol.shape, bool), cm=cm)
    return kind


def cpu_arm_step(vol, workers, per_worker, seed, pool, keep=False, batch=96):
    """returns (voxels/s, seconds, voxels [3,M], {class: {feature: array[M]}} or None)"""
    n = vol.shape[0]
    vox = sample_voxels(n, workers * per_worker, seed) if keep else np.random.default_rng(seed).integers(
        0, n, (3, workers * per_worker)).astype(np.int32)
    levels = np.arange(1, 33)
    jobs = []
    for i in range(workers):
        for b0 in range(0, per_worker, batch):          # dense per-voxel matrices: keep the batches small (1.7 MB / voxel for GLRLM)
            lo, hi = i * per_worker + b0, i * per_worker + min(b0 + batch, per_worker)
            jobs.append((np.ascontiguousarray(vox[:, lo:hi]), 32, levels, keep))
    t0 = time.perf_counter()
    out = [_cpu_worker(j) for j in jobs] if pool is None else pool.map(_cpu_worker, jobs, chunksize=1)
    dt = time.perf_counter() - t0
    feats = None
    if keep:
        feats = {c: {k: np.concatenate([o[1][c][k] for o in out]) for k in out[0][1][c]} for c in CLASSES}
    return workers * per_worker / dt, dt, vox, feats


def run_reference(args):
    """--impl reference: rank 0 only; other ranks exit quietly."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import multiprocessing as mp
    vol = synth_volume(args.size, args.kind)
    kind = cpu_arm_setup(vol)
    cores = min(os.cpu_count() or 1, args.cpu_workers)
    # bounded sample per step, sized so that the whole run stays within a few minutes whatever --steps is: at most
    # ~8 x cpu_voxels_per_worker voxels per worker over all timed steps (the rate does not depend on the batch size)
    per_worker = max(16, min(args.cpu_voxels_per_worker, (8 * args.cpu_voxels_per_worker) // max(1, args.steps)))
    pool = mp.get_context("fork").Pool(cores) if cores > 1 else None
    for w in range(args.warmup):
        cpu_arm_step(vol, cores, max(8, per_worker // 8), 100 + w, pool)
    t0 = time.perf_counter()
    nvox = 0
    for k in range(args.steps):
        cpu_arm_step(vol, cores, per_worker, k, pool)
        nvox += cores * per_worker
    total = time.perf_counter() - t0
    if pool:
        pool.close()
    value = nvox / total
    sample = f"{cores * per_worker} random centre voxels of the {args.size}^3 volume per step, batches of {per_worker}"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "voxels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, args.steps),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "voxels/s", "cores": cores,
                         "kind": "port", "detail": CPU_ARM_DETAIL[kind],
                         "sample": sample},
        "e2e": {"value": value, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args):
    return {"workload": f"full suite GLCM+GLRLM+GLSZM+GLDM+NGTDM voxel-based, synthetic {args.size}^3 Ng=32 "
                        f"kernelRadius=1 ({args.kind} levels), 75 float64 maps",
            "size": args.size, "Ng": 32, "kernelRadius": 1, "levels": args.kind,
            "l2": "inputs+outputs (>=25 GB per class) far exceed the 126 MB L2; no flush needed",
            "parallelism": f"z-slabs x{args.gpus}" if args.gpus > 1 else "single GPU"}


# ----------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 8:
                for k, nm in enumerate(names):
                    if r[4 + k].lower().startswith("active"):
                        reasons.add(nm)
        mx = max((float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------- GPU arm
class Ctx:
    """rank / device / process group of this process"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        assert self.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={self.world}"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def parity_of(outs, z0, vox, feats):
    """sampled oracle comparison of device maps {class: [F, nz, Y, X]} (planes z0.. of the volume)"""
    import torch
    from pyradiomics_b200 import _lib
    nz = next(iter(outs.values())).shape[1]
    sel = (vox[0] >= z0) & (vox[0] < z0 + nz)
    v = torch.from_numpy(vox[:, sel].astype(np.int64)).to(next(iter(outs.values())).device)
    n_fail, max_rel, worst, max_abs_small, nan_mismatch = 0, 0.0, None, 0.0, 0
    for c in outs:
        got = outs[c][:, v[0] - z0, v[1], v[2]].cpu().numpy()
        for k, name in enumerate(_lib.feature_names(c)):
            ref, g = feats[c][name][sel], got[k]
            nan_mismatch += int((np.isnan(ref) != np.isnan(g)).sum())
            ok = np.isclose(g, ref, rtol=RTOL, atol=ATOL, equal_nan=True)
            n_fail += int((~ok).sum())
            with np.errstate(invalid="ignore", divide="ignore"):
                d = np.abs(g - ref)
                big = np.abs(ref) > 1e-6
                if big.any():
                    r = float(np.nanmax(np.where(big, d / np.abs(ref), 0.0)))
                    if r > max_rel:
                        max_rel, worst = r, f"{c}.{name}"
                if (~big).any():
                    max_abs_small = max(max_abs_small, float(np.nanmax(np.where(~big, d, 0.0))))
    return {"n": int(sel.sum()), "features": sum(len(feats[c]) for c in outs), "max_rel": max_rel, "worst_feature": worst,
            "max_abs_where_ref_below_1e-6": max_abs_small, "n_outside_tolerance": n_fail, "nan_mismatch": nan_mismatch,
            "rtol": RTOL, "atol": ATOL, "ok": n_fail == 0 and nan_mismatch == 0,
            "oracle": "oracle/_ref compiled reference _cmatrices + oracle/features_np.py"}


def dump_outputs(ctx, outs, z0, n, out_dir):
    """--dump-outputs: the maps {class: [F, nz, Y, X]} of the last timed step at a fixed, seeded sample of voxels of the n^3
    volume (the same sample for every run with the same --size) -> out_dir/<class>.npy, float64 [F, voxels]; every rank
    contributes the voxels of its slab, rank 0 writes"""
    import torch
    vox = torch.from_numpy(sample_voxels(n, min(DUMP_VOXELS, n ** 3), DUMP_SEED).astype(np.int64)).to(ctx.dev)
    nz = next(iter(outs.values())).shape[1]
    mine = (vox[0] >= z0) & (vox[0] < z0 + nz)
    zl = (vox[0] - z0).clamp(0, nz - 1)
    if ctx.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
    for c, t in outs.items():
        s = torch.where(mine, t[:, zl, vox[1], vox[2]], 0.0)
        if ctx.world > 1:
            ctx.dist.all_reduce(s)
        if ctx.rank == 0:
            np.save(os.path.join(out_dir, f"{c}.npy"), s.cpu().numpy())


def measure_suite(ctx, vol, steps, warmup, classes=CLASSES, oracle=None, check_determinism=True, sample_clocks=False,
                  dump_dir=None):
    """device-resident timing of the fused kernels over `vol` (levels), z-slabs over the ranks"""
    import torch
    from pyradiomics_b200 import _lib, distributed as D, voxel
    dev, rank, world = ctx.dev, ctx.rank, ctx.world
    Z = vol.shape[0]
    z0, z1 = D.slab_range(Z, rank, world)
    r = 1
    settings = _lib.make_settings(32, 32)
    own = torch.from_numpy(vol[z0:z1].astype(np.uint8)).to(dev)
    slab = D.SlabHalo(own, r, rank, world)
    nz = z1 - z0
    outs = {c: torch.empty((_lib.lib().rb_num_features(_lib.CLASS_ID[c]), nz) + vol.shape[1:], dtype=torch.float64, device=dev)
            for c in classes}
    ev = {c: [] for c in classes}
    launches = [0]
    zchunk = max(1, (48 << 20) // (vol.shape[1] * vol.shape[2] * 13))
    glcm_chunks = -(-nz // zchunk)
    # kernels per plane chunk of a GLCM call: phase A, the eigen-solve kernels (one launch per size group where that is the
    # default: voxel_fast.cu GF_SOLVE_SPLIT = 3 -> dense <= 8: 1, dense <= 12: 2, Lanczos: 3), finish
    split = int(os.environ.get("B200_GLCM_SPLIT", "3"))
    glcm_per_chunk = 1 + (3 if split & 4 else 1) + (2 if split & 2 else 1) + (3 if split & 1 else 1) + 1

    def step(record):
        slab.exchange()
        buf = slab.buf
        alive = None
        if "glcm" in classes:
            alive = D.allreduce_alive(voxel.glcm_alive_angles(buf, settings), dev)
            launches[0] += 1                                  # glcm_alive_kernel
        for c in classes:
            if record:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            voxel.voxel_features(c, buf, settings, z0=r, z1=r + nz, out=outs[c], out_z0=r, alive=alive)
            launches[0] += glcm_per_chunk * glcm_chunks if c == "glcm" else 1
            if record:
                e1.record()
                ev[c].append((e0, e1))

    for _ in range(warmup):
        step(False)
    ctx.barrier()
    sampler = ClockSampler(ctx.local) if (sample_clocks and rank == 0) else None
    if sampler:
        sampler.start()
    launches[0] = 0
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    s0.record()
    for _ in range(steps):
        step(True)
    s1.record()
    ctx.barrier()
    ms = ctx.max_over_ranks(s0.elapsed_time(s1))
    clocks = sampler.stop() if sampler else None
    per_class_ms = {c: float(np.mean([a.elapsed_time(b) for a, b in ev[c]])) for c in classes}
    res = {"value": float(np.prod(vol.shape)) * steps / (ms * 1e-3), "ms_per_step": ms / steps, "per_class_ms": per_class_ms,
           "launches": launches[0], "clocks": clocks, "nz": nz}
    # ---- outside the timed region: the dumped outputs, bit-reproducibility and the sampled oracle comparison
    if dump_dir is not None:
        dump_outputs(ctx, outs, z0, vol.shape[0], dump_dir)
    if check_determinism:
        same = True
        for c in classes:
            again = torch.empty_like(outs[c])
            alive = D.allreduce_alive(voxel.glcm_alive_angles(slab.buf, settings), dev) if c == "glcm" else None
            voxel.voxel_features(c, slab.buf, settings, z0=r, z1=r + nz, out=again, out_z0=r, alive=alive)
            torch.cuda.synchronize()
            same = same and bool(torch.equal(again.view(torch.int64), outs[c].view(torch.int64)))
            del again
        res["deterministic"] = bool(ctx.sum_over_ranks(0.0 if same else 1.0) == 0.0)
    if oracle is not None:
        res["parity_sample"] = parity_of(outs, z0, oracle[0], oracle[1])
    del outs
    torch.cuda.empty_cache()
    return res


def plugin_e2e(ctx, vol, steps, map_dtype="float64"):
    """end to end through the reference-facing plugin call, host buffers in and out (see module docstring)"""
    import torch
    from pyradiomics_b200 import distributed as D, featureclasses as FC
    raw = raw_from_levels(vol)
    mask = np.ones(vol.shape, np.uint8)
    Z = vol.shape[0]
    z0, z1 = D.slab_range(Z, ctx.rank, ctx.world)
    kw = dict(voxelBased=True, binWidth=25, b200_map_dtype=map_dtype)
    if ctx.world > 1:
        kw["b200_zrange"] = (z0, z1)
    step_no = [0]

    phases = {}

    def one():
        FC.clear_device_cache()                    # every step pays the H2D + discretisation of its image
        step_no[0] += 1
        # the five classes of one extraction name their image like an extractor would (its sha1 is in the diagnostics):
        # the first class uploads and bins, the other four find it by that key instead of re-hashing 400 MB each
        kw["b200_image_key"] = ("bench", map_dtype, step_no[0])
        maps = {}
        for k, c in enumerate(("gldm", "glszm", "glrlm", "ngtdm", "glcm")):
            ta = time.perf_counter()
            obj = FC.FEATURE_CLASSES[c](raw, mask, **kw)
            tb = time.perf_counter()
            maps[c] = obj.execute()
            tc = time.perf_counter()
            if k == 0:
                phases["image_h2d_bin"] = phases.get("image_h2d_bin", 0.0) + (tb - ta)
            phases[c] = phases.get(c, 0.0) + (tc - tb)
        return maps

    m = one()                                        # warm-up: faults the page-locked blocks in, builds the tables
    phases.clear()
    nmaps = sum(len(v) for v in m.values())
    probe = float(np.asarray(next(iter(m["glcm"].values())).array).ravel()[0])
    del m
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        m = one()
        del m
    torch.cuda.synchronize()
    dt = ctx.max_over_ranks((time.perf_counter() - t0) / steps)
    esz = 8 if map_dtype == "float64" else 4
    d2h = ctx.sum_over_ranks(float(nmaps * (z1 - z0) * vol.shape[1] * vol.shape[2] * esz))
    h2d = ctx.sum_over_ranks(float(raw.nbytes + mask.nbytes))
    return {"value": float(np.prod(vol.shape)) / dt, "unit": "voxels/s", "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(d2h), "ms_per_step": dt * 1e3, "steps": steps, "maps": nmaps, "map_dtype": map_dtype,
            "d2h_gb_per_s_per_rank": d2h / ctx.world / dt / 1e9, "first_value_probe": probe,
            "phases_ms_rank0": {k: round(1e3 * v / steps, 2) for k, v in phases.items()},
            "scaling": "strong: ONE image per step, its z-slabs on the N GPUs" if ctx.world > 1 else "one image on one GPU",
            "api": "pyradiomics_b200.featureclasses.Radiomics{GLCM,GLRLM,GLSZM,GLDM,NGTDM}(raw int16 image, mask, voxelBased=True, "
                   "binWidth=25, b200_image_key=<step id>).execute(): H2D, discretisation once per image, fused kernels, chunked D2H into "
                   "page-locked maps; N > 1: every rank gets the whole host image and returns its z-slab (b200_zrange); max over ranks"}


def secondary_config2(ctx, kinds=("uniform", "smooth")):
    """BASELINE.json config 2: GLCM feature maps only, 256^3"""
    out = {}
    for kind in kinds:
        vol = synth_volume(256, kind)
        r = measure_suite(ctx, vol, 5, 3, classes=("glcm",), check_determinism=False)
        out[kind] = {"value": r["value"], "unit": "voxels/s", "ms_per_step": r["ms_per_step"],
                     "algorithmic_GBps": ALG_BYTES["glcm"] * r["value"] / 1e9}
    return {"workload": "GLCM-only voxel-based feature maps, synthetic 256^3 Ng=32 kernelRadius=1, 24 float64 maps", **out}


def secondary_config4(ctx, n):
    """BASELINE.json config 4: wavelet (8 sub-bands) + LoG (sigma 1,2,3) + original -> binWidth 25 -> full suite.  N > 1: the
    volume is sharded into z-slabs; the wavelet gets a ring-closed periodic halo, the LoG z pass runs on y-slabs between two
    transpositions, bin edges come from the all-reduced ROI min / max (pipeline.voxel_suite_with_filters_slab)"""
    import torch
    from pyradiomics_b200 import distributed as D, pipeline as PL
    g = torch.Generator(device=ctx.dev).manual_seed(0)               # every rank builds the same volume, keeps its slab
    x = torch.randn((n, n, n), generator=g, device=ctx.dev, dtype=torch.float32)
    k = torch.tensor([np.exp(-0.5 * (i / 2.0) ** 2) for i in range(-6, 7)], device=ctx.dev)
    k = (k / k.sum()).to(torch.float32)
    for ax in range(3):                                  # separable Gaussian smoothing, sigma 2 (SURVEY.md 8d)
        shape = [1, 1, 1, 1, 1]
        shape[2 + ax] = 13
        pad = [0, 0, 0]
        pad[ax] = 6
        x = torch.nn.functional.conv3d(x[None, None], k.view(shape), padding=pad)[0, 0]
    x = ((x - x.min()) / (x.max() - x.min()) * 800.0).to(torch.float64)
    z0, z1 = D.slab_range(n, ctx.rank, ctx.world)
    own = x[z0:z1].contiguous()
    del x
    torch.cuda.empty_cache()
    mask = torch.ones(own.shape, dtype=torch.uint8, device=ctx.dev)

    def run(vol, msk, Z):
        if ctx.world == 1:
            return PL.voxel_suite_with_filters(vol, msk, binWidth=25)
        return PL.voxel_suite_with_filters_slab(vol, msk, Z, ctx.rank, ctx.world, binWidth=25)

    if ctx.world == 1:
        run(own[:64, :64, :64].contiguous(), mask[:64, :64, :64].contiguous(), 64)      # warm-up
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    info = run(own, mask, n)
    e1.record()
    ctx.barrier()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    return {"workload": f"original + wavelet coif1 (8) + LoG sigma 1,2,3 -> binWidth 25 -> full suite, synthetic {n}^3 float volume"
                        + (f", z-slabs over {ctx.world} GPUs (periodic wavelet halo, LoG z pass on y-slabs)" if ctx.world > 1 else ""),
            "images": len(info), "ms": ms, "value": len(info) * float(n) ** 3 / (ms * 1e-3), "unit": "voxels/s (image-voxels)",
            "Ng_per_image": {nm: ng for nm, ng, _ in info}, "filter_parity": "unpinned (PyWavelets / SimpleITK absent; DESIGN.md 5)"}


def secondary_config5ii(ctx, ncases=64, n=256):
    """BASELINE.json config 5(ii): batch of independent cases, segment-based full suite, sharded by case, no collective"""
    import torch
    from pyradiomics_b200 import featureclasses as FC
    mine = [k for k in range(ncases) if k % ctx.world == ctx.rank]
    mask = np.ones((n, n, n), np.uint8)

    def case(k):
        g = torch.Generator(device=ctx.dev).manual_seed(1000 + k)
        lev = torch.randint(1, 33, (n, n, n), generator=g, device=ctx.dev, dtype=torch.int16)
        return ((lev - 1) * 25 + 3).cpu().numpy()

    def run(raw, k):
        FC.clear_device_cache()
        # b200_image_key: the case id names the image for the five classes of one case (else each class hashes its content)
        return {c: FC.FEATURE_CLASSES[c](raw, mask, binWidth=25, b200_image_key=("case", k)).execute() for c in CLASSES}

    run(case(ncases), ncases)                           # warm-up
    raws = [case(k) for k in mine]
    ctx.barrier()
    t0 = time.perf_counter()
    nfeat = 0
    for k, raw in zip(mine, raws):
        nfeat = sum(len(v) for v in run(raw, k).values())
    torch.cuda.synchronize()
    dt = ctx.max_over_ranks(time.perf_counter() - t0)
    return {"workload": f"batch of {ncases} independent synthetic {n}^3 cases, segment-based full suite ({nfeat} features per case), "
                        f"cases sharded round-robin over {ctx.world} GPU(s), no collective",
            "cases": ncases, "seconds": dt, "cases_per_s": ncases / dt, "value": ncases * float(n) ** 3 / dt, "unit": "voxels/s",
            "ms_per_case_per_gpu": 1e3 * dt / max(1, len(mine)),
            "api": "Radiomics{GLCM,GLRLM,GLSZM,GLDM,NGTDM}(raw int16 image, mask, binWidth=25, b200_image_key=<case id>).execute() per case "
                   "(host buffers)"}


def run_b200(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    sys.path.insert(0, ROOT)
    from pyradiomics_b200 import numa
    cpus = numa.bind_to_gpu(local) if not args.no_numa_bind else []       # before any page-locked allocation
    vol = synth_volume(args.size, args.kind)
    vol_s = synth_volume(args.size, "smooth") if (not args.no_secondary and args.kind == "uniform") else None

    # ---- CPU oracle legs first (fork-safe: CUDA is not initialised yet): cpu_baseline timing + parity samples
    cpu_baseline, oracle, oracle_s = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import multiprocessing as mp
        cores = min(os.cpu_count() or 1, args.cpu_workers)
        per_worker = -(-args.parity_voxels // cores)
        kind = cpu_arm_setup(vol)
        pool = mp.get_context("fork").Pool(cores) if cores > 1 else None
        cpu_arm_step(vol, cores, 8, 99, pool)
        v, dt, vox, feats = cpu_arm_step(vol, cores, per_worker, 0, pool, keep=True)
        if pool:
            pool.close()
        oracle = (vox, feats)
        cpu_baseline = {"value": v, "unit": "voxels/s", "cores": cores,
                        "kind": "port", "detail": CPU_ARM_DETAIL[kind],
                        "sample": f"{cores * per_worker} random centre voxels (a quarter on faces/edges/corners) of the same "
                                  f"{args.size}^3 volume, full suite matrices+features, {dt:.1f} s wall; the values double as the parity sample"}
        if vol_s is not None:
            cpu_arm_setup(vol_s)
            pool = mp.get_context("fork").Pool(cores) if cores > 1 else None
            _, _, vox_s, feats_s = cpu_arm_step(vol_s, cores, per_worker, 1, pool, keep=True)
            if pool:
                pool.close()
            oracle_s = (vox_s, feats_s)

    ctx = Ctx(args)
    main = measure_suite(ctx, vol, args.steps, args.warmup, oracle=oracle, sample_clocks=True, dump_dir=args.dump_outputs)
    value, per_class_ms, nz = main["value"], main["per_class_ms"], main["nz"]
    Z = args.size

    # roofline of the dominant kernel group (longest class), algorithmic bytes / event time
    dom = max(per_class_ms, key=per_class_ms.get)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = ALG_BYTES[dom] * (nz * Z * Z) / (per_class_ms[dom] * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        if prof.get("kernel_class") == dom and prof.get("voxels"):
            traffic = prof["dram_bytes_per_launch"] * (nz * Z * Z) / prof["voxels"]
            traffic_src = "profiles/roofline_traffic.json: ncu dram bytes of one plane chunk, scaled by voxels (%.0f B/voxel)" % (
                prof["dram_bytes_per_launch"] / prof["voxels"])
    except (OSError, ValueError, KeyError):
        pass
    roofline = {"bound": "hbm", "kernel": f"{dom} fused voxel kernels", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "ms_per_launch": per_class_ms[dom], "per_class_ms": per_class_ms,
                "suite_frac": 625.0 * value / ctx.world / 1e9 / peak,
                "note": "issue-bound integer / fp64 kernels, not HBM-bound: see DESIGN.md section 4"}

    e2e = None
    secondary = {}
    if not args.no_e2e:
        e2e = plugin_e2e(ctx, vol, args.e2e_steps)
        if not args.no_secondary:
            f32 = plugin_e2e(ctx, vol, args.e2e_steps, "float32")
            secondary["e2e_float32_maps"] = {k: f32[k] for k in ("value", "unit", "ms_per_step", "d2h_bytes_per_step", "map_dtype",
                                                                 "d2h_gb_per_s_per_rank")}
    if not args.no_secondary:
        if vol_s is not None:
            s = measure_suite(ctx, vol_s, 3, 3, oracle=oracle_s)
            secondary["smooth_volume"] = {
                "workload": workload_config(argparse.Namespace(size=args.size, kind="smooth", gpus=args.gpus))["workload"],
                "value": s["value"], "unit": "voxels/s", "ms_per_step": s["ms_per_step"], "per_class_ms": s["per_class_ms"],
                "deterministic": s.get("deterministic"), "parity_sample": s.get("parity_sample")}
        secondary["config2_glcm_256"] = secondary_config2(ctx)
        secondary["config4_filters_suite"] = secondary_config4(ctx, args.size)
        secondary["config5ii_segment_batch"] = secondary_config5ii(ctx)
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "voxels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args),
            "clocks": main["clocks"], "e2e": e2e, "gpu_launches": main["launches"], "roofline": roofline,
            "cpu_baseline": cpu_baseline, "parity_sample": main.get("parity_sample"),
            "deterministic": main.get("deterministic"), "numa_cpus": len(cpus), "secondary": secondary or None,
        }
        print(json.dumps(line))
    if world > 1:
        ctx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--kind", default="uniform", choices=["uniform", "smooth"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--cpu-workers", type=int, default=64)
    ap.add_argument("--cpu-voxels-per-worker", type=int, default=96)
    ap.add_argument("--parity-voxels", type=int, default=20480)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the feature maps of the last timed step, at a fixed sample of voxels, as DIR/<class>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
