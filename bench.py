#!/usr/bin/env python3
"""bench.py -- headline benchmark of the hot path (BASELINE.json): Msamples/s of the Cornell-box-class scene,
1024 x 1024 @ 1024 spp per GPU, `path` integrator, sobol sampler, box reconstruction filter.

    python bench.py --gpus N --steps K --warmup W            # this implementation (one rank per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU code on the host cores
    python bench.py --config c5 --gpus 8                     # BASELINE configs[4] as the headline of the line instead of configs[1]

One "step" = one complete render of the workload (all pixels x all samples of this rank's shard) + the film reduce.
N > 1, headline (`value`): weak scaling -- every rank renders its own 1024 sample indices of every pixel (rank r: [r*1024, (r+1)*1024)
of a 1024*N-spp image), one torch.distributed reduce(SUM) of the (H, W, 5) film over NCCL at the end of every step.  The same line also
carries `strong` (the SAME 1024-spp image split N ways) and `configs` (BASELINE configs[2..4] at their stated sizes, sharded over the N
ranks: c3 material balls 1024^2 @ 512, c4 smoke volume 512^2 @ 256, c5 10 M instanced triangles 2048^2 @ 2048).
`value` = samples rendered by all ranks / max-over-ranks device time.  `e2e` = the same metric through the C-ABI with HOST
buffers: scene description -> b2_scene_commit (BVH build + H2D upload) -> b2_render into a host film (D2H) inside the timed
region.  `parity` = relative L2 of the throughput build's image against the reference's own code (oracle/_ref/libpathref.so) on a
sixteenth of the 32 x 32 blocks at the FULL sample count, computed outside the timed region.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(scene="cornell_box S1 (32 triangles, diffuse + area light)", width=1024, height=1024, spp_per_gpu=1024,
                integrator="path maxDepth=-1 rrDepth=5", sampler="sobol scramble=0", rfilter="box")
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libpathref.so")                 # IEEE-strict build: the one the oracle is pinned against
REF_LIB_REL = os.path.join(ROOT, "oracle", "_ref", "libpathref_relflags.so")    # the reference's own release flags (oracle/Makefile)
REF_FLAGS = {"strict": "-O2 -ffp-contract=off (bit-reproducible against the oracle)",
             "release": "-O3 -march=nocona -msse2 -ftree-vectorize -mfpmath=sse -funsafe-math-optimizations -fno-math-errno -fomit-frame-pointer "
                        "(build/config-linux-gcc.py:7 without -g / -fopenmp / MTS_SSE)"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


def usable_cores():
    """Cores this process may really use: the scheduler affinity mask, cut down to the cgroup CPU quota (a 1-GPU lease of the bench
    pool reports 128 logical CPUs but a cpu.max of 16 cores: 128 worker processes there run on 16 cores' worth of time)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    cores = aff if quota is None else max(1, min(aff, int(math.floor(quota + 1e-6))))
    return cores, {"affinity": aff, "cpu_count": os.cpu_count(), "cgroup_cpu_quota": quota}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------------------
# the reference's own code on the host cores (oracle/_ref, built from /root/reference by oracle/Makefile)
# ------------------------------------------------------------------------------------------------------------------------------
_REF = {}


def bench_scene(name, width, height):
    """Scene description + render parameters of the named BASELINE config (spp filled in by the caller)."""
    from mitsuba_b200.scene import RenderParams, config3_scene, cornell_box, envmap_scene, smoke_scene, stress_scene
    if name == "env":
        return envmap_scene(width, height), dict(sampler="sobol", rfilter="gaussian")
    if name == "c2":
        return cornell_box(width, height), dict(sampler="sobol", rfilter="box")
    if name == "c3":
        return config3_scene(width, height), dict(sampler="sobol", rfilter="box")
    if name == "c4":
        return smoke_scene(width, height, res=128), dict(sampler="independent", rfilter="gaussian", integrator="volpath")
    if name == "c5":
        return stress_scene(100, width=width, height=height, instanced=True), dict(sampler="sobol", rfilter="box")
    raise ValueError(name)


def _ref_worker_init(libpath, name, width, height, spp):
    """One scene per worker process: the reference's own Scene / ShapeKDTree / MIPathTracer or VolumetricPathTracer (oracle/path_ref_shim.cpp)."""
    import ctypes as C
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ref_pins
    from mitsuba_b200.scene import RenderParams
    lib = C.CDLL(libpath)
    d, kw = bench_scene(name, width, height)
    _REF["lib"], _REF["handle"], _REF["shape"] = lib, ref_pins.reference_scene(lib, d, RenderParams(spp=spp, **kw)), (height, width, 5)


def _ref_worker_render(args):
    import ctypes as C
    first, step, want_film = args
    film = np.zeros(_REF["shape"], np.float32)
    _REF["lib"].pathref_render_blocks(_REF["handle"], first, step, film.ctypes.data_as(C.POINTER(C.c_float)))
    return film if want_film else float(film[..., 4].sum())


def reference_cpu_rate(name, width, height, spp, steps=1, warmup=1, cores=0, flags="release"):
    """Msamples/s of the reference's own code on `cores` processes (each renders every cores-th 32 x 32 block with
    SamplingIntegrator::renderBlock), or None where the library is absent."""
    libpath = REF_LIB_REL if flags == "release" and os.path.exists(REF_LIB_REL) else REF_LIB
    if not os.path.exists(libpath) or os.environ.get("B2_BENCH_ORACLE_PORT"):
        return None
    flags = "release" if libpath == REF_LIB_REL else "strict"
    import multiprocessing as mp
    usable, info = usable_cores()
    cores = cores or usable
    with mp.get_context("fork").Pool(cores, initializer=_ref_worker_init, initargs=(libpath, name, width, height, spp)) as pool:
        shares = [(i, cores, False) for i in range(cores)]
        for _ in range(warmup):
            pool.map(_ref_worker_render, shares)
        t0 = time.time()
        for _ in range(steps):
            w = pool.map(_ref_worker_render, shares)
        dt = (time.time() - t0) / max(steps, 1)
    n = width * height * spp
    if abs(sum(w) - n) > 2e-2 * n:  # film weights (gaussian: the border pixels lose a little)
        raise RuntimeError("the shares of the reference render do not add up to the whole image")
    return dict(value=n / dt / 1e6, unit="Msamples/s", cores=cores, kind="reference", ms_per_step=dt * 1e3, per_core=n / dt / 1e6 / cores,
                compiler_flags=REF_FLAGS[flags], cpu_info=info)


PARITY_STEP = 16   # the reference renders every 16th 32 x 32 block of the image at the full sample count


def reference_parity_film(name, width, height, spp):
    """Film of the reference renderer (IEEE-strict build) for the blocks with index = 0 (mod PARITY_STEP) at the FULL sample count,
    plus the mask of their interior pixels (a box-filter sample that falls exactly on a pixel corner spills into the neighbouring
    block, which the subset does not render: the outermost pixel ring of every block is left out of the comparison)."""
    if not os.path.exists(REF_LIB):
        return None
    import multiprocessing as mp
    cores, _ = usable_cores()
    t0 = time.time()
    with mp.get_context("fork").Pool(cores, initializer=_ref_worker_init, initargs=(REF_LIB, name, width, height, spp)) as pool:
        films = pool.map(_ref_worker_render, [(PARITY_STEP * p, PARITY_STEP * cores, True) for p in range(cores)])
    film = np.sum(films, axis=0)
    nbx = (width + 31) // 32
    mask = np.zeros((height, width), bool)
    for by in range((height + 31) // 32):
        for bx in range(nbx):
            if (by * nbx + bx) % PARITY_STEP == 0:
                mask[by * 32 + 1:min(height, by * 32 + 31), bx * 32 + 1:min(width, bx * 32 + 31)] = True
    return dict(film=film, mask=mask, seconds=time.time() - t0, cores=cores)


def parity_entry(ref, film_dev, spp, what):
    from mitsuba_b200 import api
    m = ref["mask"]
    a = api.develop(np.asarray(film_dev))[m].astype(np.float64)
    b = api.develop(ref["film"])[m].astype(np.float64)
    wa, wb = np.asarray(film_dev)[..., 4][m], ref["film"][..., 4][m]
    return {"rel_l2": float(np.sqrt(((a - b) ** 2).sum() / (b ** 2).sum())), "tolerance": 1e-3, "pixels": int(m.sum()), "spp": spp, "workload": what,
            "weights_equal": bool(np.allclose(wa, wb, rtol=1e-5)), "build": "throughput (FMA contraction, --use_fast_math)",
            "against": f"oracle/_ref/libpathref.so (the reference's MIPathTracer / ShapeKDTree / plugins, IEEE-strict flags), every {PARITY_STEP}th 32x32 block at the "
                       f"full sample count, interior pixels; {ref['seconds']:.0f} s on {ref['cores']} host cores"}


def cpu_reference_run(steps, warmup, sample_spp=None, threads=0):
    """The reference on the host cores, on a bounded sample of the SAME workload (`sample_spp` samples of every pixel of the
    1024 x 1024 image): the reference's own sources compiled with its own release flags (and, as a second figure, the IEEE-strict
    build the oracle is pinned against).  Falls back to the oracle port (kind "port") where the libraries are absent."""
    sample_spp = sample_spp or 16
    r = reference_cpu_rate("c2", WORKLOAD["width"], WORKLOAD["height"], sample_spp, steps, max(warmup, 1), threads, "release")
    if r is not None:
        n = WORKLOAD["width"] * WORKLOAD["height"] * sample_spp
        r.update(sample=f"{sample_spp} spp (Sobol', box filter) of every pixel of the 1024x1024 Cornell workload ({n / 1e6:.1f} Msamples per step); the reference's "
                        f"path.cpp / scene.cpp / skdtree.cpp / plugins compiled into oracle/_ref with {r['compiler_flags']}; one process per usable core "
                        f"({r['cores']} = min(affinity {r['cpu_info']['affinity']}, cgroup quota {r['cpu_info']['cgroup_cpu_quota']}))", mean_path_length=None)
        try:
            s = reference_cpu_rate("c2", WORKLOAD["width"], WORKLOAD["height"], sample_spp, 1, 1, threads, "strict")
            if s is not None:
                r["strict_build"] = {"value": s["value"], "per_core": s["per_core"], "compiler_flags": s["compiler_flags"]}
        except Exception:
            pass
        return r
    return cpu_port_run(steps, warmup, sample_spp, threads)


def cpu_port_run(steps, warmup, sample_spp=None, threads=0):
    """The CPU restatement of the reference (oracle, kind "port") on the host cores: a bounded sample of the SAME workload
    (the first `sample_spp` sample indices of every pixel of the 1024 x 1024 image)."""
    from mitsuba_b200.scene import RenderParams, cornell_box
    from oracle import oracle_api as O
    cores = threads or usable_cores()[0]
    d = cornell_box(WORKLOAD["width"], WORKLOAD["height"])
    sc = O.OracleScene(d)
    sample_spp = sample_spp or 4
    rp = RenderParams(spp=WORKLOAD["spp_per_gpu"], sampler="sobol", rfilter="box", sample_lo=0, sample_hi=sample_spp)
    for _ in range(warmup):
        sc.render(rp, threads=cores)
    t0 = time.time()
    st = None
    for _ in range(steps):
        _, st = sc.render(rp, threads=cores)
    dt = (time.time() - t0) / max(steps, 1)
    n = WORKLOAD["width"] * WORKLOAD["height"] * sample_spp
    return dict(value=n / dt / 1e6, unit="Msamples/s", cores=cores, kind="port", per_core=n / dt / 1e6 / cores,
                sample=f"sample indices [0,{sample_spp}) of every pixel of the 1024x1024 @1024spp workload ({n / 1e6:.1f} Msamples per step)",
                ms_per_step=dt * 1e3, mean_path_length=st["pathLengthSum"] / st["samples"])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    r = cpu_reference_run(args.steps, max(args.warmup, 1))
    line = {"impl": "reference", "metric": "Msamples/sec Cornell box 1024spp", "value": r["value"], "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "Cornell box (S1) 1024x1024, path/sobol/box, bounded sample on the host cores", **WORKLOAD},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "per_core", "compiler_flags", "cpu_info", "strict_build") if k in r},
            "e2e": {"value": r["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": ("the reference's own sources (MIPathTracer::Li, renderBlock, Scene, ShapeKDTree, plugins) compiled into oracle/_ref; "
                     "the Mitsuba binary itself (SCons, Boost, Xerces, OpenEXR) cannot be built offline (DESIGN.md)") if r["kind"] == "reference" else
                    "Mitsuba-0.6-equivalent CPU restatement (oracle/), not the Mitsuba binary: the reference cannot be built offline (DESIGN.md)"}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------------------------
# side measurements
# ------------------------------------------------------------------------------------------------------------------------------
def traversal_metric(ctx, hbm_gbs, n_inst=100, n_rays=1 << 22):
    """Second half of BASELINE's metric ("traversal HBM GB/s vs peak"): the closest-hit traversal kernel on the FLATTENED 10 M-triangle
    scene (1.1 GB of nodes + triangles: cannot sit in the 126 MB L2), incoherent rays from the bounding sphere (kdbench-style origins,
    src/utils/kdbench.cpp:222-229) aimed at random mesh vertices.  Reported: Grays/s, the algorithmic bytes the kernel's own counters
    imply, and -- per SURVEY.md 8d -- the DRAM bytes ncu measured for this very launch (profiles/r02_ncu_traversal.json) over the
    live duration."""
    import torch
    from mitsuba_b200 import api
    from mitsuba_b200.scene import stress_scene
    d = stress_scene(n_inst, width=64, height=64)
    t0 = time.time()
    sc = api.Scene(ctx, d)
    commit_s = time.time() - t0
    P = np.concatenate([m.P for m in d.meshes]); lo, hi = P.min(0), P.max(0)
    g = torch.Generator(device="cuda").manual_seed(0)

    def sph():
        v = torch.randn((n_rays, 3), device="cuda", generator=g)
        return v / v.norm(dim=1, keepdim=True)
    c = torch.tensor((lo + hi) / 2, device="cuda", dtype=torch.float32); r = float(np.linalg.norm(hi - lo) / 2)
    Pg = torch.tensor(np.concatenate([m.P for m in d.meshes[:-2]]), device="cuda")
    a = c + r * sph()
    b = Pg[torch.randint(0, len(Pg), (n_rays,), device="cuda", generator=g)]
    dd = b - a; L = dd.norm(dim=1, keepdim=True)
    rays = torch.cat([a, torch.zeros((n_rays, 1), device="cuda"), dd / L, 2 * L], 1).contiguous().float()
    out = torch.zeros((n_rays, 4), device="cuda")
    sc.trace_device(rays, out, n_rays, mode=2)
    st = sc.stats()
    nv, pt = st["node_visits"] / n_rays, st["prim_tests"] / n_rays
    for _ in range(3):
        sc.trace_device(rays, out, n_rays, mode=0)
    ms = min(sc.trace_device(rays, out, n_rays, mode=0) for _ in range(5))
    node_b, tri_b = int(st.get("bvh_node_bytes", 64) or 64), 48
    alg = (48 + node_b * nv + tri_b * pt) * n_rays
    res = {"scene": f"stress {n_inst}x100k = {d.n_triangles()} triangles flattened, {st['n_bvh_nodes']} BVH nodes of {node_b} B", "rays": n_rays,
           "kernel": "k_trace_rays (closest hit)", "mrays_s": n_rays / ms / 1e3, "ms": ms, "node_visits_per_ray": nv, "tri_tests_per_ray": pt,
           "algorithmic_gbs": alg / ms / 1e6, "unit": "GB/s", "peak": hbm_gbs, "algorithmic_frac": alg / ms / 1e6 / hbm_gbs, "commit_s": commit_s}
    tp = os.path.join(ROOT, "profiles", "r02_ncu_traversal.json")
    if os.path.exists(tp):
        try:
            nc = json.load(open(tp))
            res["dram_bytes_per_launch_ncu"] = nc["dram_bytes"]
            res["achieved"] = nc["dram_bytes"] / ms / 1e6   # ncu's DRAM bytes of the same launch over the live duration
            res["frac"] = res["achieved"] / hbm_gbs
            res["lanes_per_instruction_ncu"] = nc.get("lanes_per_instruction")
        except Exception:
            pass
    sc.close()
    return res


def textured_metric(ctx, with_cpu=True):
    """SURVEY.md 8f-4, reported next to the headline: the textured material-ball scene (three `bitmap` textures of 1024^2 texels, EWA
    filtering through ray differentials on camera hits, bilinear on the bounces), `path`, 1024x1024 @ 64 spp on this rank's GPU."""
    from mitsuba_b200 import api
    from mitsuba_b200.scene import RenderParams, textured_scene
    mk = lambda: textured_scene(1024, 1024, filter_type="ewa", tex_res=1024, n_theta=200, n_phi=200)
    sc = api.Scene(ctx, mk())
    rp = RenderParams(spp=64, rfilter="gaussian", sampler="sobol")
    sc.render(RenderParams(spp=4, rfilter="gaussian", sampler="sobol"))
    best = None
    for _ in range(2):
        _, st = sc.render(rp, flags=4)
        if best is None or st["ms_total"] < best["ms_total"]:
            best = st
    n = 1024 * 1024 * 64
    res = {"workload": "S2 material ball, 3 bitmap textures (1024^2, ewa, maxAnisotropy 20), ~80k triangles, path, sobol, gaussian filter, 1024x1024 @ 64 spp, 1 GPU",
           "value": n / best["ms_total"] / 1e3, "unit": "Msamples/s", "ms": best["ms_total"], "kernel": "k_shade<class, TEX> (one launch per BSDF class queue)", "kernel_ms": best["ms_shade"],
           "mean_path_length": best["path_length_sum"] / best["samples"]}
    sc.close()
    return res


def envmap_metric(ctx, with_parity=True):
    """SURVEY.md 8f-3, reported next to the headline: the config-3 material balls lit by a 1024 x 512 environment map only (seen directly with
    the EWA look-up, reflected, refracted, and sampled through its CDF tables), `path`, 1024x1024 @ 64 spp on this rank's GPU; and the film of
    that run against the reference's own EnvironmentMap + MIPathTracer on every 16th block."""
    from mitsuba_b200 import api
    from mitsuba_b200.scene import RenderParams
    d, kw = bench_scene("env", 1024, 1024)
    sc = api.Scene(ctx, d)
    rp = RenderParams(spp=64, **kw)
    sc.render(RenderParams(spp=4, **kw))
    best, film = None, None
    for _ in range(2):
        f, st = sc.render(rp, flags=4)
        if best is None or st["ms_total"] < best["ms_total"]:
            best, film = st, f
    n = 1024 * 1024 * 64
    res = {"workload": "config-3 material balls (GGX conductor + rough dielectric, ~160k triangles) lit by a 1024x512 envmap only (ewa, maxAnisotropy 10), path, sobol, "
                       "gaussian filter, 1024x1024 @ 64 spp, 1 GPU", "value": n / best["ms_total"] / 1e3, "unit": "Msamples/s", "ms": best["ms_total"],
           "kernel": "k_shade<class, TEX> (one launch per BSDF class queue)", "kernel_ms": best["ms_shade"], "mean_path_length": best["path_length_sum"] / best["samples"]}
    if with_parity:
        ref = reference_parity_film("env", 1024, 1024, 64)
        if ref is not None:
            res["parity"] = parity_entry(ref, np.asarray(film).reshape(1024, 1024, 5), 64, "the film of the timed run")
            res["parity"]["build"] = "IEEE kernels (a transmissive BSDF is in the scene: DESIGN.md section 5)"
    sc.close()
    return res


DUMP_BYTES = 64 << 20


def dump_film(out_dir, film):
    """The (H, W, 5) film a caller of the render receives, as out_dir/film.npy.  A film above DUMP_BYTES (2048^2 of c5) is written as
    film_sample.npy instead: the (n, 5) rows of a fixed seeded choice of half the budget's worth of pixels, in raster order, the same for
    every run at that size."""
    os.makedirs(out_dir, exist_ok=True)
    film = np.ascontiguousarray(film, np.float32)
    if film.nbytes <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "film.npy"), film)
        return
    flat = film.reshape(-1, film.shape[-1])
    n = DUMP_BYTES // 2 // flat[0].nbytes
    idx = np.sort(np.random.default_rng(0).choice(len(flat), n, replace=False))
    np.save(os.path.join(out_dir, "film_sample.npy"), flat[idx])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"], help="BASELINE config timed as the headline (default c2 = configs[1])")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="headline scaling mode for N > 1 (c2 only; c3-c5 are always sharded = strong)")
    ap.add_argument("--spp", type=int, default=0, help="samples per pixel (per GPU in weak mode); 0 = the config's own")
    ap.add_argument("--res", type=int, default=0)
    ap.add_argument("--pool", type=int, default=0)
    ap.add_argument("--parity", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the image comparison with the reference's own code")
    ap.add_argument("--no-configs", action="store_true", help="skip the c3 / c4 / c5 side measurements")
    ap.add_argument("--no-volpath", action="store_true", help="(kept for scripts) same as --no-configs")
    ap.add_argument("--no-traversal", action="store_true", help="skip the isolated BVH-traversal measurement (10 M triangles)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the film of the last timed headline step to DIR/film.npy (float32, H x W x 5; above 64 MB a seeded sample of "
                         "its pixels, DIR/film_sample.npy) for output-for-output comparisons")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    args.no_configs = args.no_configs or args.no_volpath
    CONF = {"c2": (1024, 1024), "c3": (1024, 512), "c4": (512, 256), "c5": (2048, 2048)}
    res0, spp0 = CONF[args.config]
    W = H = args.res or res0
    spp_arg = args.spp or spp0
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    weak = args.config == "c2" and args.scaling == "weak"
    full_size = args.config == "c2" and not args.res and not args.spp

    # CPU arms first: the reference renderer forks one process per core, which must happen before this process owns a CUDA context
    cpu_base, ref_c2, ref_c3, vol_cpu = None, None, None, None
    if rank == 0 and world == 1:
        if not args.no_cpu_baseline:
            try:
                cpu_base = cpu_reference_run(1, 1)
            except Exception as e:
                print(f"[bench] reference CPU arm failed ({e}); falling back to the oracle port", file=sys.stderr)
                cpu_base = cpu_port_run(1, 0)
            if not args.no_configs:
                try:
                    vol_cpu = reference_cpu_rate("c4", 512, 512, 8)
                except Exception as e:
                    print(f"[bench] reference CPU arm (volpath) failed: {e}", file=sys.stderr)
        if not args.no_parity and not args.parity and full_size:
            try:
                ref_c2 = reference_parity_film("c2", 1024, 1024, 1024)
                if not args.no_configs:
                    ref_c3 = reference_parity_film("c3", 1024, 1024, 512)
            except Exception as e:
                print(f"[bench] reference parity film failed: {e}", file=sys.stderr)

    import torch
    import torch.distributed as dist
    from mitsuba_b200 import api
    from mitsuba_b200.distributed import shard_range
    from mitsuba_b200.scene import RenderParams

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this implementation has no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = api.Context(local)
    dev = f"cuda:{local}"

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_render(scene, rp, film, steps, warmup, flags=4):
        """`steps` renders (+ film reduce) of this rank's shard; returns (max-over-ranks ms per step, aggregated stats)."""
        def step():
            # the reduce of the previous step may still be reading `film` on torch's stream: order b2_render's stream after it
            torch.cuda.current_stream().synchronize()
            scene.render(rp, parity=bool(args.parity), pool_size=args.pool, flags=flags, film=film)
            if world > 1:
                dist.reduce(film, dst=0, op=dist.ReduceOp.SUM)   # the one collective of the path: film merge over NVLink
            return scene.stats()
        for _ in range(warmup):
            step()
        sync()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        agg = dict(ms_generate=0.0, ms_extend=0.0, ms_shade=0.0, ms_occluded=0.0, n_generate=0, n_extend=0, n_shade=0, n_occluded=0,
                   launches=0, rays=0, shadow_rays=0, path_length_sum=0, samples=0, ms_render=0.0, unoccluded=0, iterations=0)
        ev0.record()
        t_wall = time.time()
        for _ in range(steps):
            st = step()
            for k in ("ms_generate", "ms_extend", "ms_shade", "ms_occluded", "n_generate", "n_extend", "n_shade", "n_occluded", "rays", "shadow_rays",
                      "path_length_sum", "samples", "iterations"):
                agg[k] += st[k]
            agg["unoccluded"] += st["unoccluded_shadow_rays"]
            agg["launches"] += st["kernel_launches"] + (1 if world > 1 else 0)
            agg["ms_render"] += st["ms_total"]
        ev1.record()
        sync()
        agg["wall_s"] = time.time() - t_wall
        # b2_render times itself with CUDA events on ITS stream (torch's events only see torch's stream); each b2_render call synchronises
        # its stream before returning, so the per-step device time = render ms (+ reduce, measured by torch's events)
        ms_total = max(ev0.elapsed_time(ev1), agg["ms_render"])
        t = torch.tensor([ms_total, agg["ms_render"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        agg["ms_render_max"] = float(t[1].item()) / steps
        return float(t[0].item()) / steps, agg

    # ---- headline ----
    desc, kw = bench_scene(args.config, W, H)
    t0 = time.time()
    scene = api.Scene(ctx, desc)
    commit_s = time.time() - t0
    total_spp = spp_arg * world if weak else spp_arg
    lo, hi = shard_range(total_spp, rank, world)
    rp = RenderParams(spp=total_spp, sample_lo=lo, sample_hi=hi, **kw)
    film = torch.zeros((H, W, 5), dtype=torch.float32, device=dev)
    clocks = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        scene.render(rp, parity=bool(args.parity), pool_size=args.pool, flags=4, film=film)
    sync()
    if clocks:
        clocks.start()
    ms_step, agg = timed_render(scene, rp, film, args.steps, 0)
    clock_info = clocks.stop() if clocks else None
    samples_per_step = W * H * total_spp
    value = samples_per_step / (ms_step / 1e3) / 1e6
    pool = scene.stats()["pool_size"]
    film_host = film.cpu().numpy() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_film(args.dump_outputs, film_host)

    # ---- e2e: through the C-ABI with host buffers (scene commit + render into a host film), same metric, same number of steps ----
    host_film = torch.zeros((H, W, 5), dtype=torch.float32).pin_memory()   # the step's result is read back into pinned host memory
    import ctypes as C
    p = api.make_params(rp, bool(args.parity), args.pool, False, 0)

    def e2e_step():
        sc2 = api.Scene(ctx, desc)                                  # b2_scene_create .. b2_scene_commit (H2D upload)
        rc = ctx.L.b2_render(sc2.h, C.byref(p), C.cast(host_film.data_ptr(), C.POINTER(C.c_float)))  # D2H film inside
        if rc:
            raise RuntimeError(ctx.err())
        up = sc2.stats()["bytes_uploaded"]
        sc2.close()
        return up
    e2e_step()
    sync()
    t0 = time.time()
    up = 0
    for _ in range(args.steps):
        up = e2e_step()
    sync()
    tt = torch.tensor([time.time() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e = {"value": samples_per_step * args.steps / float(tt.item()) / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": int(up) + 64,
           "d2h_bytes_per_step": int(H * W * 5 * 4), "steps": args.steps,
           "note": "scene description -> b2_scene_commit (acceleration structure + upload) -> b2_render into pinned host memory, every step"}

    # ---- strong scaling of the headline image (N > 1): the SAME 1024-spp image split N ways ----
    strong = None
    if world > 1 and args.config == "c2":
        slo, shi = shard_range(spp_arg, rank, world)
        rps = RenderParams(spp=spp_arg, sample_lo=slo, sample_hi=shi, **kw)
        ms_s, agg_s = timed_render(scene, rps, film, max(3, min(args.steps, 10)), 2)
        strong = {"value": W * H * spp_arg / (ms_s / 1e3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms_s, "spp_total": spp_arg, "spp_per_gpu": spp_arg / world,
                  "ms_render_max_over_ranks": agg_s["ms_render_max"], "ms_reduce_and_sync": ms_s - agg_s["ms_render_max"],
                  "iterations_per_step": agg_s["iterations"] / max(1, max(3, min(args.steps, 10))),
                  "note": "fixed total work: per-rank render time shrinks with N while the loop's tail (the last paths of the shard draining through "
                          "near-empty iterations) and the 21 MB film reduce do not"}

    # cross-check of the in-kernel %globaltimer stamps: one extra, untimed step with plain launches bracketed by CUDA events
    ev_check = None
    if rank == 0:
        _, stc = scene.render(rp, parity=bool(args.parity), pool_size=args.pool, flags=4 | 8, film=film)
        ev_check = {k: stc["ms_" + k] / max(1, stc["n_" + k]) for k in ("generate", "extend", "shade", "occluded")}
    scene.close()

    # ---- BASELINE configs[2..4] at their stated sizes, sharded over the ranks (side measurements: few steps) ----
    configs = {}
    if not args.no_configs and args.config == "c2" and full_size:
        for name in ("c3", "c4", "c5"):
            try:
                r0, s0 = CONF[name]
                d2, kw2 = bench_scene(name, r0, r0)
                t0 = time.time()
                sc2 = api.Scene(ctx, d2)
                cs = time.time() - t0
                l2, h2 = shard_range(s0, rank, world)
                rp2 = RenderParams(spp=s0, sample_lo=l2, sample_hi=h2, **kw2)
                f2 = torch.zeros((r0, r0, 5), dtype=torch.float32, device=dev)
                ms2, a2 = timed_render(sc2, rp2, f2, 1 if name == "c5" else 2, 1)
                configs[name] = {"workload": {"c3": "material balls: GGX rough conductor + GGX rough dielectric, ~160k triangles, 1024x1024 @ 512 spp, path/sobol/box",
                                              "c4": "smoke: 128^3 gridvolume, heterogeneous (woodcock), isotropic, volpath, independent sampler, gaussian filter, 512x512 @ 256 spp",
                                              "c5": "10 M triangles as 100 instances of a 100k-triangle shapegroup, 2048x2048 @ 2048 spp, path/sobol/box"}[name],
                                 "n_gpus": world, "value": r0 * r0 * s0 / (ms2 / 1e3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms2, "commit_s": cs,
                                 "sharding": f"sample indices split {world} ways, film reduced over NCCL" if world > 1 else "single GPU",
                                 "mean_path_length": a2["path_length_sum"] / max(1, a2["samples"])}
                if name == "c3" and ref_c3 is not None and rank == 0:
                    configs[name]["parity"] = parity_entry(ref_c3, f2.cpu().numpy(), s0, "c3 1024x1024 @ 512 spp")
                if name == "c4" and vol_cpu is not None:
                    configs[name]["cpu_baseline"] = {k: vol_cpu[k] for k in ("value", "unit", "cores", "kind", "per_core", "compiler_flags")}
                sc2.close()
            except Exception as e:  # a side measurement must not take the headline line down with it
                configs[name] = {"error": str(e)}

    if rank == 0:
        peaks, which = measured_peaks()
        shares = {k: agg["ms_" + k] for k in ("generate", "extend", "shade", "occluded")}
        dom = max(shares, key=shares.get)
        n_dom = max(1, agg["n_" + dom])
        avg_ms = shares[dom] / n_dom
        # algorithmic bytes per item of each stage (DESIGN.md section 4, "roofline model"; 16/32-byte pool records)
        rays, shadow, smp = max(1, agg["rays"]), max(1, agg["shadow_rays"]), max(1, agg["samples"])
        per_item = {"extend": 4 + 32 + 16,
                    "occluded": 48 + 16 * agg["unoccluded"] / shadow,
                    "shade": (4 + 16 + 16 + 16 + 8) + (32 + 16 + 4) + 48 * shadow / rays + 4 * smp / rays,
                    "generate": (4 + 4 + 4 + 16 + 8) + 2 * 20 + (32 + 32 + 8 + 8 + 4 + 4)}[dom]
        items = {"extend": rays, "occluded": shadow, "shade": rays, "generate": smp}[dom] / n_dom
        achieved = per_item * items / (avg_ms / 1e3) / 1e9 if avg_ms > 0 else 0.0
        traffic = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("k_" + dom)
            except Exception:
                pass
        line = {
            "metric": "Msamples/sec Cornell box 1024spp" if args.config == "c2" else f"Msamples/sec BASELINE config {args.config}", "value": value, "unit": "Msamples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": (f"Cornell box (S1) {W}x{H} @ {spp_arg} spp per GPU, path/sobol/box (BASELINE configs[1])" if args.config == "c2" else
                                    f"BASELINE {args.config}: {W}x{H} @ {total_spp} spp in total"),
                       **(WORKLOAD if args.config == "c2" else {}), "spp_per_gpu": (hi - lo), "spp_total": total_spp, "width": W, "height": H,
                       "parallelism": f"sample-index sharding x{world}, 1 film reduce", "pool_size": int(pool),
                       "l2": "path pool + film (%.0f MB) exceed the 126 MB L2; every iteration re-streams them" % ((pool * (64 + 16 + 8 + 8 + 8 + 48 + 8) + W * H * 20) / 1e6),
                       "fp": "parity (-fmad=false)" if args.parity else "fast (FMA contraction, --use_fast_math)", "commit_s": commit_s},
            "e2e": e2e,
            "gpu_launches": int(agg["launches"]),
            "clocks": clock_info,
            "roofline": {"bound": "hbm", "kernel": "k_" + dom, "achieved": achieved, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                         "frac": achieved / peaks.get("hbm_gbs", 1.0), "traffic": traffic, "peak_source": which + " (MEASURED_PEAKS.json hbm_gbs)",
                         "avg_launch_ms": avg_ms, "avg_launch_ms_cuda_events": ev_check["" + dom] if ev_check else None,
                         "timer": "%globaltimer stamps inside the kernels (max CTA end - min CTA start per launch), timed region runs as one CUDA graph per iteration; cross-checked by an untimed step with CUDA events around plain launches",
                         "share_of_step": shares[dom] / max(1e-9, sum(shares.values())),
                         "kernel_ms": shares,
                         "note": "Cornell scene (3.5 KB) is shared-memory resident: traversal is issue/latency bound, HBM traffic is queue traffic only"},
            "stats": {"mean_path_length": agg["path_length_sum"] / max(1, agg["samples"]), "rays_per_sample": agg["rays"] / max(1, agg["samples"]),
                      "shadow_rays_per_sample": agg["shadow_rays"] / max(1, agg["samples"]), "wall_s": agg["wall_s"],
                      "iterations_per_step": agg["iterations"] / args.steps},
        }
        if strong is not None:
            line["strong"] = strong
        if ref_c2 is not None and world == 1:
            par = {"c2": parity_entry(ref_c2, film_host, total_spp, "c2 1024x1024 @ 1024 spp (the film of the last timed step)")}
            if "parity" in configs.get("c3", {}):
                par["c3"] = configs["c3"]["parity"]
            line["parity"] = par
        if configs:
            line["configs"] = configs
        if not args.no_traversal:
            try:
                line["traversal"] = traversal_metric(ctx, peaks.get("hbm_gbs", 6650.0))
            except Exception as e:
                line["traversal"] = {"error": str(e)}
        if not args.no_configs and args.config == "c2" and full_size and world == 1:
            try:
                line["textured"] = textured_metric(ctx)
            except Exception as e:
                line["textured"] = {"error": str(e)}
        if not args.no_configs and args.config == "c2" and full_size and world == 1:
            try:
                line["envmap"] = envmap_metric(ctx, with_parity=not args.no_parity)
            except Exception as e:
                line["envmap"] = {"error": str(e)}
        if cpu_base is not None:
            line["cpu_baseline"] = {k: cpu_base[k] for k in ("value", "unit", "cores", "kind", "sample", "per_core", "compiler_flags", "cpu_info", "strict_build") if k in cpu_base}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
