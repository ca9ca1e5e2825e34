#!/usr/bin/env python3
"""Generates tests/golden/* from the reference tree.  Run only in the build container (needs
/root/reference and oracle/_ref/libsobolref.so built by oracle/Makefile):

    make -C oracle && python tests/gen_golden.py

Outputs (committed, so the GPU box and CI never read /root/reference):
  sfmt_kat.json   the 64-bit known-answer words (192) of src/tests/test_random.cpp:436-507 (Random(4321).nextULong())
  sobol_ref.npz   outputs of the REFERENCE's own sobol::sampleSingle / sobol::look_up
                  (src/samplers/sobolseq.h:45-60,104-133, compiled into oracle/_ref) on seeded inputs
  resample_ref.npz  MIP pyramids (every level) of seeded images, computed with the REFERENCE's own Resampler<float>
                  (include/mitsuba/core/rfilter.h:107-449) and LanczosSincFilter (src/rfilters/lanczos.cpp), compiled into
                  oracle/_ref/librfilterref.so, applied the way Bitmap::resample + TMIPMap's constructor apply them
                  (src/libcore/bitmap.cpp:2258-2327 x pass then y pass with clamping to [0, 1]; mipmap.h:246-277 level chain)
  mipmap_ref.npz  texture look-ups of the REFERENCE's own TMIPMap<Color3, Color3>::eval / evalBilinear / evalBox
                  (include/mitsuba/render/mipmap.h:499-838 with the real barray.h / spectrum.h / math.{h,cpp}, compiled into
                  oracle/_ref/libmipmapref.so) over pyramids built by the reference resampler above: seeded uv and footprints
                  (sub-texel, isotropic, needle-shaped beyond maxAnisotropy, zero) for every filter type and wrap mode
  core_ref.npz    outputs of the REFERENCE's own core math on seeded inputs (tests/ref_pins.py): MicrofacetDistribution (src/bsdfs/
                  microfacet.h), TriAccel (triaccel.h), AABB::rayIntersect (aabb.h), warp.cpp, util.cpp (fresnel*, reflect, refract,
                  coordinateSystem, computeShadingFrame), Triangle::sample (triangle.cpp), DiscreteDistribution (pmf.h), sampleTEA
                  (qmc.h) -- compiled into oracle/_ref/libcoreref.so by oracle/Makefile from oracle/core_ref_shim.cpp
  bsdf_ref.npz    eval / pdf / sample (solid-angle and discrete measures) of the REFERENCE's own BSDF plugins -- src/bsdfs/{diffuse,
                  roughconductor,roughdielectric,coating,dielectric,conductor,plastic,twosided}.cpp, instantiated from Properties and
                  called through the real BSDF interface (oracle/bsdf_ref_shim.cpp -> oracle/_ref/libbsdfref.so) -- for the 18
                  configurations of tests/bsdf_configs.py on the seeded directions of tests/ref_pins.py
  render_ref.npz  Intersection::computePartials (src/librender/intersection.cpp), the box / gaussian filter tables of
                  ReconstructionFilter::configure (src/libcore/rfilter.cpp + src/rfilters/*.cpp), ImageBlock::put (imageblock.h) and
                  the SobolSampler plugin's stream (src/samplers/sobol.cpp) -- oracle/render_ref_shim.cpp -> oracle/_ref/librenderref.so
  path_ref.npz    IMAGES rendered by the reference's own code: oracle/path_ref_shim.cpp assembles MIPathTracer (path.cpp),
                  SamplingIntegrator::renderBlock, Scene, ShapeKDTree, TriMesh, the perspective sensor, the area emitter, the Sobol'
                  sampler, the reconstruction filters, ImageBlock and the BSDF plugins from /root/reference into
                  oracle/_ref/libpathref.so.  Cornell box and material-ball scenes (tests/ref_pins.py::image_cases), film (H, W, 5)
                  + the sampleToCamera matrix the reference's sensor derives
"""
import ctypes as C, json, os, re, sys
import numpy as np

REF = os.environ.get("MTS_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "golden")


def sfmt_kat():
    src = open(os.path.join(REF, "src/tests/test_random.cpp")).read()
    m = re.search(r"static const uint64_t reference\[\] = \{(.*?)\};\s*ref<Random> rnd = new Random\((\d+)\)", src, re.S)
    words = [int(h, 16) for h in re.findall(r"0x([0-9a-fA-F]+)ULL", m.group(1))]
    assert len(words) >= 190 and int(m.group(2)) == 4321, (len(words), m.group(2))
    json.dump({"seed": 4321, "source": "src/tests/test_random.cpp:436-507", "words": [f"{w:016x}" for w in words]},
              open(os.path.join(OUT, "sfmt_kat.json"), "w"), indent=0)
    print("sfmt_kat.json:", len(words), "words")


def sobol_ref():
    L = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libsobolref.so"))
    L.sobolref_sample.restype = C.c_float
    L.sobolref_sample.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32]
    L.sobolref_look_up.restype = C.c_uint64
    L.sobolref_look_up.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64]
    rng = np.random.default_rng(20260922)
    n = 4096
    index = np.concatenate([np.arange(64, dtype=np.uint64), rng.integers(0, 1 << 40, n - 64, dtype=np.uint64)])
    dim = np.concatenate([np.arange(64, dtype=np.uint32) % 8, rng.integers(0, 1024, n - 64).astype(np.uint32)])
    scr = np.where(np.arange(n) % 3 == 0, 0, rng.integers(0, 1 << 32, n, dtype=np.uint64)).astype(np.uint32)
    samples = np.array([L.sobolref_sample(int(i), int(d), int(s)) for i, d, s in zip(index, dim, scr)], np.float32)
    m = rng.integers(2, 12, n).astype(np.uint32)
    frame = rng.integers(0, 4096, n).astype(np.uint32)
    px = (rng.integers(0, 1 << 16, n) % (1 << m)).astype(np.uint32)
    py = (rng.integers(0, 1 << 16, n) % (1 << m)).astype(np.uint32)
    scr64 = np.where(np.arange(n) % 2 == 0, 0, rng.integers(0, 1 << 63, n, dtype=np.uint64)).astype(np.uint64)
    lookup = np.array([L.sobolref_look_up(int(a), int(b), int(c), int(d), int(e)) for a, b, c, d, e in zip(m, frame, px, py, scr64)], np.uint64)
    np.savez_compressed(os.path.join(OUT, "sobol_ref.npz"), index=index, dim=dim, scramble=scr, samples=samples,
                        m=m, frame=frame, px=px, py=py, scramble64=scr64, lookup=lookup)
    print("sobol_ref.npz:", n, "samples +", n, "look_ups")


REF_BC = {"clamp": 0, "repeat": 1, "mirror": 2, "zero": 3, "one": 4}  # ReconstructionFilter::EBoundaryCondition, rfilter.h:40-53


def reference_pyramid(img, wrap_u, wrap_v, lib=None):
    """All MIP levels below level 0 of `img` (H, W, C) float32, non-negative, through the reference's compiled Resampler."""
    L = lib or C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "librfilterref.so"))
    fptr = lambda a, off=0: C.cast(a.ctypes.data + off, C.POINTER(C.c_float))
    levels, cur = [], np.ascontiguousarray(img, np.float32)
    while cur.shape[0] > 1 or cur.shape[1] > 1:
        h, w, ch = cur.shape
        nw, nh = max(1, (w + 1) // 2), max(1, (h + 1) // 2)   # mipmap.h:187-189
        src = cur
        if w != nw:  # bitmap.cpp:2258-2293: every row
            tmp = np.zeros((h, nw, ch), np.float32)
            for y in range(h):
                L.rfref_resample(REF_BC[wrap_u], 2, w, nw, fptr(src, y * w * ch * 4), 1, fptr(tmp, y * nw * ch * 4), 1, ch, 1)
            src = tmp
        if h != nh:  # bitmap.cpp:2296-2327: every column (stride = row length)
            out = np.zeros((nh, nw, ch), np.float32)
            for x in range(nw):
                L.rfref_resample(REF_BC[wrap_v], 2, h, nh, fptr(src, x * ch * 4), nw, fptr(out, x * ch * 4), nw, ch, 1)
            src = out
        cur = src
        levels.append(cur)
    return levels


def resample_ref():
    rng = np.random.default_rng(2024)
    out = {}
    k = 0
    for shape in ((32, 32, 3), (37, 50, 3), (21, 13, 1), (1, 9, 1), (16, 1, 3), (5, 64, 1)):
        for wu, wv in (("repeat", "repeat"), ("clamp", "mirror"), ("zero", "one"), ("mirror", "clamp"), ("one", "repeat")):
            img = np.maximum((rng.random(shape) * 1.3 - 0.1).astype(np.float32), 0)  # values above 1 exercise the clamp
            out[f"img{k}"] = img
            out[f"wrap{k}"] = np.array([wu, wv])
            for l, lvl in enumerate(reference_pyramid(img, wu, wv)):
                out[f"lvl{k}_{l + 1}"] = lvl
            k += 1
    out["count"] = np.array(k)
    np.savez_compressed(os.path.join(OUT, "resample_ref.npz"), **out)
    print("resample_ref.npz:", k, "pyramids")


FILTERS = {"nearest": 0, "bilinear": 1, "trilinear": 2, "ewa": 3}  # EMIPFilterType, mipmap.h:52-61


def texture_lookups(rng, n):
    """uv in [-1.5, 2.5]^2; partials (dudx, dudy, dvdx, dvdy): sub-texel to many texels, 30 % needle-shaped, 5 % exactly zero."""
    uv = (rng.random((n, 2)) * 4 - 1.5).astype(np.float32)
    mag = np.float32(10.0) ** rng.uniform(-4, -0.7, (n, 1)).astype(np.float32)
    pt = (rng.normal(size=(n, 4)).astype(np.float32) * mag).astype(np.float32)
    needle = rng.random(n) < 0.3
    pt[needle, 1] *= 0.02; pt[needle, 3] *= 0.02
    pt[rng.random(n) < 0.05] = 0.0
    return uv, pt


def half_inputs(seed=0, n=20000):
    """floats for the float -> half -> float pin: random bit patterns, [0, 2), ties, the denormal range, the overflow edge."""
    rng = np.random.default_rng(seed)
    x = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32).view(np.float32)
    x = x[np.isfinite(x)]
    extra = np.concatenate([rng.random(n).astype(np.float32) * 2, np.arange(0, 70000, 7.25).astype(np.float32), np.float32(2.0) ** np.arange(-30, 17).astype(np.float32),
                            (np.arange(0, 4096) * np.float32(2 ** -25)).astype(np.float32), (1 + np.arange(0, 4096) * np.float32(2 ** -12)).astype(np.float32),
                            np.array([65504, 65519.99, 65520, 65536, 1e30, 0.0, 6.1e-5, 5.96e-8, 2.98e-8, 2.9802322e-08, 8.9e-8], np.float32)])
    return np.concatenate([x, extra, -extra]).astype(np.float32)


def half_store(a):
    """A float array as BitmapTexture's pyramid stores it: TMIPMap<Color3, Color3h> (bitmap.cpp:177-180) rounds every texel to half when a
    level is stored (mipmap.h:226-230, :262-264; half.h:431-487 / half.cpp:78-200 = round to nearest even, overflow to infinity).  That is
    numpy's float16 conversion -- equality with the reference's own half class is pinned by tests/golden/half_ref.npz and, live, on two
    million values (tests/test_oracle_texture.py)."""
    with np.errstate(over="ignore"):
        return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


def half_ref():
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libcoreref.so"))
    x = half_inputs()
    out = np.zeros_like(x)
    lib.coreref_half_round(len(x), x.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data_as(C.POINTER(C.c_float)))
    np.savez_compressed(os.path.join(OUT, "half_ref.npz"), x=x, y=out)
    print("half_ref.npz:", len(x), "values")


class ReferenceMipmap:
    """The reference's TMIPMap over given RGB levels (list of (h, w, 3) float32), via oracle/_ref/libmipmapref.so.  The levels are rounded
    to half first (half_store): BitmapTexture instantiates TMIPMap<Color3, Color3h>, the library TMIPMap<Color3, Color3> -- over
    half-representable texels the two are the same function."""

    def __init__(self, levels, wrap_u, wrap_v, filter_type, max_anisotropy, lib=None):
        self.L = lib or C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libmipmapref.so"))
        self.L.mipref_create.restype = C.c_void_p
        self.levels = [np.ascontiguousarray(half_store(l), np.float32) for l in levels]
        sizes = np.array([[l.shape[1], l.shape[0]] for l in self.levels], np.int32)
        ptrs = (C.POINTER(C.c_float) * len(self.levels))(*[l.ctypes.data_as(C.POINTER(C.c_float)) for l in self.levels])
        aniso = max_anisotropy if filter_type == "ewa" else 1.0  # bitmap.cpp:232-235
        self.h = C.c_void_p(self.L.mipref_create(len(self.levels), sizes.ctypes.data_as(C.POINTER(C.c_int)), ptrs, REF_BC[wrap_u], REF_BC[wrap_v],
                                                 FILTERS[filter_type], C.c_float(aniso)))
        self.filter_type = filter_type

    def eval(self, uv, partials=None):
        """BitmapTexture::eval(uv, d0, d1) (bitmap.cpp:452-465) or, without partials, eval(uv) (bitmap.cpp:400-421)."""
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
        uv = np.ascontiguousarray(uv, np.float32)
        out = np.zeros((len(uv), 3), np.float32)
        if partials is None:
            (self.L.mipref_eval_box if self.filter_type == "nearest" else self.L.mipref_eval_bilinear)(self.h, 0, len(uv), fp(uv), fp(out))
        else:
            d0d1 = np.ascontiguousarray(np.asarray(partials, np.float32)[:, [0, 2, 1, 3]])  # d0 = (dudx, dvdx), d1 = (dudy, dvdy): texture.cpp:127-130
            self.L.mipref_eval(self.h, len(uv), fp(uv), fp(d0d1), fp(out))
        return out


def mipmap_ref():
    rng = np.random.default_rng(4242)
    out, k = {}, 0
    setups = ((("repeat", "repeat"), (40, 61, 3), 20.0), (("clamp", "mirror"), (33, 32, 3), 8.0), (("zero", "one"), (16, 50, 3), 2.0),
              (("mirror", "clamp"), (48, 48, 3), 20.0))
    images = [rng.random(shape).astype(np.float32) for _, shape, _ in setups]
    for j, img in enumerate(images):
        out[f"img{j}"] = img
    for ft in ("nearest", "bilinear", "trilinear", "ewa"):
        for j, ((wu, wv), shape, aniso) in enumerate(setups):
            img = images[j]
            levels = [img] + (reference_pyramid(img, wu, wv) if ft in ("trilinear", "ewa") else [])
            m = ReferenceMipmap(levels, wu, wv, ft, aniso)
            uv, pt = texture_lookups(rng, 600)
            out[f"cfg{k}"] = np.array([ft, wu, wv, str(aniso), str(j)])
            out[f"uv{k}"] = uv; out[f"pt{k}"] = pt
            out[f"filtered{k}"] = m.eval(uv, pt); out[f"unfiltered{k}"] = m.eval(uv)
            k += 1
    out["count"] = np.array(k)
    np.savez_compressed(os.path.join(OUT, "mipmap_ref.npz"), **out)
    print("mipmap_ref.npz:", k, "configurations x 600 look-ups")


def core_ref():
    sys.path.insert(0, HERE)
    import ref_pins
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libcoreref.so"))
    out = ref_pins.run(lib, "coreref_", ref_pins.inputs())
    np.savez_compressed(os.path.join(OUT, "core_ref.npz"), **out)
    print("core_ref.npz:", len(out), "arrays")


def bsdf_ref():
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, ".."))
    import ref_pins
    from bsdf_configs import configs
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libbsdfref.so"))
    x = ref_pins.bsdf_inputs()
    out = {}
    for name, b in configs().items():
        for k, v in ref_pins.run_bsdf_reference(lib, b, x).items():
            out[f"{name}/{k}"] = v
    np.savez_compressed(os.path.join(OUT, "bsdf_ref.npz"), **out)
    print("bsdf_ref.npz:", len(configs()), "BSDF configurations x", ref_pins.NB, "directions")


def render_ref():
    sys.path.insert(0, HERE)
    import ref_pins
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "librenderref.so"))
    out = ref_pins.run_render(lib, "renderref_", ref_pins.render_inputs())
    np.savez_compressed(os.path.join(OUT, "render_ref.npz"), **out)
    print("render_ref.npz:", len(out), "arrays")


def path_ref():
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, ".."))
    import ref_pins
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libpathref.so"))
    out = {}
    for name, desc, rp in ref_pins.image_cases():
        film, s2c = ref_pins.reference_render(lib, desc, rp, want_camera=True)
        out[name + "/film"], out[name + "/s2c"] = film, s2c
    np.savez_compressed(os.path.join(OUT, "path_ref.npz"), **out)
    print("path_ref.npz:", len(out) // 2, "images")


def path_ref_ext():
    """thinlens sensor, constant emitter, shapegroup / instance through the same assembled reference renderer (ref_pins.image_cases_ext);
    per image: the film, the reference's sampleToCamera and its Transform::inverse() of every instance matrix."""
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, ".."))
    import ref_pins
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libpathref.so"))
    out = {}
    n = 0
    for name, desc, rp in ref_pins.image_cases_ext():
        film, s2c = ref_pins.reference_render(lib, desc, rp, want_camera=True)
        out[name + "/film"], out[name + "/s2c"] = film, s2c
        inv = ref_pins.reference_instance_inverses(lib, desc)
        if inv:
            out[name + "/instance_inverses"] = np.stack(inv)
        n += 1
    np.savez_compressed(os.path.join(OUT, "path_ref_ext.npz"), **out)
    print("path_ref_ext.npz:", n, "images")


def path_ref_env():
    """envmap emitter through the same assembled reference renderer (ref_pins.image_cases_env); per image: the film, the reference's
    sampleToCamera and its Transform::inverse() of the map's toWorld."""
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, ".."))
    import ref_pins
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libpathref.so"))
    out = {}
    n = 0
    for name, desc, rp in ref_pins.image_cases_env():
        film, s2c = ref_pins.reference_render(lib, desc, rp, want_camera=True)
        out[name + "/film"], out[name + "/s2c"] = film, s2c
        inv = ref_pins.reference_envmap_inverse(lib, desc)
        if inv is not None:
            out[name + "/env_to_local"] = inv
        n += 1
    np.savez_compressed(os.path.join(OUT, "path_ref_env.npz"), **out)
    print("path_ref_env.npz:", n, "images")


def spectrum_inputs(seed=0, n=200):
    """Random piecewise-linear spectra: 2..60 knots somewhere in 300..900 nm, smooth and spiky, with and without zero extension."""
    rng = np.random.default_rng(seed)
    cases = []
    while len(cases) < n:
        k = len(cases)
        m = int(rng.integers(2, 60)); lo = rng.uniform(300, 500); hi = rng.uniform(550, 900)
        w = np.unique(np.round(np.sort(rng.uniform(lo, hi, m)), 2)).astype(np.float32)
        if len(w) < 2:
            continue
        v = (rng.random(len(w)) ** 2 * rng.uniform(0.1, 5)).astype(np.float32)
        if k % 5 == 0:
            v[rng.integers(len(w))] += np.float32(50)
        cases.append((w, v, int(k % 2)))
    return cases


def spectrum_ref():
    """What the reference's scene loader makes of <spectrum> samples (InterpolatedSpectrum + zeroExtend + Spectrum::fromContinuousSpectrum +
    clampNegative of src/libcore/spectrum.cpp, through oracle/_ref/libpathref.so) for spectrum_inputs(), plus its CIE observer table."""
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libpathref.so"))
    f = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    out = []
    for w, v, ze in spectrum_inputs():
        rgb = np.zeros(3, np.float32)
        assert lib.pathref_spectrum_to_rgb(len(w), f(w), f(v), ze, f(rgb)) == 0
        out.append(rgb)
    t = np.zeros((471, 4), np.float32)
    lib.pathref_cie_tables(f(t))
    np.savez_compressed(os.path.join(OUT, "spectrum_ref.npz"), rgb=np.stack(out), cie=t)
    print("spectrum_ref.npz:", len(out), "spectra")


def path_ref_tex():
    """bitmap textures through the same assembled reference renderer (ref_pins.image_cases_tex): film + the reference's sampleToCamera."""
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, ".."))
    import ref_pins
    lib = C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", "libpathref.so"))
    out = {}
    n = 0
    for name, desc, rp in ref_pins.image_cases_tex():
        film, s2c = ref_pins.reference_render(lib, desc, rp, want_camera=True)
        out[name + "/film"], out[name + "/s2c"] = film, s2c
        n += 1
    np.savez_compressed(os.path.join(OUT, "path_ref_tex.npz"), **out)
    print("path_ref_tex.npz:", n, "images")


RESAMPLE_UNSEEN = (((48, 40, 3), "mirror", "repeat"), ((9, 31, 1), "zero", "clamp"), ((64, 3, 3), "one", "mirror"))
MIPMAP_UNSEEN = (("ewa", "repeat", "mirror", 12.0), ("trilinear", "clamp", "zero", 1.0), ("ewa", "one", "clamp", 3.0))
HALF_UNSEEN = dict(seed=9, n=1_000_000)
BSDF_NOT_BIT_EXACT = ("plastic", "twosided_two")   # the last bit of one constructor constant (tests/test_oracle_reference_pins.py)


def unseen_ref():
    """The reference's answers on inputs the fixtures above do not hold, for the oracle's tests to compare against.  Outputs are kept as
    arrays (unseen_ref.npz), except the large ones compared bit for bit -- core, bsdf, instances, <env>, mipmap, half -- which are kept
    as ref_pins.digest (unseen_ref.json) to keep the fixture small.
      core/*          core math (ref_pins.run) on ref_pins.inputs(seed=99); fresnel_diffuse_reflectance: util.cpp (fast = false) at FDR_ETAS
      bsdf/*          the BSDF plugins on ref_pins.bsdf_inputs(seed=4321) (arrays for BSDF_NOT_BIT_EXACT)
      render/*        partials / filters / ImageBlock::put / Sobol' stream on ref_pins.render_inputs(seed=55)
      <case>/film     films of ref_pins.unseen_image_cases() (+ <case>/s2c, the reference's sampleToCamera)
      bitmap/<env>    the environment image the plugin reads back (Emitter::getBitmap, level 0) for ENVMAP_PROBE_CASES
      conductor_presets/*  every material of data/ior through the reference's spectrum code
      emitter/sample, instances/*  Scene::sampleEmitterDirect / rayIntersect (instanced) on ref_pins.emitter_probe_inputs()
      <env>/*         evalEnvironment / pdfEmitterDirect / sampleEmitterDirect of the environment map on ref_pins.envmap_probe_inputs()
      resample<i>/*, mipmap<i>/*  reference resampler pyramids (RESAMPLE_UNSEEN, seed 77, stored as half) and TMIPMap look-ups (MIPMAP_UNSEEN, seed 99)
      half            the half rounding of half_inputs(**HALF_UNSEEN)"""
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.join(HERE, ".."))
    import dataclasses
    import ref_pins
    from bsdf_configs import configs
    from mitsuba_b200.scene import checker_image
    from oracle import oracle_api as O
    ref = lambda name: C.CDLL(os.path.join(HERE, "..", "oracle", "_ref", name))
    f, digest = ref_pins._f, ref_pins.digest
    dig, arr = {}, {}

    lib = ref("libcoreref.so")
    dig.update({"core/" + k: digest(v) for k, v in ref_pins.run(lib, "coreref_", ref_pins.inputs(seed=99)).items()})
    lib.coreref_fresnel_diffuse_reflectance.restype = C.c_float
    dig["fresnel_diffuse_reflectance"] = [float(lib.coreref_fresnel_diffuse_reflectance(C.c_float(eta), 0)).hex() for eta in ref_pins.FDR_ETAS]

    lib, x = ref("libbsdfref.so"), ref_pins.bsdf_inputs(seed=4321)
    for name, b in configs().items():
        for k, v in ref_pins.run_bsdf_reference(lib, b, x).items():
            if name in BSDF_NOT_BIT_EXACT:
                arr[f"bsdf/{name}/{k}"] = v
            else:
                dig[f"bsdf/{name}/{k}"] = digest(v)

    arr.update({"render/" + k: v for k, v in ref_pins.run_render(ref("librenderref.so"), "renderref_", ref_pins.render_inputs(seed=55)).items()})

    lib = ref("libpathref.so")
    for name, desc, rp in ref_pins.unseen_image_cases():
        arr[name + "/film"], arr[name + "/s2c"] = ref_pins.reference_render(lib, desc, rp, want_camera=True)
    env_cases = {name: (desc, rp) for name, desc, rp in ref_pins.image_cases_env()}
    for name in ref_pins.ENVMAP_PROBE_CASES:
        h = ref_pins.reference_scene(lib, *env_cases[name])
        wh = (C.c_int * 2)()
        assert lib.pathref_environment_bitmap(h, wh, None) == 0
        bitmap = np.zeros((wh[1], wh[0], 3), np.float32)
        assert lib.pathref_environment_bitmap(h, wh, f(bitmap)) == 0
        arr["bitmap/" + name] = bitmap
    names, values = [], []
    for line in open(os.path.join(HERE, "..", "mitsuba_b200", "data", "conductor_presets.txt")):
        t = line.split()
        if t and not t[0].startswith("#"):
            e, kk = np.zeros(3, np.float32), np.zeros(3, np.float32)
            assert lib.pathref_conductor_preset(os.path.join(REF, "data").encode(), t[0].encode(), f(e), f(kk)) == 0
            names.append(t[0]); values.append(np.concatenate([e, kk]))
    arr["conductor_presets/names"], arr["conductor_presets/eta_k"] = np.array(names), np.stack(values)

    refp, smp, pos = ref_pins.emitter_probe_inputs()
    cases = {name: (desc, rp) for name, desc, rp in ref_pins.image_cases_ext()}
    h = ref_pins.reference_scene(lib, *cases["env_plus_area_cbox"])
    a = np.zeros((len(refp), 12), np.float32)
    lib.pathref_sample_emitter_direct(h, len(refp), f(refp), f(smp), f(a))
    arr["emitter/sample"] = a
    desc, rp = cases["instances_sobol"]
    h = ref_pins.reference_scene(lib, desc, rp)
    arr["instances/s2c"] = np.zeros((4, 4), np.float32)
    lib.pathref_sample_to_camera(h, f(arr["instances/s2c"]))
    arr["instances/inverses"] = np.stack(ref_pins.reference_instance_inverses(lib, desc))
    rays = O.OracleScene(desc, sample_to_camera=arr["instances/s2c"], instance_inverses=list(arr["instances/inverses"])).camera_rays(pos)
    a = np.zeros((len(pos), 24), np.float32)
    lib.pathref_intersect(h, len(pos), f(rays), f(a))
    dig.update({"instances/" + k: digest(v) for k, v in ref_pins.intersection_views(a).items()})
    for name, rays, rd, refp, dd, smp in ref_pins.envmap_probe_inputs():
        desc, rp = env_cases[name]
        inv = ref_pins.reference_envmap_inverse(lib, desc)
        if inv is not None:
            desc.envmap = dataclasses.replace(desc.envmap, to_local=inv)
            arr[name + "/to_local"] = inv
        h = ref_pins.reference_scene(lib, desc, rp)
        n = len(rays)
        ev, evd, pdf, s = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.float32), np.zeros((n, 12), np.float32)
        lib.pathref_eval_environment(h, n, 0, f(rays), f(ev))
        lib.pathref_eval_environment(h, n, 1, f(rd), f(evd))
        lib.pathref_pdf_environment_direct(h, n, f(refp), f(dd), f(pdf))
        lib.pathref_sample_emitter_direct(h, n, f(refp), f(smp), f(s))
        dig.update({name + "/eval": digest(ev), name + "/eval_diff": digest(evd), name + "/pdf": digest(pdf)})
        dig.update({f"{name}/sample_{k}": digest(v) for k, v in ref_pins.emitter_sample_views(s).items()})

    lib, rng = ref("librfilterref.so"), np.random.default_rng(77)
    for i, (shape, wu, wv) in enumerate(RESAMPLE_UNSEEN):
        img = np.maximum((rng.random(shape) * 1.2 - 0.05).astype(np.float32), 0)
        for l, lvl in enumerate(reference_pyramid(img, wu, wv, lib)):
            arr[f"resample{i}/{l + 1}"] = half_store(lvl)
    rng, img = np.random.default_rng(99), checker_image(70, 45, 6, 1)
    for i, (ft, wu, wv, aniso) in enumerate(MIPMAP_UNSEEN):
        m = ReferenceMipmap([img] + reference_pyramid(img, wu, wv), wu, wv, ft, aniso)
        uv, pt = texture_lookups(rng, 20000)
        dig[f"mipmap{i}/filtered"], dig[f"mipmap{i}/unfiltered"] = digest(m.eval(uv, pt)), digest(m.eval(uv))
    x = half_inputs(**HALF_UNSEEN)
    y = np.zeros_like(x)
    ref("libcoreref.so").coreref_half_round(len(x), f(x), f(y))
    dig["half"] = digest(y.view(np.uint32))   # the bits: the sign of zero included

    json.dump(dig, open(os.path.join(OUT, "unseen_ref.json"), "w"), indent=0, sort_keys=True)
    np.savez_compressed(os.path.join(OUT, "unseen_ref.npz"), **arr)
    print("unseen_ref.json:", len(dig), "digests; unseen_ref.npz:", len(arr), "arrays")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if "--unseen-only" in sys.argv:
        unseen_ref()
        sys.exit(0)
    if "--tex-only" in sys.argv:
        path_ref_tex()
        sys.exit(0)
    if "--spectrum-only" in sys.argv:
        spectrum_ref()
        sys.exit(0)
    if "--env-only" in sys.argv:
        path_ref_env()
        sys.exit(0)
    if "--ext-only" in sys.argv:
        path_ref_ext()
        sys.exit(0)
    if "--texture-only" in sys.argv:
        half_ref()
        mipmap_ref()
        sys.exit(0)
    path_ref()
    path_ref_ext()
    path_ref_env()
    path_ref_tex()
    spectrum_ref()
    render_ref()
    core_ref()
    bsdf_ref()
    sfmt_kat()
    sobol_ref()
    resample_ref()
    half_ref()
    mipmap_ref()
    unseen_ref()
