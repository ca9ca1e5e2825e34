"""Seeded inputs + one driver for the component functions that exist twice with the same C layout:
  coreref_*  the REFERENCE's own code (oracle/core_ref_shim.cpp -> oracle/_ref/libcoreref.so, compiled from /root/reference)
  orc_*      the oracle's restatement (oracle/mts_oracle.cpp)
tests/gen_golden.py runs the first and commits tests/golden/core_ref.npz; tests/test_oracle_reference_pins.py runs the second."""
import ctypes as C

import numpy as np

N = 400
MICROFACET = [(t, au, av, sv) for t in (0, 1, 2) for (au, av) in ((0.3, 0.3), (0.1, 0.4), (0.02, 0.02)) for sv in (1, 0) if not (t == 2 and sv)]
ETAS = (1.5, 1.0 / 1.5, 1.33, 1.0)
CONDUCTORS = (((0.2004, 0.9240, 1.1022), (3.9129, 2.4528, 2.1421)), ((0.1431, 0.3749, 1.4424), (3.9831, 2.3857, 1.6032)))
PMF_WEIGHTS = ([1.0, 2.0, 3.0, 4.0], [0.0, 1.0, 0.0, 0.0, 5.0, 0.0], [0.25] * 7 + [0.0], [3.0])


def _f(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _dirs(rng, n, upper=False):
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    if upper:
        d[:, 2] = np.abs(d[:, 2])
    return np.ascontiguousarray(d, np.float32)


def inputs(seed=31337):
    rng = np.random.default_rng(seed)
    x = {}
    x["wi_up"] = _dirs(rng, N, True)
    x["wi_up"][:8, 2] = np.float32(1e-3)  # grazing
    x["wi_up"][:8] /= np.linalg.norm(x["wi_up"][:8], axis=1, keepdims=True)
    x["m_up"] = _dirs(rng, N, True)
    x["samples"] = rng.random((N, 2)).astype(np.float32)
    x["samples"][:4] = np.array([[0, 0], [0.5, 0.5], [0.999999, 0.999999], [0, 0.999999]], np.float32)
    tris = rng.uniform(-1, 1, (N, 9)).astype(np.float32)
    tris[:6, 3:6] = tris[:6, 0:3]  # degenerate: two equal vertices
    tris[6:12, 2] = tris[6:12, 5] = tris[6:12, 8] = np.float32(0.25)  # axis-aligned
    x["tris"] = tris
    o = rng.uniform(-2, 2, (N, 3)).astype(np.float32)
    tgt = (tris[:, 0:3] * 0.3 + tris[:, 3:6] * 0.3 + tris[:, 6:9] * 0.4 + rng.normal(size=(N, 3)) * 0.3).astype(np.float32)
    d = tgt - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d[12:20, 0] = 0.0  # rays parallel to an axis plane
    rays = np.concatenate([o, np.full((N, 1), 1e-4), d, np.full((N, 1), np.inf)], 1).astype(np.float32)
    rays[20:30, 7] = np.float32(0.5)  # short intervals
    x["rays"] = np.ascontiguousarray(rays)
    lo = rng.uniform(-1, 0, (N, 3)).astype(np.float32)
    x["boxes"] = np.ascontiguousarray(np.concatenate([lo, lo + rng.uniform(0.01, 1.5, (N, 3)).astype(np.float32)], 1))
    x["cos"] = np.concatenate([np.linspace(-1, 1, N - 6), [0.0, 1e-6, -1e-6, 1.0, -1.0, 0.5]]).astype(np.float32)
    x["dirs"] = _dirs(rng, N)
    x["normals"] = _dirs(rng, N)
    x["dpdu"] = (rng.normal(size=(N, 3)) * 2).astype(np.float32)
    x["pmf_samples"] = np.concatenate([rng.random(N - 4), [0.0, 0.999999, 0.5, 0.25]]).astype(np.float32)
    x["tea"] = rng.integers(0, 2 ** 32, (64, 2), dtype=np.uint64).astype(np.uint32)
    return x


def run(lib, prefix, x):
    """All component outputs as a dict of arrays; `lib` is a ctypes CDLL exporting <prefix><name> with the layouts of core_ref_shim.cpp."""
    fn = lambda name: getattr(lib, prefix + name)
    out = {}
    for (t, au, av, sv) in MICROFACET:
        key = f"mf_{t}_{au}_{av}_{sv}"
        a = np.zeros((N, 6), np.float32)
        b = np.zeros((N, 3), np.float32)
        # the oracle's historical entry points take uint64 counts; the new ones int -- both are fine with c_int for small n
        fn("microfacet_sample")(t, C.c_float(au), C.c_float(av), sv, C.c_uint64(N) if prefix == "orc_" else N, _f(x["wi_up"]), _f(x["samples"]), _f(a))
        fn("microfacet_eval")(t, C.c_float(au), C.c_float(av), sv, C.c_uint64(N) if prefix == "orc_" else N, _f(x["wi_up"]), _f(x["m_up"]), _f(b))
        out[key + "_sample"], out[key + "_eval"] = a, b
    rec = np.zeros((N, 12), np.uint32)
    st = np.zeros(N, np.int32)
    fn("triaccel_load")(N, _f(x["tris"]), rec.ctypes.data_as(C.POINTER(C.c_uint32)), st.ctypes.data_as(C.POINTER(C.c_int)))
    out["triaccel_records"], out["triaccel_status"] = rec, st
    a = np.zeros((N, 4), np.float32)
    fn("triaccel_intersect")(N, _f(x["tris"]), _f(x["rays"]), _f(a))
    out["triaccel_hits"] = a
    a = np.zeros((N, 3), np.float32)
    fn("aabb_intersect")(N, _f(x["boxes"]), _f(x["rays"]), _f(a))
    out["aabb"] = a
    for what in range(4):
        a = np.zeros((N, 3), np.float32)
        fn("warp")(what, N, _f(x["samples"]), _f(a))
        out[f"warp{what}"] = a
    for eta in ETAS:
        a = np.zeros((N, 2), np.float32)
        fn("fresnel_dielectric_ext")(N, _f(x["cos"]), C.c_float(eta), _f(a))
        out[f"fresnel_dielectric_{eta:.4f}"] = a
    for i, (eta, k) in enumerate(CONDUCTORS):
        a = np.zeros((N, 3), np.float32)
        e, kk = np.array(eta, np.float32), np.array(k, np.float32)
        fn("fresnel_conductor_exact_rgb")(N, _f(np.abs(x["cos"])), _f(e), _f(kk), _f(a))
        out[f"fresnel_conductor_{i}"] = a
    a = np.zeros((N, 3), np.float32)
    fn("reflect")(N, _f(x["dirs"]), _f(x["normals"]), _f(a))
    out["reflect"] = a
    for eta in (1.5, 1.33):
        a = np.zeros((N, 3), np.float32)
        ct = np.where(np.arange(N) % 2 == 0, -0.7, 0.6).astype(np.float32)
        fn("refract")(N, _f(x["dirs"]), _f(x["normals"]), C.c_float(eta), _f(ct), _f(a))
        out[f"refract_{eta}"] = a
    a = np.zeros((N, 6), np.float32)
    fn("coordinate_system")(N, _f(x["normals"]), _f(a))
    out["coordinate_system"] = a
    a = np.zeros((N, 9), np.float32)
    fn("shading_frame")(N, _f(x["normals"]), _f(x["dpdu"]), _f(a))
    out["shading_frame"] = a
    a = np.zeros((N, 3), np.float32)
    fn("triangle_sample")(N, _f(x["tris"]), _f(x["samples"]), _f(a))
    out["triangle_sample"] = a
    for i, w in enumerate(PMF_WEIGHTS):
        w = np.array(w, np.float32)
        idx, idx2 = np.zeros(N, np.uint32), np.zeros(N, np.uint32)
        reused, cdf = np.zeros(N, np.float32), np.zeros(len(w), np.float32)
        f = fn("pmf")
        f.restype = C.c_float
        total = f(len(w), _f(w), N, _f(x["pmf_samples"]), idx.ctypes.data_as(C.POINTER(C.c_uint32)), idx2.ctypes.data_as(C.POINTER(C.c_uint32)), _f(reused), _f(cdf))
        out[f"pmf{i}_index"], out[f"pmf{i}_index_reuse"], out[f"pmf{i}_reused"], out[f"pmf{i}_pdf"], out[f"pmf{i}_total"] = idx, idx2, reused, cdf, np.float32(total)
    f = fn("tea")
    f.restype = C.c_uint64
    out["tea"] = np.array([[f(C.c_uint32(int(a)), C.c_uint32(int(b)), r) for r in (4, 8)] for a, b in x["tea"]], np.uint64)
    return out


# ---------------------------------------------------------------------------------------------------------------------------
# BSDF plugins: the reference's own src/bsdfs/*.cpp (oracle/bsdf_ref_shim.cpp -> oracle/_ref/libbsdfref.so) vs the oracle
# ---------------------------------------------------------------------------------------------------------------------------
PLUGIN_IDS = {"diffuse": 0, "roughconductor": 1, "roughdielectric": 2, "coating": 3, "null": 4, "twosided": 5, "dielectric": 6, "conductor": 7, "plastic": 8}
NB = 200


def reference_bsdf(lib, b):
    """Instantiate the reference plugin for a mitsuba_b200.scene.Bsdf through its Properties, children first."""
    from mitsuba_b200.scene import lookup_ior
    lib.bsdfref_create.restype = C.c_void_p
    f, s, bl, sp = {}, {}, {}, {}
    t = b.type
    if t == "diffuse":
        sp["reflectance"] = b.reflectance
    if t in ("roughconductor", "roughdielectric"):
        s["distribution"] = b.distribution
        f["alphaU"], f["alphaV"] = b.alpha_u, b.alpha_v
        bl["sampleVisible"] = b.sample_visible
    if t in ("roughconductor", "conductor"):
        s["material"] = "none"
        sp["eta"], sp["k"] = b.eta, b.k
        f["extEta"] = lookup_ior(b.ext_eta, "air")
        sp["specularReflectance"] = b.specular_reflectance
    if t in ("roughdielectric", "dielectric", "coating", "plastic"):
        f["intIOR"] = lookup_ior(b.int_ior if not (t == "plastic" and b.int_ior == "bk7") else "polypropylene", "bk7")
        f["extIOR"] = lookup_ior(b.ext_ior, "air")
        sp["specularReflectance"] = b.specular_reflectance
    if t in ("roughdielectric", "dielectric"):
        sp["specularTransmittance"] = b.specular_transmittance
    if t == "coating":
        f["thickness"] = b.thickness
        sp["sigmaA"] = b.sigma_a
    if t == "plastic":
        sp["diffuseReflectance"] = b.diffuse_reflectance
        bl["nonlinear"] = b.nonlinear
    kids = []
    if t in ("coating", "twosided"):
        kids.append(reference_bsdf(lib, b.nested))
        if t == "twosided" and b.nested_back is not None:
            kids.append(reference_bsdf(lib, b.nested_back))
    # a bitmap texture bound to one of the colour parameters (<texture name="..." type="bitmap">): built by the reference's own plugin
    from mitsuba_b200.scene import Texture
    tex, tex_name = None, None
    for name in list(sp):
        if isinstance(sp[name], Texture):
            assert tex is None and hasattr(lib, "pathref_create_tex"), "textured BSDFs need the assembled renderer (libpathref.so)"
            tex, tex_name = reference_texture(lib.raw, sp.pop(name)), name
    arr = lambda keys: (C.c_char_p * max(1, len(keys)))(*[k.encode() for k in keys])
    fv = (C.c_float * max(1, len(f)))(*[float(v) for v in f.values()])
    sv = arr([str(v) for v in s.values()])
    bv = (C.c_int * max(1, len(bl)))(*[int(bool(v)) for v in bl.values()])
    spv = (C.c_float * max(3, 3 * len(sp)))(*[float(x) for v in sp.values() for x in v])
    if tex is not None:
        h = lib.pathref_create_tex(PLUGIN_IDS[t], len(f), arr(list(f)), fv, len(s), arr(list(s)), sv, len(bl), arr(list(bl)), bv, len(sp), arr(list(sp)), spv,
                                   kids[0] if kids else None, kids[1] if len(kids) > 1 else None, tex, tex_name.encode())
    else:
        h = lib.bsdfref_create(PLUGIN_IDS[t], len(f), arr(list(f)), fv, len(s), arr(list(s)), sv, len(bl), arr(list(bl)), bv, len(sp), arr(list(sp)), spv,
                               kids[0] if kids else None, kids[1] if len(kids) > 1 else None)
    assert h, t
    return C.c_void_p(h)


def texture_pyramid(tex):
    """The MIP pyramid (float32 levels, rounded to half precision) the oracle derives from the decoded image of a scene.Texture."""
    from oracle.oracle_api import lib as olib, _p, make_texture_desc
    L = olib()
    d = tex.flat()
    L.orc_scene_new.restype = C.c_void_p
    s = C.c_void_p(L.orc_scene_new())
    L.orc_add_texture.restype = C.c_int
    assert L.orc_add_texture(s, C.byref(make_texture_desc(d)), _p(d["pixels"])) == 0
    info = (C.c_int32 * 64)(); mx, sc = C.c_float(), C.c_float()
    L.orc_texture_info(s, 0, info, C.byref(mx), C.byref(sc))
    levels = []
    for l in range(info[0]):
        w, h = info[1 + 2 * l], info[2 + 2 * l]
        a = np.empty((h, w, d["channels"]), np.float32)
        L.orc_texture_level(s, 0, l, _p(a))
        levels.append(a)
    L.orc_scene_free(s)
    return d, levels


_TEX_MEMO = {}


def reference_texture(lib, tex):
    """scene.Texture -> the reference's BitmapTexture (src/textures/bitmap.cpp), constructed from a MIP map cache file that holds the oracle's
    pyramid (path_ref_shim.cpp pathref_bitmap_texture)."""
    import hashlib, os, tempfile
    key = (id(lib), id(tex))
    if key in _TEX_MEMO:             # (the entry keeps `tex` alive, so its id cannot be handed to another object)
        return _TEX_MEMO[key][0]
    d, levels = texture_pyramid(tex)
    orig = np.maximum(np.ascontiguousarray(d["pixels"], np.float32), np.float32(0))   # clampNegative precedes the statistics (mipmap.h:229-241)
    sizes = np.array([[a.shape[1], a.shape[0]] for a in levels], np.int32)
    ptrs = (C.POINTER(C.c_float) * len(levels))(*[_f(a) for a in levels])
    stem = os.path.join(tempfile.gettempdir(), f"b2ref_tex_{os.getpid()}_" + hashlib.sha1(levels[0].tobytes() + repr(sorted((k, v) for k, v in d.items() if k != "pixels")).encode()).hexdigest()[:12])
    lib.pathref_bitmap_texture.restype = C.c_void_p
    t = lib.pathref_bitmap_texture(stem.encode(), d["channels"], len(levels), sizes.ctypes.data_as(C.POINTER(C.c_int)), ptrs, _f(orig),
                                   tex.filter_type.lower().encode(), tex.wrap_u.encode(), tex.wrap_v.encode(), C.c_float(tex.max_anisotropy),
                                   C.c_float(tex.uoffset), C.c_float(tex.voffset), C.c_float(tex.uscale), C.c_float(tex.vscale))
    for ext in (".img", ".mip"):
        try:
            os.unlink(stem + ext)
        except OSError:
            pass
    assert t
    _TEX_MEMO[key] = (C.c_void_p(t), tex, lib)
    return _TEX_MEMO[key][0]


def bsdf_inputs(seed=777):
    rng = np.random.default_rng(seed)
    x = {"wi": _dirs(rng, NB), "wo": _dirs(rng, NB), "samples": rng.random((NB, 3)).astype(np.float32)}
    x["wi"][: NB // 2, 2] = np.abs(x["wi"][: NB // 2, 2])  # half of them from the front side
    x["wi"][:6, 2] = np.float32(2e-3)  # grazing
    x["wi"][:6] /= np.linalg.norm(x["wi"][:6], axis=1, keepdims=True)
    # mirror / refracted directions for the discrete measure are produced by sample(); eval(EDiscrete) is fed with them below
    return x


def run_bsdf_reference(lib, b, x):
    h = reference_bsdf(lib, b)
    lib.bsdfref_type.restype = C.c_uint
    out = {"type": np.uint32(lib.bsdfref_type(h))}
    rgb, pdf = np.zeros((NB, 3), np.float32), np.zeros(NB, np.float32)
    lib.bsdfref_eval(h, NB, _f(x["wi"]), _f(x["wo"]), 0, _f(rgb), _f(pdf))
    out["eval"], out["pdf"] = rgb, pdf
    smp = np.zeros((NB, 10), np.float32)
    lib.bsdfref_sample(h, NB, _f(x["wi"]), _f(x["samples"]), _f(smp))
    smp[np.all(smp[:, 3:6] == 0, axis=1), 6] = 0
    out["sample"] = smp
    wo2 = np.ascontiguousarray(smp[:, 0:3])
    rgb2, pdf2 = np.zeros((NB, 3), np.float32), np.zeros(NB, np.float32)
    lib.bsdfref_eval(h, NB, _f(x["wi"]), _f(wo2), 1, _f(rgb2), _f(pdf2))  # EDiscrete at the sampled directions
    out["eval_discrete"], out["pdf_discrete"] = rgb2, pdf2
    rgb3, pdf3 = np.zeros((NB, 3), np.float32), np.zeros(NB, np.float32)
    lib.bsdfref_eval(h, NB, _f(x["wi"]), _f(wo2), 0, _f(rgb3), _f(pdf3))  # ESolidAngle at the sampled directions
    out["eval_at_sample"], out["pdf_at_sample"] = rgb3, pdf3
    return out


def run_bsdf_oracle(b, x):
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from bsdf_configs import flatten
    from oracle import oracle_api as O
    flat, bid = flatten(b)
    out = {"type": np.uint32(O.bsdf_type(flat, bid))}
    out["eval"], out["pdf"] = O.bsdf_eval(flat, bid, x["wi"], x["wo"])
    arr = O.make_bsdf_array(flat)
    smp = np.zeros((NB, 10), np.float32)
    O.lib().orc_bsdf_sample(arr, C.c_int(len(flat)), C.c_int(bid), C.c_uint64(NB), _f(x["wi"]), _f(x["samples"]), _f(smp))
    zero = np.all(smp[:, 3:6] == 0, axis=1)
    smp[zero, 0:3] = 0; smp[zero, 6] = 0; smp[zero, 7] = 0; smp[zero, 8] = 0  # wo / pdf / type / eta are unspecified after a failed sample
    smp[:, 9] = 0
    out["sample"] = smp
    wo2 = np.ascontiguousarray(smp[:, 0:3])
    out["eval_discrete"], out["pdf_discrete"] = O.bsdf_eval(flat, bid, x["wi"], wo2, discrete=True)
    out["eval_at_sample"], out["pdf_at_sample"] = O.bsdf_eval(flat, bid, x["wi"], wo2)
    return out


# ---------------------------------------------------------------------------------------------------------------------------
# uv partials, reconstruction filters, ImageBlock::put, the Sobol' sampler plugin (oracle/render_ref_shim.cpp -> librenderref.so)
# ---------------------------------------------------------------------------------------------------------------------------
NR = 300
SOBOL_CASES = [(0, 64, 64, 16, 5, 7, 3), (0, 100, 60, 64, 99, 59, 63), (12345, 256, 256, 4, 17, 200, 2), (7, 33, 1024, 1024, 0, 1000, 777), (1, 8, 8, 1, 3, 3, 0)]


def render_inputs(seed=2718):
    rng = np.random.default_rng(seed)
    x = {}
    rec = np.zeros((NR, 27), np.float32)
    n = _dirs(rng, NR)
    rec[:, 0:3] = rng.uniform(-2, 2, (NR, 3))
    rec[:, 3:6] = n
    rec[:, 6:9] = rng.normal(size=(NR, 3)) * 2
    rec[:, 9:12] = rng.normal(size=(NR, 3)) * 2
    o = rec[:, 0:3] + n * 3 + rng.normal(size=(NR, 3)).astype(np.float32)
    rec[:, 12:15] = rec[:, 15:18] = rec[:, 18:21] = o
    d = rec[:, 0:3] - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rec[:, 21:24] = d + rng.normal(size=(NR, 3)) * 0.01
    rec[:, 24:27] = d + rng.normal(size=(NR, 3)) * 0.01
    rec[:5, 6:12] = 0.0                      # dpdu = dpdv = 0
    rec[5:10, 9:12] = rec[5:10, 6:9]         # singular system
    rec[10:14, 21:24] = np.cross(n[10:14], rng.normal(size=(4, 3)))  # offset ray parallel to the surface: prx == 0 up to rounding
    x["partials"] = np.ascontiguousarray(rec, np.float32)
    pos = np.stack([rng.uniform(10 - 3, 10 + 16 + 3, NR), rng.uniform(20 - 3, 20 + 12 + 3, NR)], -1).astype(np.float32)
    val = rng.random((NR, 4)).astype(np.float32)
    val[:4, 0] = 0.0
    x["put_pos"], x["put_val"] = pos, val
    return x


def run_render(lib, prefix, x, oracle_scene=None):
    fn = lambda name: getattr(lib, prefix + name)
    out = {}
    a = np.zeros((NR, 4), np.float32)
    fn("compute_partials")(NR, _f(x["partials"]), _f(a))
    out["partials"] = a
    for kind in (0, 1):
        v, r, b = np.zeros(32, np.float32), C.c_float(), C.c_int()
        if prefix == "orc_":
            fn("filter_table")(kind, C.c_float(0.5), _f(v), C.byref(r), C.byref(b))  # gaussian.cpp:35-38 default stddev
        else:
            fn("filter_table")(kind, _f(v), C.byref(r), C.byref(b))
        out[f"filter{kind}_values"], out[f"filter{kind}_radius"], out[f"filter{kind}_border"] = v, np.float32(r.value), np.int32(b.value)
        border = b.value
        data = np.zeros((12 + 2 * border, 16 + 2 * border, 5), np.float32)
        ok = np.zeros(NR, np.int32)
        args = [10, 20, 16, 12, kind] + ([C.c_float(0.5)] if prefix == "orc_" else []) + [NR, _f(x["put_pos"]), _f(x["put_val"]), _f(data), ok.ctypes.data_as(C.POINTER(C.c_int))]
        fn("block_put")(*args)
        out[f"put{kind}_data"], out[f"put{kind}_ok"] = data, ok
    for i, (scr, W, H, spp, px, py, idx) in enumerate(SOBOL_CASES):
        s = np.zeros(24, np.float32)
        if prefix == "orc_":
            s = oracle_scene(W, H).sampler_stream("sobol", scr, spp, px, py, idx, 24)
        else:
            fn("sobol_stream")(C.c_uint64(scr), W, H, spp, px, py, idx, 24, _f(s))
        out[f"sobol{i}"] = np.asarray(s, np.float32)
    return out


# ---------------------------------------------------------------------------------------------------------------------------
# whole images: a minimal `path` renderer assembled from the reference's own sources (oracle/path_ref_shim.cpp -> libpathref.so)
# ---------------------------------------------------------------------------------------------------------------------------
def reference_scene(lib, desc, rp):
    """Build a mitsuba_b200.scene.SceneDesc as a reference Scene (the reference's own classes, oracle/path_ref_shim.cpp) -> handle."""
    from mitsuba_b200.scene import Bsdf
    lib.pathref_new.restype = C.c_void_p
    lib.pathref_bsdf.restype = C.c_void_p
    h = C.c_void_p(lib.pathref_new())

    lib.pathref_bsdf2.restype = C.c_void_p

    class _L:  # reference_bsdf() talks to `bsdfref_create`; here the same function is called pathref_bsdf
        bsdfref_create = lib.pathref_bsdf
        pathref_create_tex = lib.pathref_bsdf2
        raw = lib
    memo, mmemo, keep = {}, {}, []
    lib.pathref_medium_homogeneous.restype = C.c_void_p
    lib.pathref_medium_heterogeneous.restype = C.c_void_p

    def medium(md):
        if md is None:
            return None
        if id(md) not in mmemo:
            ph = {"isotropic": 0, "hg": 1}[md.phase]
            if md.type == "homogeneous":
                sa, ss = np.asarray(md.sigma_a, np.float32), np.asarray(md.sigma_s, np.float32)
                mmemo[id(md)] = C.c_void_p(lib.pathref_medium_homogeneous(_f(sa), _f(ss), md.strategy.encode(), C.c_float(md.sampling_density),
                                                                             C.c_float(md.medium_sampling_weight), ph, C.c_float(md.g)))
            else:
                import hashlib, os, tempfile
                dens = np.ascontiguousarray(md.density, np.float32)
                nz, ny, nx = dens.shape
                blob = b"VOL\x03" + np.array([1, nx, ny, nz, 1], "<i4").tobytes() + np.array(list(md.aabb_min) + list(md.aabb_max), "<f4").tobytes() + dens.tobytes()
                # gridvolume reads a file: one copy per content in the temp directory, shared by every process that needs it
                fname = os.path.join(tempfile.gettempdir(), "b2ref_" + hashlib.sha1(blob).hexdigest()[:16] + ".vol")
                if not os.path.exists(fname):
                    tmp = fname + f".{os.getpid()}"
                    with open(tmp, "wb") as f:
                        f.write(blob)
                    os.replace(tmp, fname)
                tw = np.ascontiguousarray(md.to_world, np.float32) if md.to_world is not None else None
                al = np.asarray(md.albedo, np.float32)
                mmemo[id(md)] = C.c_void_p(lib.pathref_medium_heterogeneous(fname.encode(), _f(tw) if tw is not None else None, _f(al), C.c_float(md.scale), ph, C.c_float(md.g)))
        return mmemo[id(md)]
    lib.pathref_shapegroup_new.restype = C.c_void_p
    groups = {}
    for m in desc.meshes:
        b = m.bsdf
        if b is None and m.interior is None and m.exterior is None:
            b = Bsdf("diffuse", reflectance=(0.0,) * 3 if m.radiance is not None else (0.5,) * 3)
        if b is not None and id(b) not in memo:
            memo[id(b)] = reference_bsdf(_L, b)
        P = np.ascontiguousarray(m.P, np.float32)
        N = np.ascontiguousarray(m.N, np.float32) if m.N is not None else None
        UV = np.ascontiguousarray(m.UV, np.float32) if m.UV is not None else None
        I = np.ascontiguousarray(m.idx, np.uint32)
        rad = np.asarray(m.radiance, np.float32) if m.radiance is not None else None
        if m.group >= 0:  # member of a <shape type="shapegroup"> (object space); instances reference the group below
            if m.group not in groups:
                groups[m.group] = C.c_void_p(lib.pathref_shapegroup_new(h))
            lib.pathref_shapegroup_add_mesh(groups[m.group], _f(P), _f(N) if N is not None else None, _f(UV) if UV is not None else None, len(P),
                                            I.ctypes.data_as(C.POINTER(C.c_uint32)), len(I), memo[id(b)])
            continue
        lib.pathref_add_mesh_media(h, _f(P), _f(N) if N is not None else None, _f(UV) if UV is not None else None, len(P),
                                   I.ctypes.data_as(C.POINTER(C.c_uint32)), len(I), memo[id(b)] if b is not None else None, _f(rad) if rad is not None else None,
                                   C.c_float(m.sampling_weight), medium(m.interior), medium(m.exterior))
    for g in groups.values():
        lib.pathref_shapegroup_configure(g)   # builds the group's kd-tree (shapegroup.cpp ShapeGroup::configure)
    for inst in desc.instances:
        lib.pathref_add_instance(h, groups[inst.group], _f(np.ascontiguousarray(inst.to_world, np.float32)))
    if desc.env_radiance is not None:          # <emitter type="constant">: added last here, yet first in Scene::m_emitters (scene.cpp:510-516 vs :322-335)
        lib.pathref_add_constant_emitter(h, _f(np.asarray(desc.env_radiance, np.float32)), C.c_float(desc.env_sampling_weight))
    if getattr(desc, "envmap", None) is not None:   # <emitter type="envmap">: the pyramid is this repository's (oracle) resampling of the image,
        # handed to the reference's EnvironmentMap as a MIP map cache file (path_ref_shim.cpp pathref_add_envmap); tables / look-ups / sampling are its own
        add_reference_envmap(lib, h, desc.envmap)
    cam = desc.camera
    assert cam.fov_axis == "x"
    tw = np.ascontiguousarray(cam.to_world, np.float32)
    # `independent` here is this repository's counter-based stream (kind 2), handed to the reference integrator through the Sampler interface
    crop = cam.crop or (0, 0, cam.width, cam.height)
    lib.pathref_setup4(h, _f(tw), C.c_float(cam.fov), C.c_float(cam.near), C.c_float(cam.far), cam.width, cam.height,
                       {"box": 0, "gaussian": 1}[rp.rfilter], {"sobol": 0, "independent": 2}[rp.sampler], rp.spp, C.c_uint64(rp.seed),
                       rp.max_depth, rp.rr_depth, int(rp.strict_normals), int(rp.hide_emitters), {"path": 0, "volpath": 1}[rp.integrator],
                       C.c_float(cam.aperture_radius), C.c_float(cam.focus_distance), *[int(v) for v in crop])
    return h


def envmap_pyramid(em):
    """The MIP pyramid (float32 RGB levels, already rounded to half precision) the oracle derives from the decoded image."""
    from oracle.oracle_api import lib as olib, _p
    L = olib()
    px = np.ascontiguousarray(em.pixels, np.float32)
    M, Minv = em.matrices()
    L.orc_scene_new.restype = C.c_void_p
    s = C.c_void_p(L.orc_scene_new())
    L.orc_add_envmap_emitter.restype = C.c_int
    assert L.orc_add_envmap_emitter(s, px.shape[1], px.shape[0], _p(px), C.c_float(em.scale), _p(M), _p(Minv), C.c_float(em.sampling_weight)) >= 0
    info = (C.c_int32 * 64)(); nrm = C.c_float()
    L.orc_envmap_info(s, 0, info, C.byref(nrm))
    levels = []
    for l in range(info[0]):
        a = np.empty((info[2 + 2 * l], info[1 + 2 * l], 3), np.float32)
        L.orc_envmap_level(s, 0, l, _p(a))
        levels.append(a)
    L.orc_scene_free(s)
    return levels


def add_reference_envmap(lib, h, em):
    import hashlib, os, tempfile
    levels = envmap_pyramid(em)
    sizes = np.array([[a.shape[1], a.shape[0]] for a in levels], np.int32)
    ptrs = (C.POINTER(C.c_float) * len(levels))(*[_f(a) for a in levels])
    tw = np.ascontiguousarray(em.to_world, np.float32) if em.to_world is not None else None
    stem = os.path.join(tempfile.gettempdir(), f"b2ref_env_{os.getpid()}_" + hashlib.sha1(levels[0].tobytes()).hexdigest()[:12])
    lib.pathref_add_envmap.restype = C.c_int
    rc = lib.pathref_add_envmap(h, stem.encode(), len(levels), sizes.ctypes.data_as(C.POINTER(C.c_int)), ptrs, _f(tw) if tw is not None else None,
                                C.c_float(em.scale), C.c_float(em.sampling_weight))
    for ext in (".img", ".mip"):       # the class has mapped the cache by now (MemoryMappedFile keeps its own handle)
        try:
            os.unlink(stem + ext)
        except OSError:
            pass
    assert rc == 0


def reference_render(lib, desc, rp, want_camera=False):
    """Render a mitsuba_b200.scene.SceneDesc with the reference's MIPathTracer / Scene / ShapeKDTree / plugins.  Returns (H, W, 5)
    (and, with want_camera, the reference's sampleToCamera matrix: camera set-up is host work, both sides should start from it)."""
    h = reference_scene(lib, desc, rp)
    cam = desc.camera
    fw, fh = cam.film_size()
    film = np.zeros((fh, fw, 5), np.float32)
    lib.pathref_render(h, _f(film))
    if want_camera:
        s2c = np.zeros((4, 4), np.float32)
        lib.pathref_sample_to_camera(h, _f(s2c))
        return film, s2c
    return film


def reference_instance_inverses(lib, desc):
    """Transform(toWorld).inverse() of every instance, computed by the reference's own Matrix4x4::invert."""
    out = []
    for inst in desc.instances:
        inv = np.zeros((4, 4), np.float32)
        lib.pathref_transform_inverse(_f(np.ascontiguousarray(inst.to_world, np.float32)), _f(inv))
        out.append(inv)
    return out


def image_cases():
    """(name, SceneDesc, RenderParams) of the image-level pins: `path`, Sobol' sampler."""
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from bsdf_configs import configs
    from mitsuba_b200.scene import RenderParams, cornell_box, material_ball
    cf = configs()
    yield "cbox_box_8spp", cornell_box(48, 48), RenderParams(spp=8, sampler="sobol", rfilter="box")
    yield "cbox_gaussian_16spp", cornell_box(40, 32), RenderParams(spp=16, sampler="sobol", rfilter="gaussian")
    yield "cbox_depth3_scramble", cornell_box(32, 32), RenderParams(spp=4, sampler="sobol", rfilter="gaussian", max_depth=3, rr_depth=2, seed=7)
    yield "cbox_strict_hidden", cornell_box(32, 32), RenderParams(spp=4, sampler="sobol", rfilter="box", strict_normals=True, hide_emitters=True)
    for name in ("roughconductor_ggx", "roughdielectric_beckmann", "coating_diffuse", "dielectric", "conductor", "roughconductor_as", "twosided_two", "plastic"):
        yield "ball_" + name, material_ball(cf[name], 40, 40, n_theta=20, n_phi=40), RenderParams(spp=8, sampler="sobol", rfilter="gaussian")
    # volpath (src/integrators/path/volpath.cpp) with the reference's medium / volume / phase plugins; `independent` = this repository's
    # counter stream served to the reference integrator through the Sampler interface
    from mitsuba_b200.scene import Medium, smoke_scene
    yield "vol_cbox_sobol", cornell_box(32, 32), RenderParams(spp=4, sampler="sobol", rfilter="box", integrator="volpath")
    yield "path_cbox_counter", cornell_box(32, 32), RenderParams(spp=4, sampler="independent", rfilter="gaussian")
    for strat in ("balance", "single"):
        d = smoke_scene(40, 40, res=8)
        d.meshes[2].interior = Medium("homogeneous", sigma_a=(0.5, 0.6, 0.7), sigma_s=(2.0, 2.5, 3.0), strategy=strat, phase="hg", g=0.3)
        yield "vol_homogeneous_" + strat, d, RenderParams(spp=8, sampler="independent", rfilter="gaussian", integrator="volpath")
    yield "vol_heterogeneous_iso", smoke_scene(40, 40, res=8, scale=6.0), RenderParams(spp=8, sampler="independent", rfilter="gaussian", integrator="volpath")
    yield "vol_heterogeneous_hg", smoke_scene(40, 40, res=16, scale=12.0, phase="hg", g=0.5), RenderParams(spp=8, sampler="independent", rfilter="gaussian", integrator="volpath")
    yield "vol_heterogeneous_sobol", smoke_scene(32, 32, res=8, scale=4.0), RenderParams(spp=4, sampler="sobol", rfilter="box", integrator="volpath", max_depth=4)


def image_cases_ext():
    """Image-level pins of the plugins that joined the assembled reference renderer later: the `thinlens` sensor
    (src/sensors/thinlens.cpp), the `constant` environment emitter (src/emitters/constant.cpp), `shapegroup` / `instance`
    (src/shapes/{shapegroup,instance}.cpp).  Fixture: tests/golden/path_ref_ext.npz."""
    import dataclasses
    from mitsuba_b200.scene import Bsdf, Instance, Mesh, RenderParams, cornell_box, cube_mesh, material_ball, smoke_scene, stress_scene, uv_sphere
    d = cornell_box(40, 40)
    d.camera = dataclasses.replace(d.camera, aperture_radius=25.0, focus_distance=1100.0)
    yield "thinlens_cbox_sobol", d, RenderParams(spp=8, sampler="sobol", rfilter="gaussian")
    d = cornell_box(32, 32)
    d.camera = dataclasses.replace(d.camera, aperture_radius=60.0, focus_distance=900.0)
    yield "thinlens_cbox_counter", d, RenderParams(spp=8, sampler="independent", rfilter="box", max_depth=4)
    # constant emitter: alone (every miss is radiance), next to an area light (emitter selection + MIS both ways), hidden, under volpath
    d = material_ball(Bsdf("roughconductor", distribution="ggx", alpha_u=0.2, alpha_v=0.2, eta=(0.2004, 0.9240, 1.1022), k=(3.9129, 2.4528, 2.1421)), 40, 40, n_theta=16, n_phi=32)
    d.meshes = [m for m in d.meshes if m.radiance is None]
    d.env_radiance = (0.7, 0.8, 0.9)
    yield "env_only_ball", d, RenderParams(spp=8, sampler="sobol", rfilter="gaussian")
    d = cornell_box(36, 36)
    d.meshes = [m for i, m in enumerate(d.meshes) if i != 1]   # open the box: drop one wall so that the environment is seen
    d.env_radiance = (0.4, 0.6, 1.0); d.env_sampling_weight = 2.0
    yield "env_plus_area_cbox", d, RenderParams(spp=8, sampler="sobol", rfilter="box")
    yield "env_hidden_cbox", d, RenderParams(spp=4, sampler="independent", rfilter="gaussian", hide_emitters=True, max_depth=5)
    # three emitters: constant (weight 0.5) + two area lights (weights 1 and 3): the emitter-selection CDF and sampleReuse over more than two entries
    d = cornell_box(32, 32)
    by = {m.name: m for m in d.meshes}
    by["short"].radiance = (2.0, 4.0, 1.0); by["short"].sampling_weight = 3.0
    d.meshes = [m for m in d.meshes if m.name != "right"]
    d.env_radiance = (0.1, 0.2, 0.3); d.env_sampling_weight = 0.5
    yield "env_two_area_lights", d, RenderParams(spp=8, sampler="independent", rfilter="box")
    d = smoke_scene(36, 36, res=8, scale=5.0)
    d.env_radiance = (0.3, 0.4, 0.6)
    yield "env_volpath_smoke", d, RenderParams(spp=8, sampler="independent", rfilter="gaussian", integrator="volpath")
    # instancing: one group of spheres placed five times (stress scene), a second group with UV tangent frames under rotation + non-uniform
    # scale + shear; flattened copy of the same geometry for the equivalence check lives in the tests
    d = stress_scene(5, 12, 12, 40, 40, instanced=True)
    P, N, UV, I = uv_sphere((0, 0, 0), 0.6, 10, 20, with_uv=True)
    aniso = Bsdf("roughconductor", distribution="beckmann", alpha_u=0.15, alpha_v=0.4, eta=(0.2004, 0.9240, 1.1022), k=(3.9129, 2.4528, 2.1421))
    d.meshes.append(Mesh(P, I, N=N, UV=UV, bsdf=aniso, group=1))
    Pc, Ic = cube_mesh((-0.4, -0.9, -0.4), (0.4, -0.6, 0.4))
    d.meshes.append(Mesh(Pc, Ic, bsdf=Bsdf("diffuse", reflectance=(0.2, 0.6, 0.3)), group=1))
    c, s_ = np.cos(0.7), np.sin(0.7)
    M = np.eye(4); M[:3, :3] = np.array([[c, 0, s_], [0, 1, 0], [-s_, 0, c]]) @ np.diag([1.3, 0.8, 1.0]); M[0, 1] = 0.2; M[:3, 3] = (0.5, 2.6, -1.0)
    d.instances.append(Instance(1, M.astype(np.float32)))
    M2 = np.eye(4); M2[:3, :3] *= 0.7; M2[:3, 3] = (-2.0, 2.2, 0.5)
    d.instances.append(Instance(1, M2.astype(np.float32)))
    yield "instances_sobol", d, RenderParams(spp=8, sampler="sobol", rfilter="box")
    yield "instances_counter_depth3", d, RenderParams(spp=8, sampler="independent", rfilter="gaussian", max_depth=3)
    # film crop window (film.cpp:36-47, perspective.cpp:133-153): the crop is the film the integrator sees (blocks, Sobol' resolution,
    # sample positions relative to it); sizes that are multiples of neither the 8x8 work tiles nor the 32x32 blocks
    d = cornell_box(96, 64)
    d.camera = dataclasses.replace(d.camera, crop=(17, 9, 43, 33))
    yield "crop_cbox_sobol", d, RenderParams(spp=8, sampler="sobol", rfilter="gaussian")
    d = cornell_box(80, 80)
    d.camera = dataclasses.replace(d.camera, crop=(40, 0, 40, 37), aperture_radius=20.0, focus_distance=1000.0)
    yield "crop_thinlens_counter", d, RenderParams(spp=4, sampler="independent", rfilter="box", max_depth=5)


def sky_image(w=64, h=32, seed=4, sun=40.0):
    """A synthetic latitude-longitude radiance map: cubed noise, a small very bright patch (sampling must find it), a darker lower half."""
    rng = np.random.default_rng(seed)
    img = (rng.random((h, w, 3)) ** 3).astype(np.float32) * 0.8
    img[h // 6:h // 6 + max(1, h // 10), w // 3:w // 3 + max(1, w // 16)] += np.float32(sun)
    img[h // 2:, :] *= np.float32(0.2)
    return img


def envmap_rotation():
    c, s = np.cos(0.6), np.sin(0.6)
    M = np.eye(4, dtype=np.float32)
    M[:3, :3] = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]], np.float32) @ np.array([[1, 0, 0], [0, np.cos(0.3), -np.sin(0.3)], [0, np.sin(0.3), np.cos(0.3)]], np.float32)
    return M


def image_cases_env():
    """Image-level pins of the `envmap` emitter (src/emitters/envmap.cpp) through the assembled reference renderer: seen directly (the
    filtered look-up with the sensor's ray differentials), as the only light, next to an area light (emitter selection + MIS both ways),
    hidden, under volpath, and with a map whose sizes are not powers of two.  Fixture: tests/golden/path_ref_env.npz."""
    from mitsuba_b200.scene import Bsdf, EnvMap, RenderParams, cornell_box, material_ball, smoke_scene
    gold = Bsdf("roughconductor", distribution="ggx", alpha_u=0.2, alpha_v=0.2, eta=(0.2004, 0.9240, 1.1022), k=(3.9129, 2.4528, 2.1421))
    d = material_ball(gold, 40, 40, n_theta=16, n_phi=32)
    d.meshes = [m for m in d.meshes if m.radiance is None]
    d.envmap = EnvMap(pixels=sky_image(), scale=1.5, to_world=envmap_rotation())
    yield "envmap_only_ball", d, RenderParams(spp=8, sampler="sobol", rfilter="gaussian")
    d = cornell_box(36, 36)
    d.meshes = [m for i, m in enumerate(d.meshes) if i != 1]
    d.envmap = EnvMap(pixels=sky_image(50, 25, seed=9, sun=15.0), scale=0.5, sampling_weight=2.0)   # identity toWorld, odd sizes (7 levels)
    yield "envmap_plus_area_cbox", d, RenderParams(spp=8, sampler="independent", rfilter="box")
    yield "envmap_hidden_cbox", d, RenderParams(spp=4, sampler="sobol", rfilter="gaussian", hide_emitters=True, max_depth=5)
    d = material_ball(Bsdf("roughdielectric", distribution="beckmann", alpha_u=0.1, alpha_v=0.1, int_ior=1.5, ext_ior=1.0), 32, 32, n_theta=12, n_phi=24)
    d.envmap = EnvMap(pixels=sky_image(32, 16, seed=2), to_world=envmap_rotation(), sampling_weight=0.5)  # the area light stays: two emitters
    yield "envmap_glass_ball", d, RenderParams(spp=8, sampler="sobol", rfilter="box")
    d = smoke_scene(36, 36, res=8, scale=5.0)
    d.envmap = EnvMap(pixels=sky_image(16, 8, seed=3, sun=5.0), scale=0.7)
    yield "envmap_volpath_smoke", d, RenderParams(spp=8, sampler="independent", rfilter="gaussian", integrator="volpath")


def reference_envmap_inverse(lib, desc):
    """Transform::inverse() of the map's toWorld as the reference computes it (float Gauss-Jordan) -- matrix set-up is host work."""
    if desc.envmap is None or desc.envmap.to_world is None:
        return None
    inv = np.zeros((4, 4), np.float32)
    lib.pathref_transform_inverse(_f(np.ascontiguousarray(desc.envmap.to_world, np.float32)), _f(inv))
    return inv


def image_cases_tex():
    """Image-level pins of `bitmap` textures through the assembled reference renderer (the reference's BitmapTexture / Texture2D /
    Intersection::computePartials and the sensors' ray differentials; the pyramid enters the plugin as a MIP map cache file holding the
    oracle's resampling of the image): all four filters, repeat / mirror / clamp wrap modes, uv scale and offset, RGB and luminance images,
    an image above 1 (energy-conservation scale) behind `twosided` through a thin lens, and textures on plastic's diffuseReflectance
    and a rough conductor's specularReflectance.  Fixture: tests/golden/path_ref_tex.npz."""
    import dataclasses
    from mitsuba_b200.scene import Bsdf, RenderParams, textured_scene
    for ft, smp, filt in (("ewa", "sobol", "gaussian"), ("trilinear", "independent", "box"), ("bilinear", "sobol", "box"), ("nearest", "sobol", "gaussian")):
        yield "tex_" + ft, textured_scene(40, 40, filter_type=ft, tex_res=32, n_theta=12, n_phi=24), RenderParams(spp=8, sampler=smp, rfilter=filt)
    d = textured_scene(36, 36, two_sided=True, tex_res=24, n_theta=10, n_phi=20)
    d.camera = dataclasses.replace(d.camera, aperture_radius=0.05, focus_distance=5.0)
    ball = d.meshes[1].bsdf.reflectance
    ball.pixels = (ball.pixels * np.float32(1.7)).astype(np.float32)
    yield "tex_twosided_thinlens_scaled", d, RenderParams(spp=8, sampler="sobol", rfilter="box")
    d = textured_scene(40, 40, tex_res=32, n_theta=12, n_phi=24)
    d.meshes[1].bsdf = Bsdf("plastic", diffuse_reflectance=d.meshes[1].bsdf.reflectance, nonlinear=True, int_ior=1.49)
    d.meshes[0].bsdf = Bsdf("twosided", nested=Bsdf("plastic", diffuse_reflectance=d.meshes[0].bsdf.reflectance, specular_reflectance=(0.8, 0.9, 1.0)))
    d.meshes[3].bsdf = Bsdf("roughconductor", distribution="ggx", alpha_u=0.3, alpha_v=0.3, eta=(0.2004, 0.9240, 1.1022), k=(3.9129, 2.4528, 2.1421),
                            specular_reflectance=d.meshes[3].bsdf.reflectance)
    yield "tex_plastic_and_conductor", d, RenderParams(spp=8, sampler="sobol", rfilter="gaussian")


# ---------------------------------------------------------------------------------------------------------------------------
# inputs the fixtures above do not hold: tests/gen_golden.py (unseen_ref) stores the reference's answers to them in
# tests/golden/unseen_ref.{json,npz}, and tests/test_oracle_*.py hold the oracle to them
# ---------------------------------------------------------------------------------------------------------------------------
FDR_ETAS = (1.5, 1.0 / 1.5, 1.33, 1.49)
ENVMAP_PROBE_CASES = ("envmap_only_ball", "envmap_plus_area_cbox")


def digest(a):
    """SHA-256 of an array's dtype, shape and values, with every NaN one NaN and -0 as +0 (the equality `same` of the tests checks): what
    the unseen-input fixture keeps of a large output that is compared bit for bit, instead of the array.  Hash an integer view to keep
    the sign of zero and the NaN payloads."""
    import hashlib
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.ascontiguousarray(np.where(np.isnan(a), a.dtype.type(np.nan), a + a.dtype.type(0)))
    return hashlib.sha256(repr((a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()


def emitter_sample_views(a):
    """The parts of Scene::sampleEmitterDirect records (n, 12) that are compared: the success flag of every record, whole successful records."""
    ok = a[:, 8] == 1
    return {"flag": a[:, 8], "ok_rows": a[ok]}


def intersection_views(a):
    """The parts of Scene::rayIntersect records (n, 24) that are compared: the hit flag of every ray, columns 0-18 and 20 of the hits."""
    hit = a[:, 21] == 1
    return {"hit": a[:, 21], "hit_cols": a[hit][:, :19], "hit_col20": a[hit, 20]}


def unseen_image_cases():
    """Two more films of the assembled reference renderer: a Cornell box and a textured scene with mirror wrapping."""
    from mitsuba_b200.scene import RenderParams, cornell_box, textured_scene
    yield "cbox_56x40", cornell_box(56, 40), RenderParams(spp=12, sampler="sobol", rfilter="gaussian", seed=3)
    yield "textured_mirror", textured_scene(44, 36, filter_type="ewa", tex_res=48, wrap="mirror", n_theta=10, n_phi=20), \
        RenderParams(spp=6, sampler="sobol", rfilter="gaussian", seed=5)


def emitter_probe_inputs():
    """Reference points / selection samples for Scene::sampleEmitterDirect (400) and film positions of camera rays into the instanced
    scene (3000)."""
    rng = np.random.default_rng(99)
    n = 400
    refp = np.zeros((n, 6), np.float32)
    refp[:, 0:3] = rng.uniform(50, 500, (n, 3)); refp[:, 3:6] = _dirs(rng, n)
    smp = rng.random((n, 2)).astype(np.float32)
    pos = (rng.random((3000, 2)) * 40).astype(np.float32)
    return refp, smp, pos


def envmap_probe_inputs(n=3000):
    """Per case of ENVMAP_PROBE_CASES: directions (poles and the seam first), the same with ray differentials from a fraction of a texel
    to strongly anisotropic footprints, reference points + directions for the direct-sampling density, and direct-sampling samples."""
    rng = np.random.default_rng(5)
    for name in ENVMAP_PROBE_CASES:
        rays = np.zeros((n, 6), np.float32); rays[:, 3:] = _dirs(rng, n)
        rays[:3, 3:] = [(0, 1, 0), (0, -1, 0), (0, 0, 1)]
        rd = np.zeros((n, 18), np.float32); rd[:, :6] = rays
        for k, sc in ((9, 0.02), (15, 0.3)):
            v = rays[:, 3:] + sc * rng.standard_normal((n, 3)).astype(np.float32) * rng.random((n, 1)).astype(np.float32) ** 2
            rd[:, k:k + 3] = v / np.linalg.norm(v, axis=1, keepdims=True)
        refp = np.zeros((n, 6), np.float32)
        refp[:, 0:3] = rng.uniform(-1, 1, (n, 3)) if name == "envmap_only_ball" else rng.uniform(50, 500, (n, 3))
        refp[:, 3:6] = _dirs(rng, n)
        dd = _dirs(rng, n).astype(np.float32)
        smp = rng.random((n, 2)).astype(np.float32)
        yield name, rays, rd, refp, dd, smp
