"""The oracle's component functions against the REFERENCE's own code.

oracle/core_ref_shim.cpp compiles the reference's microfacet.h, triaccel.h, aabb.h, triangle.cpp, warp.cpp, util.cpp, quad.cpp, math.cpp,
pmf.h and qmc.h from where they lie under /root/reference (behind the stand-in headers of oracle/shim_core/) into
oracle/_ref/libcoreref.so; tests/gen_golden.py ran it on the seeded inputs of tests/ref_pins.py and committed the outputs as
tests/golden/core_ref.npz.  The oracle must reproduce every value bit for bit (NaN = NaN)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import ref_pins
from oracle import oracle_api as O

HERE = os.path.dirname(os.path.abspath(__file__))


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype.kind == "f":
        return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.nan_to_num(a, nan=0.0), np.nan_to_num(b, nan=0.0))
    return np.array_equal(a, b)


@pytest.fixture(scope="module")
def oracle_outputs():
    return ref_pins.run(O.lib(), "orc_", ref_pins.inputs())


def test_oracle_components_match_reference_golden(oracle_outputs):
    g = np.load(os.path.join(HERE, "golden", "core_ref.npz"))
    assert len(g.files) == len(oracle_outputs) == 71
    bad = [k for k in g.files if not same(g[k], oracle_outputs[k])]
    assert not bad, bad
    # the fixture is not vacuous: hits and misses, degenerate triangles, total internal reflection, zero-weight pmf bins
    assert 0.2 < g["triaccel_hits"][:, 0].mean() < 0.95 and g["triaccel_status"].sum() >= 6
    assert (g["fresnel_dielectric_0.6667"][:, 0] == 1.0).sum() > 10 and g["aabb"][:, 0].min() == 0 and g["aabb"][:, 0].max() == 1


# The reference's outputs on inputs the fixtures above do not hold, written by tests/gen_golden.py (unseen_ref) from the libraries
# oracle/Makefile compiles out of the reference's sources: arrays, or ref_pins.digest for the large outputs compared bit for bit.  The
# `*_when_present` tests below compare the oracle with these stored outputs; they do not call the reference's libraries, and run everywhere.
UNSEEN = json.load(open(os.path.join(HERE, "golden", "unseen_ref.json")))
UNSEEN_ARRAYS = np.load(os.path.join(HERE, "golden", "unseen_ref.npz"))


def unseen_mismatches(prefix, got):
    """Names of the outputs in `got` whose digest is not the reference's stored under prefix + name (every stored one must be there)."""
    stored = {k[len(prefix):] for k in UNSEEN if k.startswith(prefix)}
    assert stored == set(got), sorted(stored ^ set(got))
    return [k for k in got if ref_pins.digest(got[k]) != UNSEEN[prefix + k]]


def test_oracle_components_match_live_reference_when_present():
    """The digests of the reference's core math on ref_pins.inputs(seed=99) and its fresnelDiffuseReflectance values (tests/golden/unseen_ref.json)."""
    got = ref_pins.run(O.lib(), "orc_", ref_pins.inputs(seed=99))
    assert len(got) == 71 and not unseen_mismatches("core/", got)
    from mitsuba_b200.scene import fresnel_diffuse_reflectance
    # util.cpp:807-859 with fast = false (Gauss-Lobatto): the loaders integrate it numerically
    for eta, ref in zip(ref_pins.FDR_ETAS, UNSEEN["fresnel_diffuse_reflectance"]):
        assert abs(float.fromhex(ref) - fresnel_diffuse_reflectance(eta)) < 2e-6


# plastic evaluates util.cpp's fresnelDiffuseReflectance(1/eta, fast = false) -- an adaptive Gauss-Lobatto quadrature in float -- once
# at construction; the host side of this repository integrates the same function with Simpson's rule in double, which can differ in
# the last bit of that constant.  Everything else is bit-exact.
LAST_BIT_OF_A_CONSTANT = {"plastic": 5e-5, "twosided_two": 5e-5}


def _bsdf_close(name, ref, got):
    tol = LAST_BIT_OF_A_CONSTANT.get(name)
    for k, r in ref.items():
        g = np.asarray(got[k])
        r = np.asarray(r)
        if tol is None:
            if not same(r, g):
                return k
        else:
            if r.dtype.kind != "f":
                if not np.array_equal(r, g):
                    return k
            elif not np.allclose(g, r, rtol=tol, atol=1e-7, equal_nan=True):
                return k
    return None


def test_oracle_bsdfs_match_reference_plugins_golden():
    """tests/golden/bsdf_ref.npz: outputs of the reference's own BSDF plugin sources (see tests/gen_golden.py).  16 of the 18
    configurations -- every microfacet model, coating, dielectric, conductor, twosided -- are reproduced bit for bit."""
    from bsdf_configs import configs
    g = np.load(os.path.join(HERE, "golden", "bsdf_ref.npz"))
    x = ref_pins.bsdf_inputs()
    exact = 0
    for name, b in configs().items():
        ref = {k.split("/", 1)[1]: g[k] for k in g.files if k.startswith(name + "/")}
        assert len(ref) == 8, name
        got = ref_pins.run_bsdf_oracle(b, x)
        assert _bsdf_close(name, ref, got) is None, (name, _bsdf_close(name, ref, got))
        exact += name not in LAST_BIT_OF_A_CONSTANT
        assert np.any(ref["sample"][:, 3:6] != 0), name  # the fixture holds successful samples
    assert exact == 16


def test_oracle_bsdfs_match_live_reference_plugins_when_present():
    """The reference's BSDF plugins on ref_pins.bsdf_inputs(seed=4321): digests (tests/golden/unseen_ref.json), arrays for the two
    configurations compared within a tolerance (tests/golden/unseen_ref.npz)."""
    from bsdf_configs import configs
    g = UNSEEN_ARRAYS
    x = ref_pins.bsdf_inputs(seed=4321)  # directions the fixture has not seen
    for name, b in configs().items():
        got = ref_pins.run_bsdf_oracle(b, x)
        assert len(got) == 8, name
        if name in LAST_BIT_OF_A_CONSTANT:
            ref = {k: g[f"bsdf/{name}/{k}"] for k in got}
            assert _bsdf_close(name, ref, got) is None, (name, _bsdf_close(name, ref, got))
        else:
            assert not unseen_mismatches(f"bsdf/{name}/", got), (name, unseen_mismatches(f"bsdf/{name}/", got))


def _oracle_scene(W, H):
    from mitsuba_b200.scene import cornell_box
    return O.OracleScene(cornell_box(W, H))


def test_oracle_partials_filters_splat_and_sobol_match_reference_golden():
    """tests/golden/render_ref.npz (see tests/gen_golden.py): Intersection::computePartials incl. its degenerate branches, the
    discretised box / gaussian filters, 300 ImageBlock::put splats per filter (block borders, clamping), and the SobolSampler plugin's
    first 24 dimensions for five (scramble, resolution, spp, pixel, sample) settings -- all bit for bit."""
    g = np.load(os.path.join(HERE, "golden", "render_ref.npz"))
    got = ref_pins.run_render(O.lib(), "orc_", ref_pins.render_inputs(), _oracle_scene)
    assert len(g.files) == len(got) == 16
    assert not [k for k in g.files if not same(g[k], got[k])]
    assert g["put1_ok"].all() and g["put1_data"][..., 4].sum() > 100
    # rejected samples (imageblock.h:136-139: negative / non-finite values): closed form, no contribution
    L = O.lib()
    pos = np.array([[15.0, 25.0]] * 4, np.float32)
    val = np.array([[-1, 0, 0, 1], [np.nan, 0, 0, 1], [np.inf, 0, 0, 1], [0, 0, 0, -0.5]], np.float32)
    data, ok = np.zeros((16, 20, 5), np.float32), np.ones(4, np.int32)
    L.orc_block_put(10, 20, 16, 12, 1, C.c_float(0.5), 4, ref_pins._f(pos), ref_pins._f(val), ref_pins._f(data), ok.ctypes.data_as(C.POINTER(C.c_int)))
    assert not ok.any() and not data.any()


def test_oracle_partials_filters_splat_and_sobol_match_live_reference_when_present():
    """tests/golden/unseen_ref.npz: the reference's outputs on ref_pins.render_inputs(seed=55)."""
    got = ref_pins.run_render(O.lib(), "orc_", ref_pins.render_inputs(seed=55), _oracle_scene)
    ref = {k[len("render/"):]: UNSEEN_ARRAYS[k] for k in UNSEEN_ARRAYS.files if k.startswith("render/")}
    assert len(ref) == len(got) == 16
    assert not [k for k in ref if not same(ref[k], got[k])]


def test_oracle_images_match_the_reference_renderer_golden():
    """tests/golden/path_ref.npz: films rendered by a `path` renderer assembled from the reference's own sources (MIPathTracer::Li,
    renderBlock, Scene, ShapeKDTree, sensor, emitter, Sobol' sampler, filters, ImageBlock, BSDF plugins; see tests/gen_golden.py).
    Starting from the sampleToCamera matrix of the reference's sensor (camera set-up is host work), the oracle reproduces every film
    BIT FOR BIT -- rgb, alpha and weight channels -- except the plastic ball (last bit of one constructor constant, see above)."""
    g = np.load(os.path.join(HERE, "golden", "path_ref.npz"))
    n = 0
    for name, desc, rp in ref_pins.image_cases():
        ref, s2c = g[name + "/film"], g[name + "/s2c"]
        film, _ = O.OracleScene(desc, sample_to_camera=s2c).render(rp)
        film = np.asarray(film).reshape(ref.shape)
        if name == "ball_plastic":
            assert np.sqrt(((film - ref) ** 2).sum() / (ref ** 2).sum()) < 1e-6
        else:
            assert np.array_equal(film, ref), (name, float(np.abs(film - ref).max()))
        assert ref[..., :3].max() > 0.1 and ref[..., 4].min() > 0
        # and the host-side derivation of the camera matrix agrees with the reference's to float rounding
        assert np.allclose(desc.camera.sample_to_camera().astype(np.float32), s2c, rtol=1e-6, atol=1e-7)
        n += 1
    assert n == 19


def _unseen_film(name):
    """A film of ref_pins.unseen_image_cases() against the reference renderer's (tests/golden/unseen_ref.npz), bit for bit."""
    desc, rp = next((d, r) for n, d, r in ref_pins.unseen_image_cases() if n == name)
    ref = UNSEEN_ARRAYS[name + "/film"]
    film, _ = O.OracleScene(desc, sample_to_camera=UNSEEN_ARRAYS[name + "/s2c"]).render(rp)
    film = np.asarray(film).reshape(ref.shape)
    assert np.array_equal(film, ref), (name, int((film != ref).sum()), float(np.abs(film - ref).max()))
    assert ref[..., :3].max() > 0.1 and ref[..., 4].min() > 0


def test_oracle_images_match_the_live_reference_renderer_when_present():
    _unseen_film("cbox_56x40")


def _ext_oracle(desc, g, name, host_inverses=False):
    inv = g[name + "/instance_inverses"] if (name + "/instance_inverses") in g.files and not host_inverses else None
    return O.OracleScene(desc, sample_to_camera=g[name + "/s2c"], instance_inverses=inv)


def test_oracle_images_of_thinlens_constant_emitter_and_instances_match_the_reference_renderer_golden():
    """tests/golden/path_ref_ext.npz: `thinlens` (src/sensors/thinlens.cpp), `constant` (src/emitters/constant.cpp; alone, next to an area
    light with samplingWeight 2, hidden, under volpath) and `shapegroup` / `instance` (src/shapes/{shapegroup,instance}.cpp; rotation,
    non-uniform scale, shear, UV tangent frames) rendered by the renderer assembled from the reference's sources -- reproduced BIT FOR
    BIT by the oracle.  Two things this pin established (both now restated in the oracle and the device host code):
      * Scene::m_emitters holds scene-level emitters first, the shapes' area emitters behind them (Scene::addChild appends the former at
        once, scene.cpp:510-516, Scene::initialize -> addShape the latter, :322-335 / :570-571), whatever the document order;
      * Transform::operator()(Point) divides by w unless w == 1 exactly, and the float Gauss-Jordan inverse of an affine toWorld can have a
        last row like (0, 3e-8, 0, 0.99999994): the reference's instanced rays go through that division.  Matrix set-up is host work,
        so the oracle is handed the reference's inverses here (like sampleToCamera); with this repository's own exactly-affine
        float64-derived inverses the images agree to the rounding of those matrices (second assertion)."""
    g = np.load(os.path.join(HERE, "golden", "path_ref_ext.npz"))
    n = 0
    for name, desc, rp in ref_pins.image_cases_ext():
        ref = g[name + "/film"]
        film = np.asarray(_ext_oracle(desc, g, name).render(rp)[0]).reshape(ref.shape)
        assert np.array_equal(film, ref), (name, float(np.abs(film - ref).max()))
        assert ref[..., :3].max() > 0.1 and ref[..., 4].min() > 0
        if desc.instances:
            own = np.asarray(_ext_oracle(desc, g, name, host_inverses=True).render(rp)[0]).reshape(ref.shape)
            assert np.array_equal(own[..., 3:], ref[..., 3:])   # same splats: alpha and weight channels
            assert np.sqrt(((own - ref) ** 2).sum() / (ref ** 2).sum()) < 1e-3
        n += 1
    assert n == 11


def test_emitter_order_and_instanced_records_match_the_live_reference_when_present():
    """Component probes behind the images above, against the reference's stored outputs (tests/golden/unseen_ref.*): Scene::sampleEmitterDirect
    on a scene with an area light AND a constant emitter (emitter selection order, bounding-sphere sampling, shadow rays) and Scene::rayIntersect
    on the instanced scene (nested kd-tree, Instance::fillIntersectionRecord) -- bit for bit, on inputs the fixture does not hold."""
    g = UNSEEN_ARRAYS
    cases = {name: (desc, rp) for name, desc, rp in ref_pins.image_cases_ext()}
    refp, smp, pos = ref_pins.emitter_probe_inputs()
    # emitter selection + direct sampling
    desc, rp = cases["env_plus_area_cbox"]
    a = g["emitter/sample"]
    b = O.OracleScene(desc).sample_emitter_direct(refp, smp)
    ok = a[:, 8] == 1
    assert np.array_equal(a[:, 8], b[:, 8]) and ok.sum() > 50
    assert np.array_equal(a[ok], b[ok])
    # samplingWeight 2 : 1 -> the environment owns [0, 2/3) of the selection sample and comes first
    far = np.linalg.norm(a[:, 9:12] - refp[:, 0:3], axis=1) > 700
    assert far[ok & (smp[:, 0] < 0.6)].all() and not far[ok & (smp[:, 0] > 0.7)].any()
    # instanced intersection records of camera rays from the reference's sampleToCamera and instance inverses
    desc, rp = cases["instances_sobol"]
    o = O.OracleScene(desc, sample_to_camera=g["instances/s2c"], instance_inverses=list(g["instances/inverses"]))
    b = o.intersect_full(o.camera_rays(pos))
    assert not unseen_mismatches("instances/", ref_pins.intersection_views(b))
    assert (b[:, 21] == 1).sum() > 1000


def _env_desc(desc, g, name):
    import dataclasses
    if (name + "/env_to_local") in g.files:
        desc.envmap = dataclasses.replace(desc.envmap, to_local=g[name + "/env_to_local"])
    return desc


def test_oracle_images_with_an_environment_map_match_the_reference_renderer_golden():
    """tests/golden/path_ref_env.npz: the reference's EnvironmentMap (src/emitters/envmap.cpp) inside the assembled reference renderer --
    seen directly by the camera (EWA look-up driven by the sensor's ray differentials, envmap.cpp:392-406), as the only light, next to an
    area light with samplingWeight 2 / 0.5, hidden, under volpath, power-of-two and odd map sizes -- reproduced BIT FOR BIT by the oracle
    (orc_envmap.h).  The pyramid the reference class reads is the oracle's resampling of the image (handed over as a MIP map cache file,
    the way a second Mitsuba run reads it); the CDF tables, look-ups, direction sampling and densities are the reference's own."""
    g = np.load(os.path.join(HERE, "golden", "path_ref_env.npz"))
    n = 0
    for name, desc, rp in ref_pins.image_cases_env():
        ref = g[name + "/film"]
        film = np.asarray(O.OracleScene(_env_desc(desc, g, name), sample_to_camera=g[name + "/s2c"]).render(rp)[0]).reshape(ref.shape)
        assert np.array_equal(film, ref), (name, float(np.abs(film - ref).max()))
        assert ref[..., :3].max() > 0.1 and ref[..., 4].min() > 0
        n += 1
    assert n == 5


def test_environment_map_lookups_sampling_and_densities_match_the_live_reference_when_present():
    """Component probes behind the images above, on inputs the fixture does not hold: Scene::evalEnvironment without and with ray
    differentials, Scene::pdfEmitterDirect and Scene::sampleEmitterDirect for the environment map -- bit for bit against the digests of the
    reference's outputs (tests/golden/unseen_ref.json)."""
    import dataclasses
    g = UNSEEN_ARRAYS
    cases = {name: (desc, rp) for name, desc, rp in ref_pins.image_cases_env()}
    L = O.lib()
    for name, rays, rd, refp, dd, smp in ref_pins.envmap_probe_inputs():
        desc, rp = cases[name]
        if (name + "/to_local") in g.files:                                        # the reference's float inverse of toWorld
            desc.envmap = dataclasses.replace(desc.envmap, to_local=g[name + "/to_local"])
        o = O.OracleScene(desc)
        n = len(rays)
        ev, evd, pdf = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.float32)
        L.orc_eval_environment(o.h, C.c_uint64(n), 0, O._p(rays), O._p(ev))       # poles and the seam of the parameterisation first
        L.orc_eval_environment(o.h, C.c_uint64(n), 1, O._p(rd), O._p(evd))        # from a fraction of a texel to strongly anisotropic footprints
        L.orc_pdf_environment_direct(o.h, C.c_uint64(n), O._p(refp), O._p(dd), O._p(pdf))
        sb = o.sample_emitter_direct(refp, smp)
        got = {"eval": ev, "eval_diff": evd, "pdf": pdf, **{"sample_" + k: v for k, v in ref_pins.emitter_sample_views(sb).items()}}
        assert not unseen_mismatches(name + "/", got), (name, unseen_mismatches(name + "/", got))
        assert ev.max() > 1 and evd.max() > 1 and pdf.max() > 0.5 and (sb[:, 8] == 1).sum() > 100


def test_oracle_images_with_bitmap_textures_match_the_reference_renderer_golden():
    """tests/golden/path_ref_tex.npz: the reference's BitmapTexture (src/textures/bitmap.cpp), Texture2D::eval (texture.cpp:124-133),
    Intersection::computePartials (intersection.cpp:23-85) and the sensors' ray differentials inside the assembled reference renderer --
    four filters, three wrap modes, uv scale / offset, RGB and luminance images, an image above 1 behind `twosided` through a thin lens,
    textures on plastic's diffuseReflectance (the sampling weight from the texture's average) and on a rough conductor's
    specularReflectance -- reproduced BIT FOR BIT by the oracle (the plastic scene: to the last bit of one constructor constant, 1e-6).  This closes what the look-up level pins (mipmap_ref.npz) left to closed
    forms: the uv transform, the partials and everything between the texture and the film."""
    g = np.load(os.path.join(HERE, "golden", "path_ref_tex.npz"))
    n = 0
    for name, desc, rp in ref_pins.image_cases_tex():
        ref = g[name + "/film"]
        film = np.asarray(O.OracleScene(desc, sample_to_camera=g[name + "/s2c"]).render(rp)[0]).reshape(ref.shape)
        if name == "tex_plastic_and_conductor":   # plastic: the last bit of one constructor constant, as for ball_plastic above
            assert np.array_equal(film[..., 3:], ref[..., 3:])
            assert np.sqrt(((film - ref) ** 2).sum() / (ref ** 2).sum()) < 1e-6
        else:
            assert np.array_equal(film, ref), (name, float(np.abs(film - ref).max()))
        assert ref[..., :3].max() > 0.1 and ref[..., 4].min() > 0
        n += 1
    assert n == 6


def test_oracle_textured_image_matches_the_live_reference_renderer_when_present():
    _unseen_film("textured_mirror")


def test_environment_map_image_the_plugin_marshals_is_the_stored_level_zero_when_present():
    """What the Mitsuba-side plugin reads back from an EnvironmentMap instance (Emitter::getBitmap -> TMIPMap::toBitmap, envmap.cpp:632-634):
    the half-precision level 0 of its pyramid -- bit for bit the oracle's level 0 -- so the pyramid b2_scene_commit rebuilds from it starts from
    the same texels the reference samples.  The images read back through the translation units the plugin's library links are stored in
    tests/golden/unseen_ref.npz."""
    cases = {name: (desc, rp) for name, desc, rp in ref_pins.image_cases_env()}
    for name in ref_pins.ENVMAP_PROBE_CASES:
        assert np.array_equal(UNSEEN_ARRAYS["bitmap/" + name], ref_pins.envmap_pyramid(cases[name][0].envmap)[0]), name


def test_conductor_material_presets_match_the_reference_spectrum_code():
    """material="Cu" etc. of the conductor plugins (roughconductor.cpp:174-190): the committed table (mitsuba_b200/data/conductor_presets.txt)
    against what the reference's InterpolatedSpectrum + Spectrum::fromContinuousSpectrum make of data/ior/*.spd (tests/golden/unseen_ref.npz),
    and against the values the reference's documentation quotes for copper."""
    from mitsuba_b200.scene import Bsdf, conductor_preset
    eta, k = conductor_preset("Cu")
    assert np.allclose(eta, (0.2004, 0.9240, 1.1022), atol=1e-4) and np.allclose(k, (3.9129, 2.4528, 2.1421), atol=1e-4)
    d = Bsdf("roughconductor", material="Au").flat()
    from mitsuba_b200.scene import lookup_ior
    assert np.allclose(d["etaC"], np.float32(conductor_preset("Au")[0]) / np.float32(lookup_ior("air", "air")), rtol=1e-6)   # / extEta (air)
    g = UNSEEN_ARRAYS
    ref = dict(zip(g["conductor_presets/names"], g["conductor_presets/eta_k"]))
    n = 0
    for line in open(os.path.join(HERE, "..", "mitsuba_b200", "data", "conductor_presets.txt")):
        t = line.split()
        if not t or t[0].startswith("#"):
            continue
        assert np.array_equal(np.float32([float.fromhex(x) for x in t[1:7]]), ref[t[0]]), t[0]
        n += 1
    assert n == len(ref) >= 60
