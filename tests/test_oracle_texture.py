"""Oracle + host side of the `bitmap` texture (SURVEY.md 8f-4): MIP pyramid, look-ups, uv partials.

The reference holds no golden vectors for mipmap.h / bitmap.cpp, so the restatement is pinned by closed-form properties (partition of
unity, known-answer weights from an independent float64 derivation, analytic uv derivatives of a plane) and by a second,
independently written implementation (the host-side pyramid builder that feeds the device)."""
import ctypes as C
import json
import math
import os

import numpy as np
import pytest

from mitsuba_b200 import api
from mitsuba_b200.scene import Bsdf, Camera, Mesh, RenderParams, SceneDesc, Texture, checker_image, look_at, textured_scene
from oracle import oracle_api as O

WRAPS = ["repeat", "clamp", "mirror", "zero", "one"]


def one_texture_scene(tex, width=32, height=32):
    """A unit quad with uv = (x, y) in front of the camera, textured with `tex`."""
    P = np.array([(0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0)], np.float32)
    I = np.array([[0, 1, 2], [0, 2, 3]], np.uint32)
    UV = np.array([(0, 0), (1, 0), (1, 1), (0, 1)], np.float32)
    quad = Mesh(P, I, UV=UV, bsdf=Bsdf("diffuse", reflectance=tex), name="quad")
    L = Mesh(P + np.array([0, 0, 3], np.float32), I[:, ::-1].copy(), bsdf=Bsdf("diffuse", reflectance=(0, 0, 0)), radiance=(5.0, 5.0, 5.0), name="light")
    cam = Camera(look_at((0.5, 0.5, 2.0), (0.5, 0.5, 0), (0, 1, 0)), fov=40.0, near=0.1, far=100.0, width=width, height=height)
    return SceneDesc([quad, L], cam)


def lanczos2(x):
    x = abs(x)
    if x < 1e-4:
        return 1.0
    if x > 2:
        return 0.0
    return math.sin(math.pi * x) * math.sin(math.pi * x / 2) / (math.pi * x * math.pi * x / 2)


def wrap_index(mode, pos, res):
    if 0 <= pos < res:
        return pos, None
    if mode == "repeat":
        return pos % res, None
    if mode == "clamp":
        return min(max(pos, 0), res - 1), None
    if mode == "mirror":
        p = pos % (2 * res)
        return (2 * res - p - 1 if p >= res else p), None
    return 0, (0.0 if mode == "zero" else 1.0)


def resample_1d(src, trg_res, mode):
    """Independent float64 statement of Resampler (rfilter.h:107-190) + resampleAndClamp for one line."""
    src_res = len(src)
    scale = src_res / trg_res
    radius = 2.0 * scale
    taps = math.ceil(radius * 2)
    out = np.zeros(trg_res)
    for i in range(trg_res):
        center = (i + 0.5) / trg_res * src_res
        start = math.floor(center - radius + 0.5)
        w = np.array([lanczos2((start + j + 0.5 - center) / scale) for j in range(taps)])
        w /= w.sum()
        acc = 0.0
        for j in range(taps):
            k, const = wrap_index(mode, start + j, src_res)
            acc += (const if const is not None else src[k]) * w[j]
        out[i] = min(1.0, max(0.0, acc))
    return out


def test_pyramid_sizes_and_single_level_filters():
    img = checker_image(37, 21, rgb=False)  # w=37, h=21
    sc = O.OracleScene(one_texture_scene(Texture(img, filter_type="ewa")))
    info = sc.texture_info(0)
    assert info["sizes"] == [(37, 21), (19, 11), (10, 6), (5, 3), (3, 2), (2, 1), (1, 1)]  # max(1, (s + 1) / 2), mipmap.h:187-189
    for ft in ("nearest", "bilinear"):  # mipmap.h:185: no pyramid
        assert O.OracleScene(one_texture_scene(Texture(img, filter_type=ft))).texture_info(0)["levels"] == 1


@pytest.mark.parametrize("wrap", WRAPS)
def test_level1_matches_float64_derivation(wrap):
    rng = np.random.default_rng(11)
    img = rng.random((9, 14)).astype(np.float32)
    sc = O.OracleScene(one_texture_scene(Texture(img, filter_type="trilinear", wrap_u=wrap, wrap_v=wrap)))
    lvl1 = sc.texture_level(0, 1)[:, :, 0]
    tmp = np.stack([resample_1d(img[y].astype(np.float64), 7, wrap) for y in range(9)])          # x pass (bitmap.cpp:2258-2293)
    ref = np.stack([resample_1d(tmp[:, x], 5, wrap) for x in range(7)], axis=1)                    # y pass (:2296-2327)
    assert lvl1.shape == (5, 7)
    assert np.abs(lvl1 - ref).max() < 2e-6 + 2.0 ** -12   # the level is stored in half precision (values in [0, 1]: spacing <= 2^-11)
    from gen_golden import half_store
    assert np.mean(lvl1 == half_store(ref)) > 0.98        # and is the half rounding of the float64 derivation (but for near-ties)


def test_constant_image_is_constant_everywhere():
    img = np.full((20, 33, 3), 0.375, np.float32)
    for ft in ("nearest", "bilinear", "trilinear", "ewa"):
        sc = O.OracleScene(one_texture_scene(Texture(img, filter_type=ft, wrap_u="mirror", wrap_v="repeat")))
        info = sc.texture_info(0)
        for l in range(info["levels"]):
            assert np.abs(sc.texture_level(0, l) - 0.375).max() < 1e-6
        rng = np.random.default_rng(3)
        uv = (rng.random((200, 2)) * 4 - 2).astype(np.float32)
        pt = ((rng.random((200, 4)) - 0.5) * np.float32(0.2)).astype(np.float32)
        assert np.abs(sc.texture_eval(0, uv) - 0.375).max() < 1e-6
        assert np.abs(sc.texture_eval(0, uv, pt) - 0.375).max() < 1e-5


def test_energy_conservation_scale():
    img = np.full((4, 4), 2.0, np.float32)  # bsdf.cpp:93-107: scaled by 0.99 / max
    sc = O.OracleScene(one_texture_scene(Texture(img, filter_type="bilinear")))
    info = sc.texture_info(0)
    assert info["maximum"] == 2.0 and abs(info["bsdf_scale"] - 0.495) < 1e-7
    assert np.allclose(sc.texture_eval(0, np.array([[0.3, 0.6]], np.float32)), 2.0 * 0.495, atol=1e-6)


@pytest.mark.parametrize("wrap", WRAPS)
def test_unfiltered_lookup_is_bilinear_at_level0(wrap):
    rng = np.random.default_rng(5)
    img = rng.random((6, 8)).astype(np.float32)
    sc = O.OracleScene(one_texture_scene(Texture(img, filter_type="ewa", wrap_u=wrap, wrap_v=wrap)))
    uv = (rng.random((300, 2)) * 3 - 1).astype(np.float32)
    got = sc.texture_eval(0, uv)[:, 0]
    from gen_golden import half_store
    img = half_store(img)   # the texels as stored (bitmap.cpp:177-180)

    def texel(x, y):
        kx, cx = wrap_index(wrap, x, 8)
        if cx is not None:
            return cx
        ky, cy = wrap_index(wrap, y, 6)
        if cy is not None:
            return cy
        return float(img[ky, kx])
    for (u, v), g in zip(uv.astype(np.float64), got):
        fu, fv = u * 8 - 0.5, v * 6 - 0.5
        x, y = math.floor(fu), math.floor(fv)
        dx, dy = fu - x, fv - y
        ref = texel(x, y) * (1 - dx) * (1 - dy) + texel(x, y + 1) * (1 - dx) * dy + texel(x + 1, y) * dx * (1 - dy) + texel(x + 1, y + 1) * dx * dy
        assert abs(ref - g) < 2e-5
    # nearest: box look-up (mipmap.h:561-564)
    sn = O.OracleScene(one_texture_scene(Texture(img, filter_type="nearest", wrap_u="repeat", wrap_v="repeat")))
    gn = sn.texture_eval(0, uv)[:, 0]
    ref = np.array([img[math.floor(v * 6) % 6, math.floor(u * 8) % 8] for u, v in uv.astype(np.float64)])
    assert np.abs(gn - ref).max() < 1e-6


def test_filtered_lookup_known_answers():
    """A linear ramp is reproduced by a symmetric filter (trilinear exactly; EWA up to the asymmetry of its discrete taps, well below
    half a texel = 7.8e-3); footprints below one texel fall back to bilinear level 0."""
    w = h = 64
    ramp = np.tile((np.arange(w, dtype=np.float32) + 0.5) / w, (h, 1))  # value = u at texel centres
    for ft in ("trilinear", "ewa"):
        sc = O.OracleScene(one_texture_scene(Texture(ramp, filter_type=ft, wrap_u="clamp", wrap_v="clamp")))
        uv = np.stack([np.linspace(0.3, 0.7, 50), np.linspace(0.35, 0.65, 50)], -1).astype(np.float32)
        for foot in (0.001, 0.03, 0.06):  # sub-texel, ~2 texels, ~4 texels
            pt = np.tile(np.array([[foot, 0.0, 0.0, foot]], np.float32), (50, 1))
            got = sc.texture_eval(0, uv, pt)[:, 0]
            assert np.abs(got - uv[:, 0]).max() < (2e-3 if ft == "trilinear" else max(6e-3, 0.25 * foot)), (ft, foot)  # EWA: a fraction of the texel of the chosen level
        tiny = np.tile(np.array([[1e-4, 0.0, 0.0, 1e-4]], np.float32), (50, 1))
        assert np.array_equal(sc.texture_eval(0, uv, tiny), sc.texture_eval(0, uv))  # mipmap.h:661-663 / :708-709 with level 0
    # strongly anisotropic footprint: clamped to maxAnisotropy (mipmap.h:673-697), still centred on the ramp value
    sc = O.OracleScene(one_texture_scene(Texture(ramp, filter_type="ewa", max_anisotropy=4.0, wrap_u="clamp", wrap_v="clamp")))
    pt = np.tile(np.array([[0.002, 0.0, 0.0, 0.1]], np.float32), (50, 1))  # thin along u, long along v
    got = sc.texture_eval(0, uv, pt)[:, 0]
    assert np.abs(got - uv[:, 0]).max() < 6e-3


def test_uv_scale_and_offset():
    img = checker_image(32, 16, 4, 2, rgb=False)
    a = O.OracleScene(one_texture_scene(Texture(img, filter_type="bilinear", uscale=2.0, vscale=0.5, uoffset=0.25, voffset=-0.125)))
    b = O.OracleScene(one_texture_scene(Texture(img, filter_type="bilinear")))
    uv = np.random.default_rng(2).random((100, 2)).astype(np.float32)
    uv2 = (uv * np.array([2.0, 0.5], np.float32) + np.array([0.25, -0.125], np.float32)).astype(np.float32)
    assert np.array_equal(a.texture_eval(0, uv), b.texture_eval(0, uv2))  # texture.cpp:125


def test_primary_uv_partials_match_finite_differences():
    """Intersection::computePartials on a plane: (dudx, dvdx) = uv(pixel + 1 in x) - uv(pixel), times 1/sqrt(spp), to first order."""
    d = textured_scene(96, 96)
    sc = O.OracleScene(d)
    spp = 16
    rng = np.random.default_rng(9)
    pos = np.stack([rng.uniform(8, 88, 400), rng.uniform(50, 94, 400)], -1).astype(np.float32)  # lower part of the image: the ground quad
    base = sc.primary_partials(pos, spp)
    px = sc.primary_partials(pos + np.array([1, 0], np.float32), spp)
    py = sc.primary_partials(pos + np.array([0, 1], np.float32), spp)
    ok = (base[:, 0] == 1) & (px[:, 0] == 1) & (py[:, 0] == 1) & (base[:, 7] == 0) & (px[:, 7] == 0) & (py[:, 7] == 0)
    assert ok.sum() > 100
    s = 1.0 / math.sqrt(spp)
    fd_x = (px[ok, 1:3] - base[ok, 1:3]) * s
    fd_y = (py[ok, 1:3] - base[ok, 1:3]) * s
    got_x = base[ok][:, [3, 5]]  # dudx, dvdx
    got_y = base[ok][:, [4, 6]]  # dudy, dvdy
    scale = np.abs(fd_x).max() + np.abs(fd_y).max()
    assert np.abs(got_x - fd_x).max() < 0.05 * scale
    assert np.abs(got_y - fd_y).max() < 0.05 * scale


def test_constant_texture_renders_like_constant_reflectance():
    img = np.full((8, 8, 3), 1.0, np.float32) * np.array([0.6, 0.4, 0.3], np.float32)
    rp = RenderParams(spp=8, sampler="sobol", rfilter="box")
    f1, s1 = O.OracleScene(one_texture_scene(Texture(img, filter_type="ewa"))).render(rp)
    from gen_golden import half_store
    f2, s2 = O.OracleScene(one_texture_scene(tuple(float(v) for v in half_store(np.array([0.6, 0.4, 0.3], np.float32))))).render(rp)  # texels are stored as half
    assert s1["rays"] == s2["rays"]
    assert np.abs(O.develop(f1) - O.develop(f2)).max() < 1e-5


def test_textured_render_differs_by_filter_only_on_primary_hits():
    """Secondary bounces use the unfiltered look-up (bitmap.cpp:400-421): with max_depth = 2 + hidden direct view the image of the
    ewa and the bilinear texture differ only through the camera-ray look-ups, so a far-away, minified texture gets blurrier with ewa."""
    noise = np.random.default_rng(4).random((256, 256)).astype(np.float32)
    rp = RenderParams(spp=4, sampler="sobol", rfilter="box", max_depth=2)
    imgs = {}
    for ft in ("bilinear", "ewa"):
        d = one_texture_scene(Texture(noise, filter_type=ft, uscale=8.0, vscale=8.0), 48, 48)
        f, _ = O.OracleScene(d).render(rp)
        imgs[ft] = O.develop(f)[8:40, 8:40, 0]
    hp = lambda a: np.abs(a[:, 1:] - a[:, :-1]).mean()  # horizontal high-pass energy
    assert hp(imgs["ewa"]) < 0.5 * hp(imgs["bilinear"])


def _desc(ft):
    t = api.b2_texture_desc()
    t.width, t.height, t.channels, t.filter_type = ft["width"], ft["height"], ft["channels"], ft["filterType"]
    t.wrap_u, t.wrap_v = ft["wrapU"], ft["wrapV"]
    t.pixels = ft["pixels"].ctypes.data_as(C.POINTER(C.c_float))
    return t


@pytest.mark.parametrize("wrap", WRAPS)
def test_host_pyramid_equals_oracle_pyramid(wrap):
    """b2_mipmap_level (the builder b2_scene_commit uses; host code, no device) against the oracle's TMIPMap restatement: bit-exact."""
    L = api.lib()
    rng = np.random.default_rng(21)
    for shape in ((64, 64, 3), (37, 50, 3), (21, 13), (1, 9), (16, 1, 3)):
        img = (rng.random(shape) * 1.3 - 0.1).astype(np.float32)  # includes negatives (clamped) and values above 1
        tex = Texture(img, filter_type="ewa", wrap_u=wrap, wrap_v="clamp" if wrap == "repeat" else wrap)
        sc = O.OracleScene(one_texture_scene(tex))
        ft = tex.flat()
        t = _desc(ft)
        n, w, h = C.c_int(), C.c_int(), C.c_int()
        assert L.b2_mipmap_level(C.byref(t), 0, C.byref(n), C.byref(w), C.byref(h), None) == 0
        info = sc.texture_info(0)
        assert n.value == info["levels"]
        for l in range(n.value):
            assert L.b2_mipmap_level(C.byref(t), l, C.byref(n), C.byref(w), C.byref(h), None) == 0
            assert (w.value, h.value) == info["sizes"][l]
            out = np.zeros((h.value, w.value, ft["channels"]), np.float32)
            assert L.b2_mipmap_level(C.byref(t), l, C.byref(n), C.byref(w), C.byref(h), out.ctypes.data_as(C.POINTER(C.c_float))) == 0
            assert np.array_equal(out, sc.texture_level(0, l)), (shape, l)


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "resample_ref.npz")


def test_pyramids_match_the_reference_resampler():
    """tests/golden/resample_ref.npz: every MIP level of 30 seeded images as the REFERENCE's own Resampler<float> + LanczosSincFilter
    produce them (compiled from /root/reference into oracle/_ref/librfilterref.so; fixture written by tests/gen_golden.py).
    Both the oracle's restatement and the product's host-side builder must reproduce them bit for bit."""
    from gen_golden import half_store
    g = np.load(GOLDEN)
    L = api.lib()
    for k in range(int(g["count"])):
        img = g[f"img{k}"]
        wu, wv = (str(x) for x in g[f"wrap{k}"])
        tex = Texture(img if img.shape[2] == 3 else img[:, :, 0], filter_type="ewa", wrap_u=wu, wrap_v=wv)
        sc = O.OracleScene(one_texture_scene(tex))
        info = sc.texture_info(0)
        t = _desc(tex.flat())
        n, w, h = C.c_int(), C.c_int(), C.c_int()
        for l in range(1, info["levels"]):
            ref = half_store(g[f"lvl{k}_{l}"])   # resampled in float (the fixture), stored as half (bitmap.cpp:177-180, mipmap.h:262-264)
            assert np.array_equal(sc.texture_level(0, l), ref), (k, l, "oracle")
            out = np.zeros(ref.shape, np.float32)
            assert L.b2_mipmap_level(C.byref(t), l, C.byref(n), C.byref(w), C.byref(h), out.ctypes.data_as(C.POINTER(C.c_float))) == 0
            assert np.array_equal(out, ref), (k, l, "host builder")
        assert f"lvl{k}_{info['levels']}" not in g.files  # same number of levels


# the reference's outputs on inputs the fixtures above do not hold (tests/gen_golden.py, unseen_ref): the `*_when_present` tests below
# compare with these stored outputs and do not call the reference's libraries
UNSEEN = json.load(open(os.path.join(os.path.dirname(GOLDEN), "unseen_ref.json")))
UNSEEN_ARRAYS = np.load(os.path.join(os.path.dirname(GOLDEN), "unseen_ref.npz"))


def test_live_reference_resampler_when_present():
    """Same comparison on images the fixture does not hold: the levels the reference resampler (oracle/_ref/librfilterref.so) made of them,
    stored as half, in tests/golden/unseen_ref.npz."""
    from gen_golden import RESAMPLE_UNSEEN, half_store
    rng = np.random.default_rng(77)
    for i, (shape, wu, wv) in enumerate(RESAMPLE_UNSEEN):
        img = np.maximum((rng.random(shape) * 1.2 - 0.05).astype(np.float32), 0)
        tex = Texture(img if shape[2] == 3 else img[:, :, 0], filter_type="trilinear", wrap_u=wu, wrap_v=wv)
        sc = O.OracleScene(one_texture_scene(tex))
        levels = [UNSEEN_ARRAYS[f"resample{i}/{l}"] for l in range(1, sc.texture_info(0)["levels"])]
        assert f"resample{i}/{len(levels) + 1}" not in UNSEEN_ARRAYS.files  # same number of levels
        for l, ref in enumerate(levels):
            assert np.array_equal(sc.texture_level(0, l + 1), ref), (i, l + 1)
        assert np.array_equal(sc.texture_level(0, 0), half_store(img if shape[2] == 3 else img[:, :, :1]).reshape(sc.texture_level(0, 0).shape))


def golden_lookup_cases():
    g = np.load(os.path.join(os.path.dirname(GOLDEN), "mipmap_ref.npz"))
    for k in range(int(g["count"])):
        ft, wu, wv, aniso, j = (str(x) for x in g[f"cfg{k}"])
        tex = Texture(g[f"img{j}"], filter_type=ft, wrap_u=wu, wrap_v=wv, max_anisotropy=float(aniso))
        yield k, tex, g[f"uv{k}"], g[f"pt{k}"], g[f"filtered{k}"], g[f"unfiltered{k}"]


def test_lookups_match_the_reference_mipmap():
    """tests/golden/mipmap_ref.npz: look-ups of the REFERENCE's own TMIPMap<Color3, Color3> (mipmap.h compiled from /root/reference into
    oracle/_ref/libmipmapref.so, over pyramids from the reference resampler; fixture written by tests/gen_golden.py) for every filter
    type, four wrap-mode pairs and three anisotropy limits.  The oracle reproduces them bit for bit."""
    n = 0
    for k, tex, uv, pt, filtered, unfiltered in golden_lookup_cases():
        sc = O.OracleScene(one_texture_scene(tex))
        assert np.array_equal(sc.texture_eval(0, uv, pt), filtered), (k, tex.filter_type)
        assert np.array_equal(sc.texture_eval(0, uv), unfiltered), (k, tex.filter_type)
        n += 1
    assert n == 16


def test_live_reference_mipmap_when_present():
    """Look-ups on a checkerboard the fixture does not hold, against the digests of what the reference's TMIPMap (oracle/_ref/libmipmapref.so)
    returns over the reference resampler's pyramid (tests/golden/unseen_ref.json)."""
    from gen_golden import MIPMAP_UNSEEN, texture_lookups
    from ref_pins import digest
    rng = np.random.default_rng(99)
    img = checker_image(70, 45, 6, 1)
    for i, (ft, wu, wv, aniso) in enumerate(MIPMAP_UNSEEN):
        tex = Texture(img, filter_type=ft, wrap_u=wu, wrap_v=wv, max_anisotropy=aniso)
        sc = O.OracleScene(one_texture_scene(tex))
        uv, pt = texture_lookups(rng, 20000)
        assert digest(sc.texture_eval(0, uv, pt)) == UNSEEN[f"mipmap{i}/filtered"]
        assert digest(sc.texture_eval(0, uv)) == UNSEEN[f"mipmap{i}/unfiltered"]


def test_half_storage_rounding_matches_the_reference_half_class():
    """tests/golden/half_ref.npz: float -> half -> float through the reference's own half class (include/mitsuba/core/half.h +
    src/libcore/half.cpp compiled into oracle/_ref/libcoreref.so) on random bit patterns, ties, denormals and the overflow edge.  The
    oracle's roundToHalf (orc_texture.h) and numpy's float16 conversion (gen_golden.half_store, used to build the expected pyramids)
    reproduce it bit for bit; the product's host builder is held to the oracle's pyramids above."""
    from gen_golden import half_inputs, half_store
    g = np.load(os.path.join(os.path.dirname(GOLDEN), "half_ref.npz"))
    x, y = g["x"], g["y"]
    assert len(x) > 50000 and np.array_equal(x, half_inputs())
    out = np.zeros_like(x)
    O.lib().orc_half_round(C.c_uint64(len(x)), x.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data_as(C.POINTER(C.c_float)))
    assert np.array_equal(out.view(np.uint32), y.view(np.uint32))
    assert np.array_equal(half_store(x).view(np.uint32), y.view(np.uint32))
    # three million fresh values: oracle and numpy agree on all of them, and with the reference (digest of the bits in tests/golden/unseen_ref.json)
    from gen_golden import HALF_UNSEEN
    from ref_pins import digest
    x = half_inputs(**HALF_UNSEEN)
    out = np.zeros_like(x)
    O.lib().orc_half_round(C.c_uint64(len(x)), x.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data_as(C.POINTER(C.c_float)))
    assert np.array_equal(half_store(x).view(np.uint32), out.view(np.uint32)) and digest(out.view(np.uint32)) == UNSEEN["half"]


def test_stored_texels_are_half_representable_and_the_maximum_is_not():
    """Only the stored texels are rounded: minimum / maximum / average come from the float image (barray.h:103-126), so the energy
    conservation scale of bsdf.cpp:88-111 uses the unrounded maximum."""
    from gen_golden import half_store
    rng = np.random.default_rng(5)
    img = (rng.random((21, 30, 3)) * 1.7).astype(np.float32)
    sc = O.OracleScene(one_texture_scene(Texture(img, filter_type="ewa")))
    info = sc.texture_info(0)
    for l in range(info["levels"]):
        lvl = sc.texture_level(0, l)
        assert np.array_equal(lvl, half_store(lvl))
    assert np.array_equal(sc.texture_level(0, 0), half_store(img))
    uv = np.array([[(10 + 0.5) / 30, (7 + 0.5) / 21]], np.float32)           # a texel centre: bilinear weight 1 on that texel
    scale = np.float32(0.99) * (np.float32(1) / img.max())
    got = sc.texture_eval(0, uv)[0]
    assert np.allclose(got, half_store(img[7, 10]) * scale, rtol=2e-6) or np.allclose(got, half_store(img[7, 10]), rtol=2e-6)


def test_constant_texture_on_plastic_renders_like_the_constant_and_sets_the_sampling_weight():
    """plastic.diffuseReflectance bound to a bitmap (plastic.cpp:158-159,199-202,271,304,415): a one-colour image must render like the constant
    (texels are stored as half), and the specular sampling weight is derived from the texture's average the way the constructor does."""
    from gen_golden import half_store
    col = np.array([0.6, 0.4, 0.3], np.float32)
    img = np.full((8, 8, 3), 1.0, np.float32) * col
    rp = RenderParams(spp=8, sampler="sobol", rfilter="box")
    d1 = one_texture_scene(None)
    d1.meshes[0].bsdf = Bsdf("plastic", diffuse_reflectance=Texture(img, filter_type="ewa"))
    d2 = one_texture_scene(None)
    d2.meshes[0].bsdf = Bsdf("plastic", diffuse_reflectance=tuple(float(v) for v in half_store(col)))
    w1, w2 = d1.meshes[0].bsdf.flat()["specSamplingWeight"], d2.meshes[0].bsdf.flat()["specSamplingWeight"]
    assert abs(w1 - w2) < 2e-4 and 0.6 < w1 < 0.75            # 1 / (1 + lum(0.6, 0.4, 0.3)); the texture's average is of the unrounded floats
    d2.meshes[0].bsdf.flat = lambda f=d2.meshes[0].bsdf.flat: dict(f(), specSamplingWeight=w1)   # same weight: same lobe choices
    f1, s1 = O.OracleScene(d1).render(rp)
    f2, s2 = O.OracleScene(d2).render(rp)
    assert s1["rays"] == s2["rays"]
    assert np.abs(O.develop(f1) - O.develop(f2)).max() < 1e-5
    # an image above 1 is scaled for energy conservation (bsdf.cpp:88-111), and so is the average the weight is computed from
    t = Texture((img * np.float32(2.0)).astype(np.float32))
    assert abs(t.average_luminance() - 0.99 / 1.2 * (0.6 * 2 * 0.212671 + 0.4 * 2 * 0.715160 + 0.3 * 2 * 0.072169)) < 1e-5


@pytest.mark.parametrize("plugin", ["roughconductor", "conductor"])
def test_constant_texture_on_specular_reflectance_renders_like_the_constant(plugin):
    """specularReflectance of roughconductor / conductor bound to a bitmap (roughconductor.cpp:285,369,415; conductor.cpp:221-256)."""
    from gen_golden import half_store
    col = np.array([0.9, 0.6, 0.3], np.float32)
    img = np.full((4, 4, 3), 1.0, np.float32) * col
    rp = RenderParams(spp=8, sampler="sobol", rfilter="box")
    kw = dict(eta=(0.2004, 0.9240, 1.1022), k=(3.9129, 2.4528, 2.1421))
    if plugin == "roughconductor":
        kw.update(distribution="ggx", alpha_u=0.3, alpha_v=0.3)
    d1, d2 = one_texture_scene(None), one_texture_scene(None)
    d1.meshes[0].bsdf = Bsdf(plugin, specular_reflectance=Texture(img), **kw)
    d2.meshes[0].bsdf = Bsdf(plugin, specular_reflectance=tuple(float(v) for v in half_store(col)), **kw)
    f1, s1 = O.OracleScene(d1).render(rp)
    f2, s2 = O.OracleScene(d2).render(rp)
    assert s1["rays"] == s2["rays"]
    assert np.abs(O.develop(f1) - O.develop(f2)).max() < 1e-5 and O.develop(f1).max() > 1e-3
