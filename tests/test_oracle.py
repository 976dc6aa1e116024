"""The CPU oracle (oracle/pb2_oracle.cpp) against (a) golden vectors recorded from the unmodified reference
(tests/make_golden.py), (b) the reference's own known-answer tests for this path (src/tests/shapes.cpp,
src/tests/sampling.cpp), and (c) digests of further reference results (tests/golden/reference_digests.json).
Everything here runs on the CPU; bit-exact unless said otherwise.
"""
import json
import os

import numpy as np
import pytest

import golden_cases as gc
from conftest import GOLDEN, SCENES

SCENE_CASES = ["soup", "killeroo_like", "materials", "instances", "specular", "substrate", "metal", "uber", "roughglass", "lights", "params"]


def reference_digests():
    with open(os.path.join(GOLDEN, "reference_digests.json")) as f:
        return json.load(f)


def load_scene(pb, name):
    if name == "soup":
        return gc.soup_scene(pb)
    return pb.HostScene.from_file(os.path.join(SCENES, name + ".pbrt"))


def same_bvh(a, b):
    """LinearBVHNode arrays are equal where the reference defines them: `axis` of a leaf and the pad byte are
    uninitialised memory in the reference (bvh.cpp:640-658 never writes them)."""
    if len(a) != len(b):
        return False
    interior = a["n_prims"] == 0
    return (a["bmin"].tobytes() == b["bmin"].tobytes() and a["bmax"].tobytes() == b["bmax"].tobytes()
            and np.array_equal(a["offset"], b["offset"]) and np.array_equal(a["n_prims"], b["n_prims"])
            and np.array_equal(a["axis"][interior], b["axis"][interior]))


def recompute(pb, oracle, hs):
    """Everything tests/make_golden.py records, from `oracle`."""
    sc = oracle.scene(hs)
    nodes = hs.nodes()
    xres, yres = hs.film.contents.full_resolution[0], hs.film.contents.full_resolution[1]
    spp = hs.params.contents.samples_per_pixel
    pix, sn = gc.sample_ids(xres, yres, spp, 3000, 13)
    hpix, hsn, hdim = gc.sample_ids(xres, yres, spp, 4000, 14, max_dim=200)
    li, pfilm = sc.li_samples(pix, sn)
    img, _, st = sc.render(n_threads=2)
    return dict(hits=sc.intersect(gc.rays_for(pb, nodes, 1500, 11)), occluded=sc.intersect_p(gc.rays_for(pb, nodes, 1500, 12, shadow=True)),
                halton=oracle.halton(hs.film, hs.params, hpix, hsn, hdim), light_distribution=sc.light_distribution(gc.points_for(nodes, 400, 15)),
                li=li, pfilm=pfilm, image=img, rays=np.array([st.camera_rays, st.regular_rays, st.shadow_rays], np.int64), bvh=sc.bvh())


@pytest.mark.parametrize("name", SCENE_CASES)
def test_port_matches_reference_golden(pb, port, name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    hs = load_scene(pb, name)
    r = recompute(pb, port, hs)
    assert r["hits"].tobytes() == g["hits"].tobytes(), "Scene::Intersect: every field of every hit must be bit-identical"
    assert np.array_equal(r["occluded"], g["occluded"])
    assert np.array_equal(gc.bits(r["halton"]), gc.bits(g["halton"]))
    assert np.array_equal(gc.bits(r["light_distribution"]), gc.bits(g["light_distribution"]))
    assert np.array_equal(gc.bits(r["pfilm"]), gc.bits(g["pfilm"]))
    assert np.array_equal(gc.bits(r["li"]), gc.bits(g["li"])), "PathIntegrator::Li per sample must be bit-identical"
    assert np.array_equal(gc.bits(r["image"]), gc.bits(g["image"])), "whole image (after the XYZ round trip) must be bit-identical"
    assert np.array_equal(r["rays"], g["rays"]), "camera / regular / shadow ray counters"
    nodes, prims = r["bvh"]
    assert same_bvh(nodes, g["bvh_nodes"]) and np.array_equal(prims, g["bvh_prims"]), "BVHAccel linear nodes + primitive order"


@pytest.mark.parametrize("name", SCENE_CASES)
def test_port_matches_compiled_reference_live(pb, port, name):
    """Byte for byte what the compiled reference computed for the scene (recorded by tests/make_golden.py)."""
    a = np.load(os.path.join(GOLDEN, name + ".npz"))
    b = recompute(pb, port, load_scene(pb, name))
    for k in ("hits", "occluded", "halton", "light_distribution", "li", "pfilm", "image", "rays"):
        assert a[k].tobytes() == b[k].tobytes(), k


@pytest.mark.parametrize("case", sorted(gc.FILTER_CASES))
def test_port_filters_match_reference_golden(pb, port, case):
    """Reconstruction filters (src/filters/) through Film's 16x16 weight table (film.cpp:68-77, film.h:121-161)."""
    g = np.load(os.path.join(GOLDEN, "filters.npz"))
    hs = pb.HostScene.from_string(gc.filter_scene_text(SCENES, case))
    img, _, st = port.scene(hs).render(n_threads=1)   # one thread: overlapping tiles merge in a fixed order
    assert np.array_equal(gc.bits(img), gc.bits(g["image_" + case])), "image must be bit-identical to the reference's"
    assert [st.camera_rays, st.regular_rays, st.shadow_rays] == [int(x) for x in g["rays_" + case]]


@pytest.mark.parametrize("strategy", gc.LIGHT_STRATEGIES)
def test_port_delta_lights_other_strategies_live(pb, port, strategy):
    """The compiled reference's results for tests/scenes/lights.pbrt under another light-sampling strategy, as digests."""
    want = reference_digests()["lights_" + strategy]
    b = recompute(pb, port, pb.HostScene.from_string(gc.light_strategy_scene_text(SCENES, strategy)))
    for k in ("light_distribution", "li", "image"):
        assert gc.digest(b[k]) == want[k], k
    assert b["rays"].tolist() == want["rays"]


def test_port_filters_match_compiled_reference_live(pb, port):
    """Byte for byte the compiled reference's image for every filter case (recorded by tests/make_golden.py)."""
    g = np.load(os.path.join(GOLDEN, "filters.npz"))
    for case in sorted(gc.FILTER_CASES):
        hs = pb.HostScene.from_string(gc.filter_scene_text(SCENES, case))
        b, _, _ = port.scene(hs).render(n_threads=1)
        assert g["image_" + case].tobytes() == b.tobytes(), case


@pytest.mark.parametrize("case", sorted(gc.ANALYTIC_SCENES))
def test_reference_analytic_scenes(pb, port, case):
    """The reference's RenderTest.RadianceMatches for Path / perspective / Halton (analytic_scenes.cpp): radiance 1 +- 0.02."""
    hs = pb.HostScene.from_string(gc.analytic_scene_text(case))
    img, _, _ = port.scene(hs).render(n_threads=0)
    assert img.shape == (10, 10, 3)
    assert abs(float(img.mean()) - gc.ANALYTIC_EXPECTED) <= gc.ANALYTIC_DELTA, float(img.mean())


@pytest.mark.parametrize("name,maxprims", [("killeroo_like", 4), ("killeroo_like", 1), ("killeroo_like", 16), ("random20k", 4)])
def test_port_hlbvh_matches_reference_golden(pb, port, name, maxprims):
    """BVHAccel with splitmethod "hlbvh" (bvh.cpp:404-638): node array and primitive order of the compiled reference."""
    g = np.load(os.path.join(GOLDEN, "hlbvh.npz"))
    text = gc.random_mesh_scene_text(20000, 5) if name == "random20k" else open(os.path.join(SCENES, name + ".pbrt")).read()
    hs = pb.HostScene.from_string(gc.with_accelerator(text, "hlbvh", maxprims))
    nodes, prims = port.scene(hs, max_prims_in_node=maxprims, split_method=1).bvh()
    assert same_bvh(nodes, g["nodes_%s_%d" % (name, maxprims)]) and np.array_equal(prims, g["prims_%s_%d" % (name, maxprims)])


def test_low_discrepancy_golden(port):
    g = np.load(os.path.join(GOLDEN, "lowdiscrepancy.npz"))
    for b in (0, 1, 2, 3, 10, 50, 127, 500, 999):
        assert np.array_equal(gc.bits(port.radical_inverse(b, g["a"])), gc.bits(g["ri_%d" % b]))
        assert np.array_equal(gc.bits(port.radical_inverse(b, g["a"], scrambled=True)), gc.bits(g["sri_%d" % b]))


def test_radical_inverse_base2_is_bit_reversal(port):
    """src/tests/sampling.cpp:15-20 (LowDiscrepancy.RadicalInverse)."""
    a = np.arange(0, 1024, dtype=np.uint64)
    got = port.radical_inverse(0, a)

    def rev32(n):
        return int("{:032b}".format(n)[::-1], 2)
    want = np.array([rev32(int(x)) * 2.0 ** -32 for x in a], np.float32)
    assert np.array_equal(got, want)


def test_radical_inverse_against_naive_digits(port):
    """src/tests/sampling.cpp:22-74: compare with a straightforward double-precision digit reversal (1e-5)."""
    primes = [2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37, 41, 43, 47, 53]
    a = np.array([0, 1, 2, 1151, 32351, 4363211, 681122], np.uint64)
    for bi in range(1, 16):
        base = primes[bi]
        got = port.radical_inverse(bi, a)
        for x, v in zip(a, got):
            n, inv, val, scale = int(x), 1.0 / base, 0.0, 1.0 / base
            while n:
                val += (n % base) * scale
                n //= base
                scale *= inv
            assert abs(val - float(v)) < 1e-5


def test_triangle_bad_case_misses(pb, port):
    """src/tests/shapes.cpp:544-559 (Triangle.BadCases): this exact ray must miss this exact triangle."""
    text = """
Camera "perspective"
Film "image" "integer xresolution" [4] "integer yresolution" [4]
WorldBegin
Shape "trianglemesh" "integer indices" [0 1 2]
  "point P" [-1113.45459 -79.049614 -56.2431908  -1113.45459 -87.0922699 -56.2431908  -1113.45459 -79.2490845 -56.2431908]
WorldEnd
"""
    hs = pb.HostScene.from_string(text)
    rays = np.zeros(1, pb.RAY_DTYPE)
    rays["o"] = (-1081.47925, 99.9999542, 87.7701111)
    rays["d"] = (-32.1072998, -183.355865, -144.607635)
    rays["t_max"] = 0.9999
    sc = port.scene(hs)
    # the triangle is degenerate (collinear vertices): Triangle::Intersect rejects it at triangle.cpp:308-314.
    # IntersectP has no such check without an alpha mask (triangle.cpp:531), so only Intersect is pinned.
    assert sc.intersect(rays)["prim"][0] == -1


def tessellated_sphere_scene(pb, n_theta=16, n_phi=16, seed=12111):
    """The jittered unit-sphere mesh of src/tests/shapes.cpp:28-129 (Triangle.Watertight)."""
    rng = np.random.RandomState(seed)
    verts = []
    for t in range(n_theta):
        for p in range(n_phi):
            theta = np.pi * t / (n_theta - 1)
            phi = 2 * np.pi * p / n_phi
            v = np.array([np.sin(theta) * np.cos(phi), np.sin(theta) * np.sin(phi), np.cos(theta)])
            verts.append(v * (1 + 0.05 * rng.uniform(-1, 1)) if 0 < t < n_theta - 1 else v)
    idx = []
    for t in range(n_theta - 1):
        for p in range(n_phi):
            p1 = (p + 1) % n_phi
            a, b, c, d = t * n_phi + p, t * n_phi + p1, (t + 1) * n_phi + p, (t + 1) * n_phi + p1
            idx += [a, c, b, b, c, d]
    P = " ".join("%.9g" % x for v in verts for x in v)
    I = " ".join(str(i) for i in idx)
    text = 'Camera "perspective"\nFilm "image" "integer xresolution" [4] "integer yresolution" [4]\nWorldBegin\n' \
           'Shape "trianglemesh" "integer indices" [%s] "point P" [%s]\nWorldEnd\n' % (I, P)
    return pb.HostScene.from_string(text), np.array(verts, np.float32)


def test_triangle_mesh_is_watertight(pb, port):
    """src/tests/shapes.cpp:94-129: rays from inside a closed tessellated sphere always hit, also through vertices."""
    hs, verts = tessellated_sphere_scene(pb)
    sc = port.scene(hs)
    rng = np.random.RandomState(1)
    n = 20000
    rays = np.zeros(n, pb.RAY_DTYPE)
    rays["o"] = rng.uniform(-0.5, 0.5, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays["d"] = d.astype(np.float32)
    # half of the rays are aimed exactly at mesh vertices (the hard case of the reference test)
    tgt = verts[rng.randint(0, len(verts), n // 2)]
    rays["d"][: n // 2] = tgt - rays["o"][: n // 2]
    rays["t_max"] = np.inf
    assert (sc.intersect(rays)["prim"] >= 0).all()
    assert sc.intersect_p(rays).all()


def test_spawned_rays_do_not_reintersect(pb, port):
    """src/tests/shapes.cpp:154-205 (Triangle.Reintersect): rays leaving a hit point, offset by the hit's error
    bounds (OffsetRayOrigin), must not hit the same triangle again, for coordinates spanning many magnitudes."""
    rng = np.random.RandomState(7)
    for scale in (1e-3, 1.0, 1e4):
        tri = (rng.uniform(-1, 1, (3, 3)) * scale).astype(np.float32)
        text = 'Camera "perspective"\nFilm "image" "integer xresolution" [4] "integer yresolution" [4]\nWorldBegin\n' \
               'Shape "trianglemesh" "integer indices" [0 1 2] "point P" [%s]\nWorldEnd\n' % " ".join("%.9g" % x for x in tri.ravel())
        hs = pb.HostScene.from_string(text)
        sc = port.scene(hs)
        n = 2000
        b = rng.dirichlet([1, 1, 1], n).astype(np.float32)
        target = (b[:, :, None] * tri[None]).sum(axis=1)
        rays = np.zeros(n, pb.RAY_DTYPE)
        rays["o"] = (target + rng.normal(size=(n, 3)) * 3 * scale).astype(np.float32)
        rays["d"] = target - rays["o"]
        rays["t_max"] = np.inf
        h = sc.intersect(rays)
        ok = h["prim"] >= 0
        assert ok.mean() > 0.9
        # spawn in random directions from the reported hit point, origin offset exactly as Interaction::SpawnRay does
        w = rng.normal(size=(n, 3)).astype(np.float32)
        p, pe, nrm = h["p"], h["p_error"], h["n"]
        d = (np.abs(nrm) * pe).sum(axis=1, keepdims=True)
        off = d * nrm
        off[(w * nrm).sum(axis=1) < 0] *= -1
        po = (p + off).astype(np.float32)
        up = off > 0
        dn = off < 0
        po[up] = np.nextafter(po[up], np.float32(np.inf))
        po[dn] = np.nextafter(po[dn], np.float32(-np.inf))
        rays2 = np.zeros(n, pb.RAY_DTYPE)
        rays2["o"] = po
        rays2["d"] = w
        rays2["t_max"] = np.inf
        assert (sc.intersect(rays2[ok])["prim"] == -1).all()


@pytest.mark.parametrize("partial", [False, True])
def test_sphere_spawned_rays_do_not_reintersect(pb, port, partial):
    """FullSphere.Reintersect / PartialSphere.Reintersect / ParialSphere.Normal (src/tests/shapes.cpp:427-497)."""
    found = 0
    for i in range(40):
        text, rays, rng = gc.sphere_reintersect_case(pb, i, partial)
        hs = pb.HostScene.from_string(text)
        sc = port.scene(hs)
        h = sc.intersect(rays)
        h = h[h["prim"] >= 0]
        found += len(h)
        if len(h) == 0:
            continue
        # the normal is radial (ParialSphere.Normal)
        pn = h["p"] / np.linalg.norm(h["p"], axis=1, keepdims=True)
        nn = h["n"] / np.linalg.norm(h["n"], axis=1, keepdims=True)
        assert np.allclose((pn * nn).sum(axis=1), 1, atol=1e-5)
        out = gc.spawned_rays(pb, h, rng)
        assert (sc.intersect(out)["prim"] == -1).all() and not sc.intersect_p(out).any()
    assert found > 1000


def test_empty_and_degenerate_inputs(pb, port):
    hs = gc.soup_scene(pb)
    sc = port.scene(hs)
    assert len(sc.intersect(np.zeros(0, pb.RAY_DTYPE))) == 0
    rays = np.zeros(3, pb.RAY_DTYPE)
    rays["o"] = (0, 0, 50)
    rays["d"] = [(0, 0, -1), (0, 0, 1), (0, 0, -1)]
    rays["t_max"] = [np.inf, np.inf, 0.0]
    h = sc.intersect(rays)
    assert h["prim"][0] >= 0 and h["prim"][1] == -1 and h["prim"][2] == -1


def test_killeroo_simple_fingerprint_of_the_surveyed_reference(pb, port, tmp_path):
    """SURVEY.md section 9: `pbrt --outfile k8.pfm scenes/killeroo-simple.pbrt` of the reference binary gives md5
    5424ce0f17db0c040e0f988ebcfe4b4d with 16 870 506 regular + 6 157 124 shadow ray tests.  The same file (stored in
    tests/golden/killeroo/) parsed by THIS repo's host front end (parser, loop subdivision, transforms, SAH BVH builder),
    rendered by the port and written by our PFM writer must give those bytes: one test pins the port, the parser, the
    subdivision and the builder to the surveyed binary."""
    import hashlib
    from bench import stage_killeroo
    hs = pb.HostScene.from_file(stage_killeroo(str(tmp_path)))
    d = hs.desc.contents
    assert d.n_prims == 66533 and d.n_nodes == 59188 + 59189
    img, _, st = port.scene(hs).render(n_threads=0)
    assert img.shape == (700, 700, 3)
    assert (int(st.camera_rays), int(st.regular_rays), int(st.shadow_rays)) == (3920000, 16870506, 6157124)
    out = str(tmp_path / "k8.pfm")
    img = np.ascontiguousarray(img, np.float32)
    assert pb.lib().pb2h_write_pfm(out.encode(), pb.ptr(img), 700, 700) == 0
    assert hashlib.md5(open(out, "rb").read()).hexdigest() == "5424ce0f17db0c040e0f988ebcfe4b4d"


def test_library_texture_pyramids_are_the_reference_mipmaps(pb):
    """The MIP pyramid the library builds on the host (Lanczos resampling of the 37x23 / 20x12 / 24x10 images to a power of
    two, the clamp, the box-filtered levels under each wrap mode) against MIPMap::pyramid recorded from the compiled
    reference: every texel of every level BIT FOR BIT, for every texture of tests/scenes/textured.pbrt."""
    g = np.load(os.path.join(GOLDEN, "textures.npz"))
    hs = load_scene(pb, "textured")
    textures = hs.textures()
    assert len(textures) == 10
    resampled = 0
    for i, t in enumerate(textures):
        levels = pb.texture_pyramid(t)
        assert np.array_equal(np.array([[lv.shape[1], lv.shape[0]] for lv in levels], np.int32), g["levels_%d" % i])
        assert np.array_equal(gc.bits(np.concatenate([lv.ravel() for lv in levels])), gc.bits(g["pyramid_%d" % i])), i
        resampled += (levels[0].shape[1], levels[0].shape[0]) != (t.width, t.height)
        assert levels[-1].shape[:2] == (1, 1)
    assert resampled >= 4


def test_library_texture_pyramids_match_reference_live(pb):
    """... and against the reference on random images of awkward sizes (1 x N, N x 1, primes, already a power of two): shape
    and digest of every level of the reference's pyramid."""
    want = reference_digests()["pyramids"]
    for case, t, _texels in gc.pyramid_textures(pb):
        got = [[list(lv.shape), gc.digest(lv)] for lv in pb.texture_pyramid(t)]
        assert got == want[case], case


def test_sobol_sampler_matches_reference_golden(pb):
    """SobolSampler::SampleDimension(GetIndexForSample(k), dim) - index from pixel and sample number (SobolIntervalToIndex), the
    two pixel dimensions remapped into the pixel, 198 more dimensions - computed on the host by the functions the kernels
    compile, from generator matrices that tools/make_sobol_tables.py derives from the Joe-Kuo direction numbers: BIT FOR BIT
    the values recorded from the compiled reference (tests/golden/sobol.npz)."""
    g = np.load(os.path.join(GOLDEN, "sobol.npz"))
    hs = load_scene(pb, "sobol")
    assert hs.params.contents.sampler == pb.PB2_SAMPLER_SOBOL and hs.params.contents.samples_per_pixel == 8
    hpix, hsn, hdim = gc.sample_ids(80, 50, 8, 4000, 14, max_dim=200)
    got = pb.sobol_samples_host(hs.film, hs.params, hpix, hsn, hdim)
    assert np.array_equal(gc.bits(got), gc.bits(g["halton"]))
    assert (hdim < 2).sum() > 10 and (got[hdim < 2] < 1).all()


def test_sobol_tables_are_the_reference_tables(pb):
    """The generator matrices (from scipy's copy of the Joe-Kuo direction numbers) equal the reference's SobolMatrices32, and
    the two SobolIntervalToIndex tables the library derives from dimensions 0 and 1 by inverting a matrix over GF(2) equal
    VdCSobolMatrices / VdCSobolMatricesInv for every resolution from 2 to 2^25 pixels (digests of the reference's tables)."""
    import ctypes as C
    want = reference_digests()
    mats = np.fromfile(os.path.join(os.path.dirname(pb.__file__), "lib", "sobol_matrices32.bin"), "<u4").reshape(1024, 52)
    assert gc.digest(mats) == want["sobol_matrices32"]
    film = pb.FilmDesc()
    film.filter_radius[0] = film.filter_radius[1] = 0.5
    pp = pb.PathParams(samples_per_pixel=1, sampler=pb.PB2_SAMPLER_SOBOL)
    for m in range(1, 26):
        res = 1 << m
        film.full_resolution[0], film.full_resolution[1] = res, 1
        film.cropped_pixel_bounds[0], film.cropped_pixel_bounds[1], film.cropped_pixel_bounds[2], film.cropped_pixel_bounds[3] = 0, 0, res, 1
        _, tab = pb.sobol_samples_host(C.byref(film), C.byref(pp), np.zeros((1, 2), np.int32), np.zeros(1, np.int64), np.zeros(1, np.int32), tables=True)
        assert gc.digest(tab) == want["vdc_sobol"][str(m)], m


def test_environment_map_distribution_is_the_reference_distribution(pb):
    """An InfiniteAreaLight's sampling distribution over its environment map - the map's pyramid (40 x 20 resampled to 64 x 32),
    128 x 64 trilinear look-ups, luminance, sin(theta), one Distribution1D per row and the marginal - computed by the library
    on the host: BIT FOR BIT InfiniteAreaLight::distribution recorded from the compiled reference."""
    g = np.load(os.path.join(GOLDEN, "env_distribution.npz"))
    hs = load_scene(pb, "envmap")
    d = hs.desc.contents
    env = [d.delta_lights[i].env_tex for i in range(d.n_lights) if d.lights[i].type == pb.PB2_LIGHT_INFINITE]
    assert len(env) == 1 and env[0] >= 1
    nu, nv, table = pb.env_distribution(d.textures[env[0] - 1])
    assert (nu, nv) == (int(g["nu"]), int(g["nv"])) == (128, 64)
    assert np.array_equal(gc.bits(table), gc.bits(g["table"]))


@pytest.mark.parametrize("scene", gc.TEXTURE_EVAL_SCENES)
def test_texture_nodes_evaluate_like_the_reference_textures(pb, scene):
    """Texture::Evaluate(si) for every texture of the textured golden scenes - image maps (EWA and trilinear) behind their uv
    mappings with the point's differentials, constants, scale, mix (nested), checkerboards (point-sampled and box-filtered in
    closed form) and uv textures - computed on the host by the functions the kernels compile: BIT FOR BIT what the reference's
    own texture objects return (tests/golden/texture_evaluations.npz)."""
    g = np.load(os.path.join(GOLDEN, "texture_evaluations.npz"))
    hs = load_scene(pb, scene)
    d = hs.desc.contents
    uv, duv = gc.texture_eval_inputs(2000, 7)
    kinds = set()
    for t in range(d.n_textures):
        got = pb.texture_eval_host(d.textures, d.n_textures, t, uv, duv)
        want = g["%s_%d" % (scene, t)]
        assert np.array_equal(gc.bits(got), gc.bits(want)) or np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(gc.bits(got[~np.isnan(got)]), gc.bits(want[~np.isnan(want)])), (scene, t)
        kinds.add(d.textures[t].kind)
    if scene == "checker":
        assert {pb.PB2_TEXKIND_CHECKERBOARD, pb.PB2_TEXKIND_UV, pb.PB2_TEXKIND_MIX, pb.PB2_TEXKIND_IMAGE, pb.PB2_TEXKIND_CONSTANT} <= kinds


@pytest.mark.parametrize("scene", gc.DIFFERENTIAL_SCENES)
def test_ray_differentials_match_the_reference(pb, scene):
    """The footprint of a pixel on a surface: the camera ray's offset rays (perspective.cpp:117-144 - pinhole and thin lens -
    taken to world space and scaled by 1 / sqrt(spp)) and SurfaceInteraction::ComputeDifferentials (interaction.cpp:101-147) at
    the first hit (triangles, spheres, instanced objects), computed on the host by the two functions the shade kernel compiles:
    BIT FOR BIT the reference's values (tests/golden/differentials.npz: 3000 camera samples per scene)."""
    rec = np.load(os.path.join(GOLDEN, "differentials.npz"))[scene]
    hs = load_scene(pb, scene)
    L = pb.lib()
    inp = np.ascontiguousarray(rec[:, 0:10])          # pFilm, pLens, o, d
    out = np.zeros((len(rec), 12), np.float32)
    assert L.pb2_camera_differentials_host(hs.camera, hs.film, hs.params, len(rec), pb.ptr(inp), pb.ptr(out)) == 0
    assert np.array_equal(gc.bits(out), gc.bits(np.ascontiguousarray(rec[:, 10:22])))
    hit = rec[:, 22] > 0
    assert hit.sum() > 2000
    inp2 = np.ascontiguousarray(np.concatenate([rec[hit, 23:35], rec[hit, 10:22]], 1))   # p, n, dpdu, dpdv; the offset rays
    duv = np.zeros((int(hit.sum()), 4), np.float32)
    assert L.pb2_uv_differentials_host(int(hit.sum()), pb.ptr(inp2), pb.ptr(duv)) == 0
    want = np.ascontiguousarray(rec[hit, 35:39])
    assert np.array_equal(gc.bits(duv), gc.bits(want)) and (np.abs(want) > 0).mean() > 0.9
    if scene == "textured_lens":
        assert hs.camera.contents.lens_radius > 0 and not np.array_equal(rec[:, 4:7], rec[:, 10:13])   # the offset rays start on the lens


@pytest.mark.parametrize("scene", gc.BSDF_SCENES)
def test_shade_kernel_bsdf_functions_match_the_reference_bsdf(pb, scene):
    """The functions the shade kernel compiles - makeBsdf (matte with and without sigma, plastic, substrate, metal, uber with
    opacity / Kr / Kt, mirror, smooth and rough glass), bsdfF, bsdfPdf, bsdfSampleF - evaluated on the host for every material
    record of a scene at 1500 random shading frames: f and Pdf over the non-specular lobes, the non-specular Sample_f of
    EstimateDirect and the all-lobes Sample_f of the path's continuation (direction, value, pdf, sampled flags) are BIT FOR BIT
    what the reference's Material::ComputeScatteringFunctions + BSDF return (tests/golden/bsdf.npz)."""
    g = np.load(os.path.join(GOLDEN, "bsdf.npz"))
    hs = load_scene(pb, scene)
    d = hs.desc.contents
    types = set()
    for m in range(d.n_materials):
        got = pb.bsdf_eval_host(d.materials[m], gc.bsdf_frames(1500, 17 + m))
        want = g["%s_%d" % (scene, m)]
        same = gc.bits(got) == gc.bits(want)
        same[:, 18] |= want[:, 17] == 0          # the sampled flags mean something only when a direction was sampled
        assert same.all(), (scene, m, d.materials[m].type, np.where(~same.all(0))[0])
        assert (want[:, 17] != 0).mean() > 0.3   # (half of the frames see the surface from below the shading hemisphere or so)
        types.add(d.materials[m].type)
    assert pb.PB2_MAT_MATTE in types
