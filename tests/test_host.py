"""Host-side C++ front end (parser, pbrt API state machine, transforms, loop subdivision, SAH BVH build, film)
against golden vectors recorded from the reference and against the oracle port.  CPU only."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_cases as gc
from conftest import GOLDEN, SCENES
from test_oracle import same_bvh


def test_host_bvh_equals_reference_bvh(pb):
    """The host SAH builder reproduces BVHAccel's LinearBVHNode array and primitive order (src/accelerators/bvh.cpp:183-402)."""
    for name in ("soup", "killeroo_like", "materials", "instances", "specular", "substrate"):
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        hs = gc.soup_scene(pb) if name == "soup" else pb.HostScene.from_file(os.path.join(SCENES, name + ".pbrt"))
        assert same_bvh(hs.nodes(), g["bvh_nodes"]), name
        assert np.array_equal(hs.bvh_prims(), g["bvh_prims"]), name


def test_host_bvh_equals_port_bvh_other_split_methods(pb, port):
    for split, code in (("middle", 2), ("equal", 3), ("sah", 0)):
        text = open(os.path.join(SCENES, "killeroo_like.pbrt")).read().replace("WorldBegin", 'Accelerator "bvh" "string splitmethod" "%s" "integer maxnodeprims" [2]\nWorldBegin' % split)
        hs = pb.HostScene.from_string(text)
        nodes, prims = port.scene(hs, max_prims_in_node=2, split_method=code).bvh()
        assert same_bvh(hs.nodes(), nodes) and np.array_equal(hs.bvh_prims(), prims), split


def test_loop_subdivision_matches_reference(pb):
    g = np.load(os.path.join(GOLDEN, "loopsubdiv.npz"))
    for tag in ("closed", "open"):
        for lv in (1, 2, 3):
            P, N, I = pb.loop_subdivide(lv, g[tag + "_I"], g[tag + "_P"])
            assert np.array_equal(gc.bits(P), gc.bits(g["%s_%d_P" % (tag, lv)]))
            assert np.array_equal(gc.bits(N), gc.bits(g["%s_%d_N" % (tag, lv)]))
            assert np.array_equal(I, g["%s_%d_I" % (tag, lv)])


def test_camera_matrices_match_reference(pb):
    g = np.load(os.path.join(GOLDEN, "camera.npz"))
    hs = gc.soup_scene(pb, xres=1920, yres=1080)
    cam = hs.camera.contents
    assert np.array_equal(gc.bits(np.ctypeslib.as_array(cam.raster_to_camera)), gc.bits(g["raster_to_camera"]))
    assert np.array_equal(gc.bits(np.ctypeslib.as_array(cam.dx_camera)), gc.bits(g["dx"]))
    assert np.array_equal(gc.bits(np.ctypeslib.as_array(cam.dy_camera)), gc.bits(g["dy"]))


def scene_with_transform(pb, directive):
    text = 'Camera "perspective"\nFilm "image" "integer xresolution" [4] "integer yresolution" [4]\nWorldBegin\n%s\n' \
           'Shape "sphere" "float radius" [1]\nWorldEnd\n' % directive
    hs = pb.HostScene.from_string(text)
    s = hs.desc.contents.spheres[0]
    return np.ctypeslib.as_array(s.object_to_world).copy(), np.ctypeslib.as_array(s.world_to_object).copy()


def test_transform_directives_match_reference(pb):
    """LookAt / Rotate / Translate / Scale produce the reference's matrix bits (src/core/transform.cpp)."""
    g = np.load(os.path.join(GOLDEN, "transforms.npz"))
    names = {0: "LookAt", 1: "Rotate", 3: "Translate", 4: "Scale"}
    for i in range(int(g["n"])):
        kind = int(g["kind_%d" % i])
        if kind not in names:
            continue
        directive = names[kind] + " " + " ".join("%.9g" % x for x in g["args_%d" % i])
        m, mi = scene_with_transform(pb, directive)
        # the directive multiplies the CTM (identity here) by the transform, api.cpp:903-964, which turns a -0
        # entry into +0 in the reference as well; the golden holds the bare transform, so zeros compare unsigned
        unsigned_zero = lambda a: np.where(a == 0, np.float32(0), a).astype(np.float32)  # noqa: E731
        assert np.array_equal(gc.bits(unsigned_zero(m)), gc.bits(unsigned_zero(g["m_%d" % i]))), directive
        assert np.array_equal(gc.bits(unsigned_zero(mi)), gc.bits(unsigned_zero(g["minv_%d" % i]))), directive


def test_tokenizer_and_parameter_lists(pb):
    """Comments, quoted strings, bracketed and bare single values, legacy type names (src/core/parser.cpp:98-320, 413-485)."""
    text = '''
# a comment line
Camera "perspective" "float fov" 45   # bare single value
Film "image" "integer xresolution" [ 8 ] "integer yresolution" [8] "string filename" ["x.pfm"]
Sampler "halton" "integer pixelsamples" 2
WorldBegin   Material "matte" "color Kd" [.1 .2 .3] "float sigma" 0
AttributeBegin AreaLightSource "diffuse" "rgb L" [1 2 3] "bool twosided" "true"
Shape "trianglemesh" "point3 P" [0 0 0 1 0 0 0 1 0] "integer indices" [0 1 2] "point2 uv" [0 0 1 0 0 1] AttributeEnd
Shape "trianglemesh" "point P" [0 0 1 1 0 1 0 1 1 1 1 1] "integer indices" [0 1 2 1 3 2] "normal N" [0 0 1 0 0 1 0 0 1 0 0 1]
WorldEnd
'''
    hs = pb.HostScene.from_string(text)
    d = hs.desc.contents
    assert d.n_prims == 3 and d.n_meshes == 2 and d.n_lights == 1 and d.n_materials == 1
    assert d.meshes[0].has_uv == 1 and d.meshes[0].has_n == 0 and d.meshes[1].has_n == 1
    assert d.lights[0].two_sided == 1 and tuple(d.lights[0].L) == (1.0, 2.0, 3.0) and abs(d.lights[0].area - 0.5) < 1e-7
    m = d.materials[0]
    assert m.type == 1 and np.allclose(tuple(m.kd), (0.1, 0.2, 0.3))
    assert hs.params.contents.samples_per_pixel == 2 and hs.camera.contents.fov == 45.0
    assert tuple(hs.film.contents.full_resolution) == (8, 8)
    assert d.light_strategy == pb.PB2_LIGHTDIST_UNIFORM  # a single light always gets the uniform distribution


def test_defaults_when_scene_file_is_silent(pb):
    """src/core/api.cpp:166-177 and the Create* defaults: 1280x720, halton 16 spp, path maxdepth 5, fov 90, matte Kd .5."""
    hs = pb.HostScene.from_string('WorldBegin\nShape "sphere"\nWorldEnd\n')
    assert tuple(hs.film.contents.full_resolution) == (1280, 720)
    p = hs.params.contents
    assert p.samples_per_pixel == 16 and p.max_depth == 5 and p.rr_threshold == 1.0
    assert hs.camera.contents.fov == 90.0
    assert tuple(hs.film.contents.filter_radius) == (0.5, 0.5)
    m = hs.desc.contents.materials[0]
    assert m.type == 1 and tuple(m.kd) == (0.5, 0.5, 0.5)


def test_unsupported_plugins_are_reported_not_silently_replaced(pb):
    before = pb.lib().pb2h_error_count()
    pb.HostScene.from_string('Sampler "halton"\nWorldBegin\nMaterial "translucent"\nShape "sphere"\nWorldEnd\n')
    assert pb.lib().pb2h_error_count() > before


def test_film_resolve_is_the_xyz_round_trip(pb):
    """Film::MergeFilmTile (RGB->XYZ) + WriteImage (XYZ->RGB, /weight, clamp) on a known rgbw buffer (film.cpp:117-211)."""
    hs = pb.HostScene.soup(10, xres=8, yres=4, spp=1)
    rng = np.random.RandomState(2)
    rgbw = rng.rand(4, 8, 4).astype(np.float32)
    rgbw[..., 3] = rng.randint(1, 5, (4, 8))
    rgbw[0, 0] = 0
    out = hs.resolve(rgbw)
    f32 = np.float32
    rgb = rgbw[..., :3]
    to_xyz = np.array([[0.412453, 0.357580, 0.180423], [0.212671, 0.715160, 0.072169], [0.019334, 0.119193, 0.950227]], f32)
    to_rgb = np.array([[3.240479, -1.537150, -0.498535], [-0.969256, 1.875991, 0.041556], [0.055648, -0.204043, 1.057311]], f32)

    def apply(mat, v):  # left-to-right float32 sums like the reference's inline functions
        return np.stack([(mat[i, 0] * v[..., 0] + mat[i, 1] * v[..., 1]) + mat[i, 2] * v[..., 2] for i in range(3)], -1).astype(f32)
    want = apply(to_rgb, apply(to_xyz, rgb))
    w = rgbw[..., 3:4]
    want = np.where(w != 0, np.maximum(0, want * (f32(1) / np.where(w != 0, w, 1))), want).astype(f32)
    assert np.allclose(out, want, rtol=0, atol=1e-6)
    assert (out[0, 0] == 0).all()


def test_object_instancing_directives(pb):
    """pbrtObjectBegin/End/Instance (src/core/api.cpp:1520-1588): an object with several primitives gets its own
    accelerator, a one-primitive object is instanced directly, every ObjectInstance becomes a TransformedPrimitive
    carrying the CTM, and the scene BVH is built over the scene-level primitives only."""
    hs = pb.HostScene.from_file(os.path.join(SCENES, "instances.pbrt"))
    d = hs.desc.contents
    assert d.n_instances == 5 and d.n_bvhs == 2
    prim_type = np.ctypeslib.as_array(d.prim_type, shape=(d.n_prims,))
    n_top = hs.bvh_range(0)[3]
    assert n_top == 9 and (prim_type[:n_top] == pb.PB2_PRIM_INSTANCE).sum() == 5 and (prim_type[n_top:] == pb.PB2_PRIM_INSTANCE).sum() == 0
    assert sorted(hs.bvh_prims(0)) == list(range(9))
    assert sorted(hs.bvh_prims(1)) == list(range(9, 16))            # the pyramid's 6 triangles + its sphere
    inst = [d.instances[i] for i in range(5)]
    assert [i.bvh for i in inst] == [1, 1, 1, -1, -1]
    assert inst[3].lone_prim == inst[4].lone_prim == d.n_bvh_prims - 1  # the flag's triangle, once, past every BVH range
    eye = np.eye(4, dtype=np.float32).ravel()
    assert np.array_equal(np.array(inst[0].instance_to_world), eye)    # ObjectInstance under the identity CTM
    m = np.array(inst[1].instance_to_world).reshape(4, 4)
    w = np.array(inst[1].world_to_instance).reshape(4, 4)
    assert np.allclose(m @ w, np.eye(4), atol=1e-6) and np.allclose(m[:3, 3], [-2, .5, 0])
    assert np.linalg.det(np.array(inst[2].instance_to_world).reshape(4, 4)[:3, :3]) < 0   # the mirrored instance
    # the errors the reference reports
    before = pb.lib().pb2h_error_count()
    pb.HostScene.from_string('WorldBegin\nShape "sphere"\nObjectInstance "nope"\nWorldEnd\n')
    assert pb.lib().pb2h_error_count() == before + 1
    pb.HostScene.from_string('WorldBegin\nShape "sphere"\nObjectBegin "a"\nObjectBegin "b"\nObjectEnd\nObjectEnd\nWorldEnd\n')
    assert pb.lib().pb2h_error_count() > before + 1


def test_mirror_and_glass_parameters(pb):
    """CreateMirrorMaterial / CreateGlassMaterial defaults and parameter names (mirror.cpp:60-66, glass.cpp:95-112)."""
    hs = pb.HostScene.from_file(os.path.join(SCENES, "specular.pbrt"))
    d = hs.desc.contents
    mats = [d.materials[i] for i in range(d.n_materials)]
    mirrors = [m for m in mats if m.type == pb.PB2_MAT_MIRROR]
    glasses = [m for m in mats if m.type == pb.PB2_MAT_GLASS]
    assert len(mirrors) == 2 and len(glasses) == 2
    assert np.allclose(tuple(mirrors[0].kr), (.9, .85, .8)) and np.allclose(tuple(mirrors[1].kr), (.9, .9, .9))   # default Kr 0.9
    assert glasses[0].eta == np.float32(1.5) and tuple(glasses[0].kr) == (1, 1, 1) and tuple(glasses[0].kt) == (1, 1, 1)
    assert glasses[1].eta == np.float32(1.33) and np.allclose(tuple(glasses[1].kt), (.8, .95, .85))
    assert all(g.uroughness == 0 and g.vroughness == 0 for g in glasses)
    hs = pb.HostScene.from_string('WorldBegin\nMaterial "glass" "float uroughness" 0.2\nShape "sphere"\nWorldEnd\n')
    d = hs.desc.contents
    rough = [d.materials[i] for i in range(d.n_materials) if d.materials[i].type == pb.PB2_MAT_GLASS][0]
    assert rough.uroughness == np.float32(.2) and rough.vroughness == 0 and rough.remap_roughness == 1


def test_threaded_bvh_build_is_the_sequential_tree(pb, port):
    """Above 65 536 primitives the host builder hands subtrees to other threads; every subtree owns a fixed range of
    the ordered-primitive list, so the LinearBVHNode array and the primitive order must still be the reference's
    (the port builds sequentially, in the reference's order)."""
    hs = pb.HostScene.soup(300000, seed=7, jitter=0.01, xres=16, yres=16, spp=1)
    nodes, prims = port.scene(hs).bvh()
    first_nodes, first_prims = hs.nodes(), hs.bvh_prims()
    assert same_bvh(first_nodes, nodes) and np.array_equal(first_prims, prims)
    again = pb.HostScene.soup(300000, seed=7, jitter=0.01, xres=16, yres=16, spp=1)   # replaces the parsed scene
    assert again.nodes().tobytes() == first_nodes.tobytes() and np.array_equal(again.bvh_prims(), first_prims)


def test_pixel_filter_directive_fills_the_film_description(pb):
    """MakeFilter (api.cpp:862-878) + Create*Filter defaults (src/filters/*.cpp) as recorded from the reference's Film."""
    g = np.load(os.path.join(GOLDEN, "filters.npz"))
    want_types = {"gaussian": pb.PB2_FILTER_GAUSSIAN, "mitchell": pb.PB2_FILTER_MITCHELL, "sinc": pb.PB2_FILTER_SINC,
                  "triangle": pb.PB2_FILTER_TRIANGLE, "box_wide": pb.PB2_FILTER_BOX}
    for case in gc.FILTER_CASES:
        hs = pb.HostScene.from_string(gc.filter_scene_text(SCENES, case))
        f = hs.film.contents
        got = np.array([f.filter_type, *f.filter_radius, *f.filter_param, *f.cropped_pixel_bounds], np.float64)
        assert np.array_equal(got, g["film_" + case]), case
        if case in want_types:
            assert f.filter_type == want_types[case]
    f = pb.HostScene.from_string(gc.filter_scene_text(SCENES, "sinc")).film.contents
    assert list(f.filter_radius) == [4, 4] and f.filter_param[0] == 3
    before = pb.lib().pb2h_error_count()
    f = pb.HostScene.from_string('PixelFilter "lanczos9"\nWorldBegin\nWorldEnd\n').film.contents
    assert pb.lib().pb2h_error_count() > before and f.filter_type == pb.PB2_FILTER_BOX


def test_uber_and_metal_parameters(pb):
    """CreateUberMaterial / CreateMetalMaterial (uber.cpp:106-131, metal.cpp:120-140): defaults, the "eta"-over-"index"
    rule, the roughness fall-backs of ComputeScatteringFunctions, and the copper defaults recorded from the reference."""
    f32 = np.float32
    hs = pb.HostScene.from_file(os.path.join(SCENES, "uber.pbrt"))
    d = hs.desc.contents
    ub = [d.materials[i] for i in range(d.n_materials) if d.materials[i].type == pb.PB2_MAT_UBER]
    assert len(ub) == 5
    dflt = ub[0]
    assert tuple(dflt.kd) == (.25,) * 3 and tuple(dflt.ks) == (.25,) * 3 and tuple(dflt.kr) == (0,) * 3 and tuple(dflt.kt) == (0,) * 3
    assert tuple(dflt.opacity) == (1,) * 3 and dflt.eta == f32(1.5) and dflt.uroughness == f32(.1) == dflt.vroughness and dflt.remap_roughness == 1
    assert ub[1].eta == f32(1.33) and ub[1].uroughness == f32(.05) == ub[1].vroughness and np.allclose(tuple(ub[1].opacity), (.8, .7, .6))
    assert ub[2].eta == f32(1.6)                                   # "eta" wins over "index"
    assert ub[3].uroughness == f32(.3) and ub[3].vroughness == f32(.04) and ub[3].remap_roughness == 0
    assert tuple(ub[4].opacity) == (0, 0, 0)
    hs = pb.HostScene.from_string('WorldBegin\nMaterial "uber" "float roughness" .3 "float uroughness" .02\nShape "sphere"\nWorldEnd\n')
    m = [hs.desc.contents.materials[i] for i in range(hs.desc.contents.n_materials) if hs.desc.contents.materials[i].type == pb.PB2_MAT_UBER][0]
    assert m.uroughness == f32(.02) == m.vroughness                # uber: "vroughness" falls back to the u value (uber.cpp:77-80)
    hs = pb.HostScene.from_file(os.path.join(SCENES, "metal.pbrt"))
    d = hs.desc.contents
    me = [d.materials[i] for i in range(d.n_materials) if d.materials[i].type == pb.PB2_MAT_METAL]
    assert len(me) == 3
    g = np.load(os.path.join(GOLDEN, "metal_defaults.npz"))
    assert np.array_equal(gc.bits(np.array(tuple(me[0].metal_eta), f32)), gc.bits(g["eta"]))
    assert np.array_equal(gc.bits(np.array(tuple(me[0].metal_k), f32)), gc.bits(g["k"]))
    assert me[0].uroughness == f32(.01) == me[0].vroughness and me[0].remap_roughness == 1
    assert me[1].uroughness == f32(.05) and me[1].vroughness == f32(.4)
    assert me[2].uroughness == f32(.15) == me[2].vroughness and me[2].remap_roughness == 0
    hs = pb.HostScene.from_string('WorldBegin\nMaterial "metal" "float roughness" .3 "float uroughness" .02\nShape "sphere"\nWorldEnd\n')
    m = [hs.desc.contents.materials[i] for i in range(hs.desc.contents.n_materials) if hs.desc.contents.materials[i].type == pb.PB2_MAT_METAL][0]
    assert m.uroughness == f32(.02) and m.vroughness == f32(.3)    # metal: each falls back to "roughness" (metal.cpp:67-70)


def test_light_source_directives(pb):
    """pbrtLightSource (api.cpp:1302-1316) + CreatePointLight / CreateSpotLight / CreateDistantLight (point.cpp:84-92,
    spot.cpp:103-125, distant.cpp:92-100): Scene::lights keeps file order with the area lights, "from" / "to" / "scale"
    and the CTM are applied as the reference does."""
    f32 = np.float32
    hs = pb.HostScene.from_file(os.path.join(SCENES, "lights.pbrt"))
    d = hs.desc.contents
    assert [d.lights[i].type for i in range(d.n_lights)] == [pb.PB2_LIGHT_POINT, pb.PB2_LIGHT_AREA, pb.PB2_LIGHT_AREA, pb.PB2_LIGHT_SPOT,
                                                            pb.PB2_LIGHT_DISTANT, pb.PB2_LIGHT_DISTANT]
    assert all(d.lights[i].prim == -1 for i in (0, 3, 4, 5)) and d.lights[1].prim >= 0
    assert tuple(d.delta_lights[0].p) == (f32(-2.2), f32(-1.5), f32(2.5)) and tuple(d.lights[0].L) == (9, 7, 5)
    spot = d.delta_lights[3]
    assert np.allclose(tuple(d.lights[3].L), (20, 24, 21)) and spot.total_width_deg == 28 and spot.falloff_start_deg == 19   # coneangle - conedeltaangle
    w2l = np.array(tuple(spot.world_to_light), np.float64).reshape(3, 3)
    assert np.allclose(w2l @ w2l.T, np.eye(3), atol=1e-6)          # rotations only on this light's CTM
    # the spot looks from "from" to "to" (both under the CTM): WorldToLight maps that direction to +z
    ang = np.radians(20)
    rot = np.array([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1]])
    frm, to = rot @ (np.array([0, -2.5, 3.2]) + [.3, 0, 0]), rot @ (np.array([.4, .2, 0]) + [.3, 0, 0])
    assert np.allclose(tuple(spot.p), frm, atol=1e-5)
    dirw = (to - frm) / np.linalg.norm(to - frm)
    assert np.allclose(w2l @ dirw, (0, 0, 1), atol=1e-5)
    assert tuple(d.delta_lights[4].p) == (1, -2, 4)                # from - to, not normalised
    assert np.allclose(tuple(d.delta_lights[5].p), (-.2, -.1, 2)) and np.allclose(tuple(d.lights[5].L), (.15, .2, .3))   # defaults: L 1, from 0; Scale 1 1 2
    nodes = hs.nodes()
    c = (nodes["bmin"][0].astype(f32) + nodes["bmax"][0].astype(f32)) / f32(2)
    assert abs(d.delta_lights[4].world_radius - np.linalg.norm(c - nodes["bmax"][0])) < 1e-5
    before = pb.lib().pb2h_error_count()
    hs = pb.HostScene.from_string('WorldBegin\nLightSource "goniometric"\nShape "sphere"\nWorldEnd\n')
    assert pb.lib().pb2h_error_count() > before and hs.desc.contents.n_lights == 0


@pytest.mark.parametrize("name,maxprims", [("killeroo_like", 4), ("killeroo_like", 1), ("killeroo_like", 16), ("random20k", 4)])
def test_hlbvh_build_equals_reference(pb, name, maxprims):
    """splitmethod "hlbvh": Morton codes, the stable 30-bit sort, treelets on the top 12 bits, emitLBVH and the SAH tree
    over the treelet roots (bvh.cpp:404-638) give the reference's node array byte for byte and its primitive order."""
    g = np.load(os.path.join(GOLDEN, "hlbvh.npz"))
    text = gc.random_mesh_scene_text(20000, 5) if name == "random20k" else open(os.path.join(SCENES, name + ".pbrt")).read()
    hs = pb.HostScene.from_string(gc.with_accelerator(text, "hlbvh", maxprims))
    assert same_bvh(hs.nodes(), g["nodes_%s_%d" % (name, maxprims)])
    assert np.array_equal(hs.bvh_prims(0), g["prims_%s_%d" % (name, maxprims)])


def _to_byte(rgb):
    f32 = np.float32
    v = rgb.astype(f32)
    g = np.where(v <= f32(0.0031308), f32(12.92) * v, f32(1.055) * np.power(np.maximum(v, 0), f32(1 / 2.4), dtype=f32) - f32(0.055)).astype(f32)
    return np.clip(f32(255) * g + f32(0.5), 0, 255).astype(np.uint8)


def test_image_writers_exr_png_tga(pb, tmp_path):
    """WriteImage (imageio.cpp:81-122): the container follows the extension.  EXR: half RGB, data window = the cropped
    pixels inside the display window; PNG / TGA: gamma-corrected bytes (TO_BYTE, imageio.cpp:100).  Decoded here by
    hand-written readers of the three containers."""
    import struct
    import zlib
    rng = np.random.RandomState(3)
    w, h = 7, 5
    rgb = (rng.rand(h, w, 3) ** 3 * 4).astype(np.float32)
    rgb[0, 0] = (0, 1e-9, 6.1e-5)          # zero, flush-to-zero, half denormal range
    rgb[0, 1] = (65504, 65520, 1e9)         # largest half, the tie that rounds to infinity, overflow
    rgb[0, 2] = (1 + 2 ** -11, 1 + 3 * 2 ** -11, 0.0031308)   # ties to even in both directions
    L = pb.lib()
    path = str(tmp_path / "out.exr").encode()
    assert L.pb2h_write_image(path, pb.ptr(rgb), w, h, 20, 10, 3, 2) == 0
    b = open(path, "rb").read()
    assert struct.unpack_from("<II", b, 0) == (20000630, 2)
    pos, attrs = 8, {}
    while b[pos] != 0:
        name_end = b.index(b"\0", pos)
        type_end = b.index(b"\0", name_end + 1)
        size = struct.unpack_from("<I", b, type_end + 1)[0]
        attrs[b[pos:name_end].decode()] = (b[name_end + 1:type_end].decode(), b[type_end + 5:type_end + 5 + size])
        pos = type_end + 5 + size
    pos += 1
    assert attrs["compression"] == ("compression", b"\0") and attrs["lineOrder"][1] == b"\0"
    assert struct.unpack("<4i", attrs["dataWindow"][1]) == (3, 2, 3 + w - 1, 2 + h - 1)
    assert struct.unpack("<4i", attrs["displayWindow"][1]) == (0, 0, 19, 9)
    chl = attrs["channels"][1]
    assert [chl[i * 18:i * 18 + 1] for i in range(3)] == [b"B", b"G", b"R"] and all(struct.unpack_from("<i", chl, i * 18 + 2)[0] == 1 for i in range(3))
    offsets = struct.unpack_from("<%dQ" % h, b, pos)
    got = np.zeros((h, w, 3), np.float16)
    for y, off in enumerate(offsets):
        yy, nbytes = struct.unpack_from("<ii", b, off)
        assert yy == 2 + y and nbytes == w * 6
        planes = np.frombuffer(b, np.float16, 3 * w, off + 8).reshape(3, w)
        got[y] = planes[::-1].T              # B, G, R planes -> rgb
    assert offsets[-1] + 8 + w * 6 == len(b)
    with np.errstate(over="ignore"):
        want = rgb.astype(np.float16)        # IEEE round-to-nearest-even, overflow to inf: what half(float) does
    assert np.array_equal(got.view(np.uint16), want.view(np.uint16))
    assert np.isinf(got[0, 1, 1]) and got[0, 1, 0] == 65504 and got[0, 0, 1] == 0 and got[0, 0, 2] != 0

    img = np.clip(rgb, 0, 2)
    path = str(tmp_path / "out.png").encode()
    assert L.pb2h_write_image(path, pb.ptr(img), w, h, w, h, 0, 0) == 0
    b = open(path, "rb").read()
    assert b[:8] == bytes([0x89, 80, 78, 71, 13, 10, 26, 10])
    pos, chunks = 8, []
    while pos < len(b):
        n, typ = struct.unpack_from(">I4s", b, pos)
        data = b[pos + 8:pos + 8 + n]
        assert struct.unpack_from(">I", b, pos + 8 + n)[0] == zlib.crc32(typ + data)
        chunks.append((typ, data))
        pos += 12 + n
    assert [c[0] for c in chunks] == [b"IHDR", b"IDAT", b"IEND"]
    assert struct.unpack(">IIBBBBB", chunks[0][1]) == (w, h, 8, 2, 0, 0, 0)
    raw = np.frombuffer(zlib.decompress(chunks[1][1]), np.uint8).reshape(h, 1 + 3 * w)
    assert (raw[:, 0] == 0).all()
    px = raw[:, 1:].reshape(h, w, 3).astype(int)
    assert np.abs(px - _to_byte(img).astype(int)).max() <= 1 and (px == _to_byte(img)).mean() > 0.95   # powf vs numpy's pow at .5 boundaries

    path = str(tmp_path / "out.tga").encode()
    assert L.pb2h_write_image(path, pb.ptr(img), w, h, w, h, 0, 0) == 0
    b = open(path, "rb").read()
    assert b[:3] == bytes([0, 0, 2]) and struct.unpack_from("<HHHHBB", b, 8) == (0, 0, w, h, 24, 0x20) and len(b) == 18 + 3 * w * h
    bgr = np.frombuffer(b, np.uint8, 3 * w * h, 18).reshape(h, w, 3)
    assert np.array_equal(bgr[..., ::-1], px)
    # a big image crosses the 65535-byte stored-block limit of deflate
    big = rng.rand(120, 300, 3).astype(np.float32)
    path = str(tmp_path / "big.png").encode()
    assert L.pb2h_write_image(path, pb.ptr(big), 300, 120, 300, 120, 0, 0) == 0
    b = open(path, "rb").read()
    n = struct.unpack_from(">I", b, 33)[0]
    raw = np.frombuffer(zlib.decompress(b[41:41 + n]), np.uint8).reshape(120, 901)
    assert np.abs(raw[:, 1:].reshape(120, 300, 3).astype(int) - _to_byte(big).astype(int)).max() <= 1
    assert L.pb2h_write_image(str(tmp_path / "out.bmp").encode(), pb.ptr(img), w, h, w, h, 0, 0) != 0


def test_quick_render_option(pb):
    """--quick (pbrt.cpp:116-117): Film divides the resolution by 4 (film.cpp:228-229), Halton takes one sample (halton.cpp:136)."""
    text = open(os.path.join(SCENES, "materials.pbrt")).read()
    pb.lib().pb2h_set_quick_render(1)
    try:
        hs = pb.HostScene.from_string(text)
        assert tuple(hs.film.contents.full_resolution) == (12, 8) and hs.params.contents.samples_per_pixel == 1
    finally:
        pb.lib().pb2h_set_quick_render(0)
    hs = pb.HostScene.from_string(text)
    assert tuple(hs.film.contents.full_resolution) == (48, 32) and hs.params.contents.samples_per_pixel == 8


def test_constant_valued_texture_directives(pb):
    """Texture "..." "constant" / "scale" / "mix" of constants (pbrtTexture api.cpp:1189-1245, constant.cpp, scale.cpp,
    mix.cpp) resolve to the value a material parameter naming them gets; textures that vary over the surface are reported."""
    f32 = np.float32
    text = """WorldBegin
Texture "base" "spectrum" "constant" "rgb value" [.2 .4 .6]
Texture "rough" "float" "constant" "float value" .25
Texture "dim" "color" "scale" "texture tex1" "base" "rgb tex2" [.5 .5 2]
Texture "blend" "spectrum" "mix" "texture tex1" "base" "rgb tex2" [1 1 1] "float amount" .25
Texture "r2" "float" "mix" "texture tex1" "rough" "float tex2" 1 "texture amount" "rough"
AttributeBegin
  Texture "base" "spectrum" "constant" "rgb value" [9 9 9]
AttributeEnd
Material "plastic" "texture Kd" "dim" "texture Ks" "blend" "texture roughness" "r2"
Shape "sphere"
Material "matte" "texture Kd" "base"
Shape "sphere" "float radius" 2
Material "uber" "texture uroughness" "rough"
Shape "sphere" "float radius" 3
WorldEnd
"""
    before = pb.lib().pb2h_error_count()
    hs = pb.HostScene.from_string(text)
    assert pb.lib().pb2h_error_count() == before
    d = hs.desc.contents
    mats = [d.materials[i] for i in range(d.n_materials)]
    plastic = [m for m in mats if m.type == pb.PB2_MAT_PLASTIC][0]
    assert tuple(plastic.kd) == (f32(.2) * f32(.5), f32(.4) * f32(.5), f32(.6) * f32(2))
    amt = f32(.25)
    assert tuple(plastic.ks) == tuple((f32(1) - amt) * f32(v) + amt * f32(1) for v in (.2, .4, .6))
    assert plastic.roughness == (f32(1) - amt) * amt + amt * f32(1)
    matte = [m for m in mats if m.type == pb.PB2_MAT_MATTE and tuple(m.kd) != (.5, .5, .5)][0]
    assert tuple(matte.kd) == (f32(.2), f32(.4), f32(.6))          # the redefinition inside the attribute block is gone again
    uber = [m for m in mats if m.type == pb.PB2_MAT_UBER][0]
    assert uber.uroughness == f32(.25) == uber.vroughness
    hs = pb.HostScene.from_string('WorldBegin\nTexture "img" "spectrum" "dots"\n'
                                  'Material "matte" "texture Kd" "img"\nShape "sphere"\nWorldEnd\n')
    assert pb.lib().pb2h_error_count() >= before + 2                 # the directive and the parameter that names it


def test_image_texture_directives(pb, tmp_path):
    """Texture "..." "imagemap" (imagemap.cpp:113-197): the readers (PFM, PNG with every scanline filter, run-length TGA), the
    flip in y, scale / inverse gamma / luminance (imagemap.h:97-106), the mapping and filter parameters, the slots of the
    materials that name the textures (with the u / v roughness fall-backs), alpha / shadowalpha masks, and the errors."""
    import ctypes as C
    f32 = np.float32
    tex = os.path.join(SCENES, "textures")
    dec = np.load(os.path.join(tex, "decoded_8bit.npz"))
    text = """WorldBegin
Texture "png" "spectrum" "imagemap" "string filename" "%(t)s/tiles_20x12.png" "float scale" 2 "float maxanisotropy" 4 "string wrap" "clamp"
Texture "png-linear" "spectrum" "imagemap" "string filename" "%(t)s/tiles_20x12.png" "bool gamma" "false" "float uscale" 3 "float vdelta" .5
Texture "tga" "color" "imagemap" "string filename" "%(t)s/tiles_24x10.tga" "bool gamma" "false" "bool trilinear" "true" "string wrap" "black"
Texture "tga-y" "float" "imagemap" "string filename" "%(t)s/tiles_24x10.tga"
Texture "holes" "float" "imagemap" "string filename" "%(t)s/holes_16x16.pfm"
Texture "missing" "float" "imagemap" "string filename" "%(t)s/nothing.pfm"
Texture "zero" "float" "constant" "float value" 0
Material "plastic" "texture Kd" "png" "texture Ks" "tga" "texture roughness" "tga-y"
Shape "sphere"
Material "uber" "texture Kd" "png-linear" "texture roughness" "tga-y" "texture vroughness" "holes" "texture index" "missing"
Shape "sphere" "float radius" 2
Material "metal" "texture roughness" "holes" "float uroughness" .3
Shape "sphere" "float radius" 3
Material "matte"
Shape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 0 1 0 0 0 1 0] "texture alpha" "holes" "texture shadowalpha" "tga-y"
Shape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 1 1 0 1 0 1 1] "texture alpha" "zero"
Shape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 2 1 0 2 0 1 2] "float shadowalpha" 0
WorldEnd
""" % {"t": tex}
    before = pb.lib().pb2h_error_count()
    hs = pb.HostScene.from_string(text)
    assert pb.lib().pb2h_error_count() == before + 1          # nothing.pfm cannot be read (a grey 1 x 1 texture replaces it)
    d = hs.desc.contents
    T = {}
    mats = {d.materials[i].type: d.materials[i] for i in range(d.n_materials)}

    def texels(t):
        return np.ctypeslib.as_array(t.texels, shape=(t.height, t.width, t.channels))

    def igc(v):   # InverseGammaCorrect in float (pbrt.h:298-301)
        v = np.asarray(v, f32)
        return np.where(v <= f32(0.04045), v * f32(1) / f32(12.92), np.power((v + f32(0.055)) * f32(1) / f32(1.055), f32(2.4)).astype(f32))

    plastic, uber, metal = mats[pb.PB2_MAT_PLASTIC], mats[pb.PB2_MAT_UBER], mats[pb.PB2_MAT_METAL]
    png = d.textures[plastic.tex[pb.PB2_TEX_KD] - 1]
    assert (png.channels, png.width, png.height, png.wrap, png.do_trilinear, png.max_anisotropy) == (3, 20, 12, pb.PB2_WRAP_CLAMP, 0, 4.0)
    want = f32(2) * igc(dec["png"][::-1].astype(f32) / f32(255))            # row 0 of the texels is the image's LAST row
    assert np.allclose(texels(png), want, rtol=2e-6, atol=0)                 # (powf may differ from numpy's in the last bit)
    lin = d.textures[uber.tex[pb.PB2_TEX_KD] - 1]
    assert np.array_equal(texels(lin), dec["png"][::-1].astype(f32) / f32(255))
    assert (lin.su, lin.sv, lin.du, lin.dv, lin.wrap) == (3.0, 1.0, 0.0, 0.5, pb.PB2_WRAP_REPEAT)
    tga = d.textures[plastic.tex[pb.PB2_TEX_KS] - 1]
    assert (tga.channels, tga.width, tga.height, tga.wrap, tga.do_trilinear) == (3, 24, 10, pb.PB2_WRAP_BLACK, 1)
    assert np.array_equal(texels(tga), dec["tga"][::-1].astype(f32) / f32(255))
    tga_y = d.textures[plastic.tex[pb.PB2_TEX_ROUGHNESS] - 1]
    c = dec["tga"][::-1].astype(f32) / f32(255)
    y = f32(0.212671) * c[..., 0] + f32(0.715160) * c[..., 1] + f32(0.072169) * c[..., 2]
    assert tga_y.channels == 1 and np.allclose(texels(tga_y)[..., 0], igc(y), rtol=2e-6, atol=0)   # .tga: gamma defaults to true
    # uber.cpp:71-80: u <- "roughness" (no "uroughness" given), v <- "vroughness"; "index" names the unreadable file
    assert uber.tex[pb.PB2_TEX_UROUGHNESS] == plastic.tex[pb.PB2_TEX_ROUGHNESS] and uber.tex[pb.PB2_TEX_ROUGHNESS] == 0
    holes = d.textures[uber.tex[pb.PB2_TEX_VROUGHNESS] - 1]
    assert (holes.channels, holes.width, holes.height) == (1, 16, 16) and set(np.unique(texels(holes))) == {0.0, 1.0}
    grey = d.textures[uber.tex[pb.PB2_TEX_ETA] - 1]
    assert (grey.channels, grey.width, grey.height) == (1, 1, 1) and texels(grey).ravel()[0] == f32(0.212671) * f32(.5) + f32(0.715160) * f32(.5) + f32(0.072169) * f32(.5)
    # metal.cpp:67-70: "uroughness" is a constant, v falls back to the "roughness" texture
    assert metal.tex[pb.PB2_TEX_UROUGHNESS] == 0 and metal.uroughness == f32(.3) and metal.tex[pb.PB2_TEX_VROUGHNESS] == uber.tex[pb.PB2_TEX_VROUGHNESS]
    meshes = [d.meshes[i] for i in range(d.n_meshes)]
    assert meshes[0].alpha_tex == uber.tex[pb.PB2_TEX_VROUGHNESS] and meshes[0].shadow_alpha_tex == plastic.tex[pb.PB2_TEX_ROUGHNESS]
    zero = d.textures[meshes[1].alpha_tex - 1]
    assert meshes[1].shadow_alpha_tex == 0 and (zero.width, zero.height) == (1, 1) and texels(zero).ravel()[0] == 0
    assert meshes[2].alpha_tex == 0 and texels(d.textures[meshes[2].shadow_alpha_tex - 1]).ravel()[0] == 0
    # outside the scope: other mappings, a float texture where a spectrum is expected, an unreadable container
    for bad in ('Texture "t" "spectrum" "imagemap" "string filename" "%s/holes_16x16.pfm" "string mapping" "spherical"\nMaterial "matte" "texture Kd" "t"' % tex,
                'Texture "t" "float" "imagemap" "string filename" "%s/holes_16x16.pfm"\nMaterial "matte" "texture Kd" "t"' % tex,
                'Texture "t" "spectrum" "imagemap" "string filename" "%s/tiles.exr"\nMaterial "matte" "texture Kd" "t"' % tex):
        before = pb.lib().pb2h_error_count()
        pb.HostScene.from_string('WorldBegin\n%s\nShape "sphere"\nWorldEnd\n' % bad)
        assert pb.lib().pb2h_error_count() > before, bad


def test_plymesh_reader(pb, tmp_path):
    """Shape "plymesh" (src/shapes/plymesh.cpp): ASCII, binary little- and big-endian files with normals and uv give the
    same mesh as the equivalent "trianglemesh"; a quad becomes (0,1,2),(3,0,2) (plymesh.cpp:137-145), a pentagon is skipped
    with a warning (plymesh.cpp:112-116)."""
    import struct
    rng = np.random.RandomState(4)
    P = rng.rand(6, 3).astype(np.float32)
    N = rng.normal(size=(6, 3)).astype(np.float32)
    UV = rng.rand(6, 2).astype(np.float32)
    faces = [[0, 1, 2], [2, 3, 4, 5], [0, 1, 2, 3, 4], [5, 1, 3]]
    want_idx = [0, 1, 2, 2, 3, 4, 5, 2, 4, 5, 1, 3]
    header = ("ply\nformat %s 1.0\ncomment test\nelement vertex 6\nproperty float x\nproperty float y\nproperty float z\n"
              "property float nx\nproperty float ny\nproperty float nz\nproperty float u\nproperty float v\n"
              "element face 4\nproperty list uchar int vertex_indices\nend_header\n")
    files = {}
    body = "".join(" ".join("%.9g" % x for x in np.concatenate([P[i], N[i], UV[i]])) + "\n" for i in range(6))
    body += "".join("%d %s\n" % (len(f), " ".join(map(str, f))) for f in faces)
    files["ascii"] = (header % "ascii" + body).encode()
    for fmt, e in (("binary_little_endian", "<"), ("binary_big_endian", ">")):
        b = b"".join(struct.pack(e + "8f", *np.concatenate([P[i], N[i], UV[i]])) for i in range(6))
        b += b"".join(struct.pack(e + "B%di" % len(f), len(f), *f) for f in faces)
        files[fmt] = (header % fmt).encode() + b
    scene = ('Camera "perspective"\nFilm "image" "integer xresolution" [4] "integer yresolution" [4]\nWorldBegin\nTranslate .1 .2 .3\n%s\nWorldEnd\n')
    tri = 'Shape "trianglemesh" "integer indices" [%s] "point P" [%s] "normal N" [%s] "float uv" [%s]' % (
        " ".join(map(str, want_idx)), " ".join("%.9g" % x for x in P.ravel()), " ".join("%.9g" % x for x in N.ravel()),
        " ".join("%.9g" % x for x in UV.ravel()))
    hs = pb.HostScene.from_string(scene % tri)
    d = hs.desc.contents

    def arrays(d):
        nv = d.n_vertices
        return (np.ctypeslib.as_array(d.P, shape=(nv, 3)).copy(), np.ctypeslib.as_array(d.N, shape=(nv, 3)).copy(),
                np.ctypeslib.as_array(d.UV, shape=(nv, 2)).copy(), np.ctypeslib.as_array(d.tri_index, shape=(d.n_tris * 3,)).copy())
    want = arrays(d)
    assert d.n_tris == 4
    for fmt, data in files.items():
        path = tmp_path / (fmt + ".ply")
        path.write_bytes(data)
        hs = pb.HostScene.from_string(scene % ('Shape "plymesh" "string filename" "%s"' % path))
        got = arrays(hs.desc.contents)
        for a, b in zip(got, want):
            assert np.array_equal(a, b), fmt


def _mesh_world_points(hs):
    d = hs.desc.contents
    return np.ctypeslib.as_array(d.P, shape=(d.n_vertices, 3)).copy()


def test_include_named_materials_and_coordinate_systems(pb, tmp_path):
    """Include (parser.cpp:1013-1024, relative to the including file), MakeNamedMaterial / NamedMaterial (api.cpp:1247-1300),
    CoordinateSystem / CoordSysTransform (api.cpp:842-868), Transform / ConcatTransform (column-major, api.cpp:796-840)."""
    f32 = np.float32
    inc = tmp_path / "geometry.pbrt"
    inc.write_text('NamedMaterial "shiny"\nShape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 0 1 0 0 0 1 0]\n')
    main = tmp_path / "main.pbrt"
    main.write_text("""Camera "perspective"
Film "image" "integer xresolution" [4] "integer yresolution" [4]
WorldBegin
MakeNamedMaterial "shiny" "string type" "plastic" "rgb Kd" [.1 .2 .3] "float roughness" .07
MakeNamedMaterial "dull" "string type" "matte" "rgb Kd" [.9 .8 .7]
Translate 1 2 3
CoordinateSystem "shifted"
AttributeBegin
  Scale 2 2 2
  Include "geometry.pbrt"
AttributeEnd
AttributeBegin
  Identity
  Transform [0 1 0 0  -1 0 0 0  0 0 1 0  5 6 7 1]
  ConcatTransform [1 0 0 0  0 1 0 0  0 0 1 0  0 0 10 1]
  NamedMaterial "dull"
  Shape "trianglemesh" "integer indices" [0 1 2] "point P" [1 0 0 0 1 0 0 0 1]
AttributeEnd
TransformBegin
  Identity
  CoordSysTransform "shifted"
  NamedMaterial "nosuch"
  Shape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 0 1 0 0 0 1 0]
TransformEnd
WorldEnd
""")
    before = pb.lib().pb2h_error_count()
    hs = pb.HostScene.from_file(str(main))
    assert pb.lib().pb2h_error_count() == before + 1          # only the unknown named material (api.cpp:1290-1293)
    P = _mesh_world_points(hs)
    # mesh 1: Translate(1,2,3) * Scale(2)
    assert np.array_equal(P[0:3], np.array([[1, 2, 3], [3, 2, 3], [1, 4, 3]], f32))
    # mesh 2: column-major matrix = rotation by 90 degrees about z then translation (5,6,7); ConcatTransform adds z + 10 first
    assert np.array_equal(P[3:6], np.array([[5, 7, 17], [4, 6, 17], [5, 6, 18]], f32))
    # mesh 3: the named coordinate system is the CTM at the time it was named
    assert np.array_equal(P[6:9], np.array([[1, 2, 3], [2, 2, 3], [1, 3, 3]], f32))
    d = hs.desc.contents
    pm = np.ctypeslib.as_array(d.prim_material, shape=(d.n_prims,))
    kinds = [(d.materials[m].type, tuple(np.float32(x) for x in d.materials[m].kd)) for m in pm]
    assert kinds[0] == (pb.PB2_MAT_PLASTIC, (f32(.1), f32(.2), f32(.3))) and kinds[1] == (pb.PB2_MAT_MATTE, (f32(.9), f32(.8), f32(.7)))
    # an unknown NamedMaterial leaves the current material in place: at world level that is the default matte (api.cpp:207-210)
    assert kinds[2] == (pb.PB2_MAT_MATTE, (f32(.5), f32(.5), f32(.5)))


def test_camera_film_sampler_and_integrator_parameters(pb):
    """CreatePerspectiveCamera (perspective.cpp:246-290), CreateFilm (film.cpp:213-252), CreateHaltonSampler (halton.cpp:133-140),
    CreatePathIntegrator (path.cpp:190-213): every parameter reaches the ABI structs with the reference's defaults and rules."""
    f32 = np.float32

    def parse(camera="", film="", sampler="", integrator=""):
        return pb.HostScene.from_string('Camera "perspective" %s\nFilm "image" "integer xresolution" [30] "integer yresolution" [20] %s\n'
                                        'Sampler "halton" %s\nIntegrator "path" %s\nWorldBegin\nShape "sphere"\nWorldEnd\n' % (camera, film, sampler, integrator))
    hs = parse()
    cam, film, pp = hs.camera.contents, hs.film.contents, hs.params.contents
    assert tuple(cam.screen_window) == (-1.5, 1.5, -1, 1) and cam.fov == 90 and cam.lens_radius == 0 and cam.focal_distance == f32(1e6)
    assert (cam.shutter_open, cam.shutter_close) == (0, 1)
    assert tuple(film.cropped_pixel_bounds) == (0, 0, 30, 20) and film.scale == 1 and np.isinf(film.max_sample_luminance)
    assert pp.samples_per_pixel == 16 and pp.sample_at_pixel_center == 0 and pp.max_depth == 5 and pp.rr_threshold == 1
    assert tuple(pp.pixel_bounds) == (0, 0, 30, 20)
    hs = parse(camera='"float frameaspectratio" .5 "float halffov" 20 "float lensradius" .1 "float focaldistance" 3 "float shutteropen" .8 "float shutterclose" .2')
    cam = hs.camera.contents
    assert tuple(cam.screen_window) == (-1, 1, -2, 2) and cam.fov == 40 and cam.lens_radius == f32(.1) and cam.focal_distance == 3
    assert (cam.shutter_open, cam.shutter_close) == (f32(.2), f32(.8))           # swapped with a warning (perspective.cpp:253-257)
    hs = parse(camera='"float screenwindow" [-2 1 -.5 .25] "float fov" 30')
    assert tuple(hs.camera.contents.screen_window) == (-2, 1, f32(-.5), f32(.25))
    hs = parse(film='"float cropwindow" [.1 .5 .25 .75] "float scale" 2.5 "float maxsampleluminance" 10',
               sampler='"integer pixelsamples" 3 "bool samplepixelcenter" "true"',
               integrator='"integer maxdepth" 9 "float rrthreshold" .25 "integer pixelbounds" [2 9 1 12]')
    film, pp = hs.film.contents, hs.params.contents
    assert tuple(film.cropped_pixel_bounds) == (3, 5, 15, 15)                     # ceil(res * crop) (film.cpp:55-60)
    assert film.scale == 2.5 and film.max_sample_luminance == 10
    assert pp.samples_per_pixel == 3 and pp.sample_at_pixel_center == 1 and pp.max_depth == 9 and pp.rr_threshold == f32(.25)
    # pixelbounds is given as x0 x1 y0 y1 and intersected with the camera's sample bounds (path.cpp:195-207)
    assert tuple(pp.pixel_bounds) == (3, 5, 9, 12)


def test_sobol_sampler_directive(pb):
    """Sampler "sobol" (sobol.cpp:65-70, sobol.h:51-57): the sample count is rounded up to a power of two (with a warning),
    "samplepixelcenter" does not exist for it."""
    hs = pb.HostScene.from_string('Sampler "sobol" "integer pixelsamples" 5\nWorldBegin\nShape "sphere"\nWorldEnd\n')
    pp = hs.params.contents
    assert pp.sampler == pb.PB2_SAMPLER_SOBOL and pp.samples_per_pixel == 8 and pp.sample_at_pixel_center == 0
    hs = pb.HostScene.from_string('Sampler "sobol"\nWorldBegin\nShape "sphere"\nWorldEnd\n')
    assert hs.params.contents.samples_per_pixel == 16 and hs.params.contents.sampler == pb.PB2_SAMPLER_SOBOL
    hs = pb.HostScene.from_string('WorldBegin\nShape "sphere"\nWorldEnd\n')
    assert hs.params.contents.sampler == pb.PB2_SAMPLER_HALTON


@pytest.mark.parametrize("header,world,renders", [
    ('Sampler "02sequence" "integer pixelsamples" 4', '', False), ('Camera "orthographic"', '', False), ('Integrator "bdpt"', '', False),
    ('Accelerator "kdtree"', 'Shape "sphere"', True), ('PixelFilter "lanczos"', 'Shape "sphere"', True),
    ('', 'Shape "cylinder"', True), ('', 'LightSource "goniometric"\nShape "sphere"', True),
    ('', 'MakeNamedMedium "fog" "string type" "homogeneous"\nShape "sphere"', True), ('', 'ActiveTransform StartTime\nShape "sphere"', True)])
def test_plugins_outside_the_scope_are_reported(pb, header, world, renders):
    """Every plugin name or directive of the reference that this path does not implement produces an Error() - never a
    silent substitute.  Without a sampler, camera or integrator there is nothing to render (api.cpp:1662-1714 returns no
    integrator either); the others continue with the reported fallback or without the skipped directive."""
    before = pb.lib().pb2h_error_count()
    text = "%s\nWorldBegin\n%s\nWorldEnd\n" % (header, world)
    if renders:
        hs = pb.HostScene.from_string(text)
        assert hs.params.contents.samples_per_pixel == 16
    else:
        with pytest.raises(RuntimeError):
            pb.HostScene.from_string(text)
    assert pb.lib().pb2h_error_count() > before


def test_wide4_records_keep_the_reference_order(pb):
    """Groundwork for the next trace kernel (pbrt_v3_b200/csrc/device/pb2_wide4.cuh): the binary BVH collapsed into four-child
    records and traversed near-first per collapsed level tests the same primitives in the same order as BVHAccel::Intersect's
    loop (bvh.cpp:662-700).  Host-only check with the kernels' slab test; primitives are stood in for by their boxes."""
    import ctypes as C
    L = pb.lib()
    fn = L.pb2_debug_wide4_sequences
    fn.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32] + [C.c_void_p] * 4
    fn.restype = C.c_int
    for maker in (lambda: pb.HostScene.soup(4000, seed=11, jitter=0.25, xres=16, yres=16, spp=1),
                  lambda: pb.HostScene.from_string(gc.with_accelerator(gc.random_mesh_scene_text(3000, 3), "sah", 1)),
                  lambda: pb.HostScene.from_string(gc.with_accelerator(gc.random_mesh_scene_text(5, 3), "sah", 16))):
        hs = maker()
        d = hs.desc.contents
        nodes, prims = np.ascontiguousarray(hs.nodes()), np.ascontiguousarray(hs.bvh_prims(0))
        P = np.ctypeslib.as_array(d.P, shape=(d.n_vertices, 3))
        idx = np.ctypeslib.as_array(d.tri_index, shape=(d.n_tris, 3))
        tri = P[idx][np.ctypeslib.as_array(d.prim_index, shape=(d.n_prims,))]
        bounds = np.ascontiguousarray(np.concatenate([tri.min(axis=1), tri.max(axis=1)], 1), np.float32)
        n = 3000
        rays = gc.rays_for(pb, nodes, n, 2)
        rng = np.random.RandomState(3)
        target = tri[rng.randint(0, len(tri), n)].mean(axis=1)
        aimed = (target - rays["o"]).astype(np.float32)
        od = np.ascontiguousarray(np.concatenate([rays["o"], np.where((np.arange(n) < n // 20)[:, None], rays["d"], aimed)], 1), np.float32)
        max_len = 512
        sb, sw = np.zeros((n, max_len), np.int32), np.zeros((n, max_len), np.int32)
        lb, lw = np.zeros(n, np.int32), np.zeros(n, np.int32)
        assert fn(pb.ptr(nodes), len(nodes), pb.ptr(prims), pb.ptr(bounds), pb.ptr(od), n, max_len, pb.ptr(sb), pb.ptr(sw), pb.ptr(lb), pb.ptr(lw)) == 0
        assert np.array_equal(lb, lw) and lb.max() <= max_len
        assert np.array_equal(sb, sw)
        assert lb.sum() > n // 2                  # leaves were reached (several per ray on the dense soup)


def test_radical_inverse_digit_tables_equal_the_digit_loop(pb):
    """The shade kernels evaluate ScrambledRadicalInverse (lowdiscrepancy.cpp:405-424) through per-dimension digit tables
    (pb2_sampler.cuh: several digits per look-up).  The host build of the same function must give the digit loop's bits for
    every dimension and any 32-bit index: random indices, the sample indices a render uses, block boundaries of the tables."""
    L = pb.lib()
    rng = np.random.RandomState(1)
    idx = np.concatenate([rng.randint(0, 2 ** 32, 300000, dtype=np.uint64), rng.randint(0, 3000000, 200000, dtype=np.uint64),
                          np.arange(100000, dtype=np.uint64)]).astype(np.uint32)
    dim = rng.randint(2, 1000, len(idx)).astype(np.int32)
    dim[: len(idx) // 2] = rng.randint(2, 40, len(idx) // 2)
    for d in (2, 3, 4, 5, 10, 25, 30, 100, 999):
        edge = np.array([0, 1, 2, 3124, 3125, 3126, 8191, 8192, 2 ** 31, 2 ** 32 - 1, 9765624, 9765625, 9765626], np.uint32)
        idx = np.concatenate([idx, edge])
        dim = np.concatenate([dim, np.full(len(edge), d, np.int32)])
    a, b = np.zeros(len(idx), np.float32), np.zeros(len(idx), np.float32)
    L.pb2_debug_radical_inverse_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    assert L.pb2_debug_radical_inverse_tables(pb.ptr(idx), pb.ptr(dim), len(idx), pb.ptr(a), pb.ptr(b)) == 0
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert 0 <= a.min() and a.max() < 1


def test_infinite_light_is_flattened_with_its_transform(pb):
    """LightSource "infinite" (constant radiance; src/lights/infinite.cpp:177-188 for the parameters): first in Scene::lights,
    L * scale, both 3x3 matrices of the CTM, the world radius of Preprocess; an environment map is reported, not silently used."""
    hs = pb.HostScene.from_file(os.path.join(SCENES, "envlight.pbrt"))
    d = hs.desc.contents
    assert d.n_lights == 3 and [d.lights[i].type for i in range(3)] == [pb.PB2_LIGHT_INFINITE, pb.PB2_LIGHT_AREA, pb.PB2_LIGHT_AREA]
    assert np.allclose(list(d.lights[0].L), [.45 * 1.2, .6, .9 * .8]) and d.lights[0].prim == -1
    dl = d.delta_lights[0]
    l2w, w2l = np.array(dl.light_to_world).reshape(3, 3), np.array(dl.world_to_light).reshape(3, 3)
    assert np.allclose(l2w @ w2l, np.eye(3), atol=1e-6) and not np.allclose(l2w, np.eye(3))
    nodes = hs.nodes()
    assert np.isclose(dl.world_radius, 0.5 * np.linalg.norm(nodes["bmax"][0] - nodes["bmin"][0]), rtol=1e-6)
    text = open(os.path.join(SCENES, "envlight.pbrt")).read().replace('"rgb L" [.45 .6 .9]', '"rgb L" [.45 .6 .9] "string mapname" "sky.exr"')
    before = pb.lib().pb2h_error_count()
    hs2 = pb.HostScene.from_string(text)
    # an unreadable map (OpenEXR input is outside the scope) is reported and leaves the constant light (infinite.cpp:58-62)
    assert pb.lib().pb2h_error_count() >= before + 1 and hs2.desc.contents.lights[0].type == pb.PB2_LIGHT_INFINITE
    assert hs2.desc.contents.delta_lights[0].env_tex == 0 and hs2.desc.contents.n_textures == 0


def test_infinite_light_environment_map_is_flattened(pb):
    """LightSource "infinite" "string mapname": the texels are ReadImage(mapname) * (L * scale), NOT flipped in y (infinite.cpp:50-57),
    as one three-channel texture with MIPMap's default parameters, named by pb2_delta_light.env_tex."""
    import struct
    hs = pb.HostScene.from_file(os.path.join(SCENES, "envmap.pbrt"))
    d = hs.desc.contents
    assert d.lights[0].type == pb.PB2_LIGHT_INFINITE and d.delta_lights[0].env_tex == 1 and d.n_textures == 1
    t = d.textures[0]
    assert (t.channels, t.width, t.height, t.wrap, t.do_trilinear, t.max_anisotropy) == (3, 40, 20, pb.PB2_WRAP_REPEAT, 0, 8.0)
    raw = open(os.path.join(SCENES, "textures", "sky_40x20.pfm"), "rb").read()
    body = np.frombuffer(raw[-40 * 20 * 12:], "<f4").reshape(20, 40, 3)[::-1]    # PFM stores the bottom row first
    L = np.float32([.5, .6, .7]) * np.float32([1.2, 1, .9])
    got = np.ctypeslib.as_array(t.texels, shape=(20, 40, 3))
    assert np.array_equal(got, body * L)


def test_bumpmap_parameter(pb):
    """"bumpmap" (GetFloatTextureOrNull, e.g. matte.cpp:70-71) on every material: an image texture goes into the record's
    PB2_TEX_BUMP slot, a constant (plain float or constant texture) becomes a 1 x 1 image, a spectrum texture is refused."""
    tex = os.path.join(SCENES, "textures")
    hs = pb.HostScene.from_file(os.path.join(SCENES, "bumpmap.pbrt"))
    d = hs.desc.contents
    mats = [d.materials[i] for i in range(d.n_materials)]
    bumped = [m for m in mats if m.tex[pb.PB2_TEX_BUMP]]
    assert sorted(m.type for m in bumped) == sorted([pb.PB2_MAT_PLASTIC, pb.PB2_MAT_MATTE, pb.PB2_MAT_PLASTIC, pb.PB2_MAT_MIRROR, pb.PB2_MAT_GLASS,
                                                     pb.PB2_MAT_MATTE, pb.PB2_MAT_UBER])
    const = [m for m in bumped if m.type == pb.PB2_MAT_MATTE and not m.tex[pb.PB2_TEX_KD]][0]
    t = d.textures[const.tex[pb.PB2_TEX_BUMP] - 1]
    assert (t.channels, t.width, t.height) == (1, 1, 1) and t.texels[0] == np.float32(0.15)
    for i in range(d.n_textures):
        if d.textures[i].width == 32:
            assert d.textures[i].channels == 1
    before = pb.lib().pb2h_error_count()
    pb.HostScene.from_string('WorldBegin\nTexture "t" "spectrum" "imagemap" "string filename" "%s/tiles_37x23.pfm"\n'
                             'Material "matte" "texture bumpmap" "t"\nShape "sphere"\nWorldEnd\n' % tex)
    assert pb.lib().pb2h_error_count() > before


def test_texture_combinators(pb):
    """Texture "scale" / "mix" with an operand that varies (scale.cpp:40-52, mix.cpp:40-54): nodes of the description's texture
    array whose children precede them; constant operands become constant nodes; combinators of constants alone stay folded."""
    hs = pb.HostScene.from_file(os.path.join(SCENES, "texcombine.pbrt"))
    d = hs.desc.contents
    tex = [d.textures[i] for i in range(d.n_textures)]
    kinds = [t.kind for t in tex]
    assert kinds.count(pb.PB2_TEXKIND_SCALE) == 3 and kinds.count(pb.PB2_TEXKIND_MIX) == 3
    for i, t in enumerate(tex):
        if t.kind in (pb.PB2_TEXKIND_SCALE, pb.PB2_TEXKIND_MIX):
            n = 3 if t.kind == pb.PB2_TEXKIND_MIX else 2
            assert all(1 <= t.child[c] <= i for c in range(n)) and not t.texels
            assert all(tex[t.child[c] - 1].channels == t.channels for c in range(2))
            if n == 3:
                assert tex[t.child[2] - 1].channels == 1
    washed = [t for t in tex if t.kind == pb.PB2_TEXKIND_MIX and tex[t.child[0] - 1].kind == pb.PB2_TEXKIND_SCALE][0]   # two levels
    assert tuple(np.float32(v) for v in tex[washed.child[1] - 1].value) == (np.float32(.8),) * 3 and tex[washed.child[2] - 1].value[0] == np.float32(.3)
    # constants alone: folded into the material record, no texture nodes
    hs = pb.HostScene.from_string('WorldBegin\nTexture "a" "spectrum" "scale" "rgb tex1" [.5 .5 .5] "rgb tex2" [.5 1 2]\n'
                                  'Material "matte" "texture Kd" "a"\nShape "sphere"\nWorldEnd\n')
    assert hs.desc.contents.n_textures == 0 and tuple(hs.desc.contents.materials[0].kd) == (.25, .5, 1.0)


def test_openexr_reader(pb, tmp_path):
    """ReadImage for OpenEXR scan-line files (imageio.cpp:125-151 reads them through OpenEXR's RgbaInputFile): half channels
    stored B, G, R; ZIP blocks of 16 lines (the last one short) with the byte-delta predictor and the even / odd byte split,
    blocks stored raw when they do not shrink, uncompressed files, and the RLE and PIZ codecs - the committed files of
    tests/scenes/make_textures.py (those under tests/golden/openexr/ written by the OpenEXR library itself) and the container
    this library writes itself."""
    tex = os.path.join(SCENES, "textures")
    want = np.load(os.path.join(tex, "decoded_8bit.npz"))["exr"]
    for kind in ("zip", "zips", "none"):
        got = pb.read_image(os.path.join(tex, "tiles_24x18_%s.exr" % kind))
        assert got.shape == (18, 24, 3) and np.array_equal(got, want), kind
    assert want[3, 5, 0] == 1000.0 and 0 < want[3, 5, 1] < 0.0011          # values beyond 8 bits, a subnormal-range half
    # the writer of Film::WriteImage (half, uncompressed) and this reader are inverse to each other on half values
    out = str(tmp_path / "roundtrip.exr")
    assert pb.lib().pb2h_write_image(out.encode(), pb.ptr(np.ascontiguousarray(want)), 24, 18, 24, 18, 0, 0) == 0
    assert np.array_equal(pb.read_image(out), want)
    # as a texture: the directive reads it like any other container (no gamma for .exr)
    hs = pb.HostScene.from_string('WorldBegin\nTexture "t" "spectrum" "imagemap" "string filename" "%s/tiles_24x18_zip.exr"\n'
                                  'Material "matte" "texture Kd" "t"\nShape "sphere"\nWorldEnd\n' % tex)
    t = hs.desc.contents.textures[0]
    assert np.array_equal(np.ctypeslib.as_array(t.texels, shape=(18, 24, 3)), want[::-1])
    # files written by the OpenEXR library itself (tests/golden/openexr/, made by tests/scenes/make_textures.py), one picture
    # under every lossless codec: PIZ (value table + wavelet + Huffman with run lengths) in blocks of 32 lines, the last one
    # short, also stored in decreasing line order
    ilm = os.path.join(GOLDEN, "openexr")
    want = np.load(os.path.join(ilm, "decoded.npz"))["exr"]
    for codec in ("rle", "zips", "zip", "piz", "piz_decreasing"):
        got = pb.read_image(os.path.join(ilm, "tiles_40x70_%s.exr" % codec))
        assert got.shape == (70, 40, 3) and np.array_equal(got.view(np.uint32), want.view(np.uint32)), codec
    # the lossy codecs are reported, not misread
    before = pb.lib().pb2h_error_count()
    with pytest.raises(RuntimeError):
        pb.read_image(os.path.join(ilm, "tiles_40x70_b44.exr"))
    assert pb.lib().pb2h_error_count() > before
