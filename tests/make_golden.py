"""Generates tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref, built from /root/reference by
oracle/Makefile.ref) on the seeded inputs of tests/golden_cases.py.  Run in the build container:

    python tests/make_golden.py

The fixtures travel with the repo; the tests compare the oracle port (everywhere) and the CUDA path (on the GPU box)
against them, so that parity is pinned to the reference even where /root/reference does not exist.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import golden_cases as gc  # noqa: E402
import pbrt_v3_b200 as pb  # noqa: E402
from oracle import pyoracle  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def canonical_nodes(nodes):
    """LinearBVHNode::axis of a leaf and the pad byte are never written by the reference (bvh.cpp:640-658): zero them, so
    that regenerating the fixtures reproduces the files (the tests ignore those bytes, tests/test_oracle.py same_bvh)."""
    nodes = nodes.copy()
    nodes["axis"][nodes["n_prims"] > 0] = 0
    nodes["pad"] = 0
    return nodes


def record_scene(ref, hs, name, n_rays=1500, n_samples=3000, n_points=400):
    rs = ref.scene(hs)
    nodes = hs.nodes()
    xres, yres = hs.film.contents.full_resolution[0], hs.film.contents.full_resolution[1]
    spp = hs.params.contents.samples_per_pixel
    rays = gc.rays_for(pb, nodes, n_rays, 11)
    srays = gc.rays_for(pb, nodes, n_rays, 12, shadow=True)
    pix, sn = gc.sample_ids(xres, yres, spp, n_samples, 13)
    hpix, hsn, hdim = gc.sample_ids(xres, yres, spp, 4000, 14, max_dim=200)
    pts = gc.points_for(nodes, n_points, 15)
    li, pfilm = rs.li_samples(pix, sn)
    img, _, st = rs.render(n_threads=0)
    ref_nodes, ref_prims = rs.bvh()
    np.savez_compressed(os.path.join(OUT, name + ".npz"),
                        hits=rs.intersect(rays), occluded=rs.intersect_p(srays),
                        halton=ref.halton(hs.film, hs.params, hpix, hsn, hdim),
                        light_distribution=rs.light_distribution(pts), li=li, pfilm=pfilm, image=img,
                        rays=np.array([st.camera_rays, st.regular_rays, st.shadow_rays], np.int64),
                        bvh_nodes=canonical_nodes(ref_nodes), bvh_prims=ref_prims)
    print(name, "image mean", img.mean(), "rays", st.camera_rays, st.regular_rays, st.shadow_rays)


def record_filters(ref):
    """One image per reconstruction-filter case (tests/golden_cases.py FILTER_CASES), rendered by one thread."""
    out = {}
    for case in gc.FILTER_CASES:
        hs = pb.HostScene.from_string(gc.filter_scene_text(os.path.join(ROOT, "tests", "scenes"), case))
        img, _, st = ref.scene(hs).render(n_threads=1)
        out["image_" + case] = img
        out["rays_" + case] = np.array([st.camera_rays, st.regular_rays, st.shadow_rays], np.int64)
        f = hs.film.contents
        out["film_" + case] = np.array([f.filter_type, *f.filter_radius, *f.filter_param, *f.cropped_pixel_bounds], np.float64)
        print("filter", case, "image mean", img.mean())
    np.savez_compressed(os.path.join(OUT, "filters.npz"), **out)


def record_hlbvh(ref):
    """BVHAccel's linear nodes and primitive order with splitmethod "hlbvh" (bvh.cpp:404-638).  The reference hands out the
    ordered-primitive slots of the treelets through an atomic counter, so the order is only reproducible with one
    worker thread: ref_li_samples switches the reference to one thread before the scenes are built."""
    warm = gc.soup_scene(pb)
    ref.scene(warm).li_samples(np.zeros((1, 2), np.int32), np.zeros(1, np.int64))
    out = {}
    cases = [("killeroo_like", open(os.path.join(ROOT, "tests", "scenes", "killeroo_like.pbrt")).read(), mp) for mp in (4, 1, 16)]
    cases.append(("random20k", gc.random_mesh_scene_text(20000, 5), 4))
    for name, text, mp in cases:
        hs = pb.HostScene.from_string(gc.with_accelerator(text, "hlbvh", mp))
        nodes, prims = ref.scene(hs, max_prims_in_node=mp, split_method=1).bvh()
        out["nodes_%s_%d" % (name, mp)], out["prims_%s_%d" % (name, mp)] = canonical_nodes(nodes), prims
        print("hlbvh", name, mp, len(nodes), "nodes")
    np.savez_compressed(os.path.join(OUT, "hlbvh.npz"), **out)


def record_textures(ref):
    """MIPMap::Lookup of the reference for every image texture of tests/scenes/textured.pbrt (EWA and trilinear, the three
    wrap modes, resampled and power-of-two pyramids, one- and three-channel) over tests/golden_cases.py's footprints,
    and a checksum of every pyramid level."""
    hs = pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "textured.pbrt"))
    out = {}
    for i, t in enumerate(hs.textures()):
        st, dst = gc.texture_lookup_inputs(3000, 100 + i)
        out["lookup_%d" % i] = ref.texture_lookup(t, st, dst)
        levels = ref.texture_pyramid(t)
        out["levels_%d" % i] = np.array([[lv.shape[1], lv.shape[0]] for lv in levels], np.int32)
        out["pyramid_%d" % i] = np.concatenate([lv.ravel() for lv in levels])
    np.savez_compressed(os.path.join(OUT, "textures.npz"), **out)
    print("textures:", len(hs.textures()), "textures recorded")


def record_texture_evaluations(ref):
    """Texture::Evaluate of the reference's own texture objects (ImageTexture's filter behind a UVMapping2D, ConstantTexture,
    ScaleTexture, MixTexture, Checkerboard2DTexture, UVTexture) for every texture of the textured golden scenes, at the points
    and differentials of tests/golden_cases.py."""
    out = {}
    for scene in gc.TEXTURE_EVAL_SCENES:
        hs = pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", scene + ".pbrt"))
        d = hs.desc.contents
        uv, duv = gc.texture_eval_inputs(2000, 7)
        for t in range(d.n_textures):
            out["%s_%d" % (scene, t)] = ref.texture_evaluate(d.textures, d.n_textures, t, uv, duv)
    np.savez_compressed(os.path.join(OUT, "texture_evaluations.npz"), **out)
    print("texture evaluations:", len(out), "textures")


def record_differentials(ref):
    """Camera rays with their differentials, first hits and the (u, v) differentials there, from the reference
    (GenerateRayDifferential + ScaleDifferentials, Scene::Intersect, SurfaceInteraction::ComputeDifferentials)."""
    out = {}
    for scene in gc.DIFFERENTIAL_SCENES:
        hs = pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", scene + ".pbrt"))
        f = hs.film.contents
        pix, sn = gc.sample_ids(f.full_resolution[0], f.full_resolution[1], hs.params.contents.samples_per_pixel, 3000, 13)
        out[scene] = ref.scene(hs).camera_differentials(pix, sn)
    np.savez_compressed(os.path.join(OUT, "differentials.npz"), **out)
    print("differentials:", {k: int((v[:, 22] > 0).sum()) for k, v in out.items()})


def record_bsdfs(ref):
    """BSDF::f / Pdf / Sample_f of the reference for every material record of the material golden scenes at random frames."""
    out = {}
    for scene in gc.BSDF_SCENES:
        hs = pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", scene + ".pbrt"))
        d = hs.desc.contents
        for m in range(d.n_materials):
            out["%s_%d" % (scene, m)] = ref.bsdf_eval(d.materials[m], gc.bsdf_frames(1500, 17 + m))
    np.savez_compressed(os.path.join(OUT, "bsdf.npz"), **out)
    print("bsdf:", len(out), "materials")


def record_env_distribution(ref):
    """InfiniteAreaLight::distribution of the reference for the environment map of tests/scenes/envmap.pbrt."""
    hs = pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "envmap.pbrt"))
    d = hs.desc.contents
    env = [d.delta_lights[i].env_tex for i in range(d.n_lights) if d.lights[i].type == pb.PB2_LIGHT_INFINITE][0]
    nu, nv, table = ref.env_distribution(d.textures[env - 1])
    np.savez_compressed(os.path.join(OUT, "env_distribution.npz"), nu=nu, nv=nv, table=table)
    print("env distribution", nu, nv)


def record_reference_digests(ref):
    """sha256 digests (tests/golden_cases.py digest) of reference outputs that tests compare bit for bit: the light
    distribution, Li samples, image and ray counts of tests/scenes/lights.pbrt under the other two light-sampling strategies,
    MIPMap::pyramid of random images of awkward sizes, and the Sobol tables (SobolMatrices32, VdCSobolMatrices /
    VdCSobolMatricesInv for every resolution from 2 to 2^25 pixels)."""
    import json
    out = {}
    for strategy in gc.LIGHT_STRATEGIES:
        hs = pb.HostScene.from_string(gc.light_strategy_scene_text(os.path.join(ROOT, "tests", "scenes"), strategy))
        rs = ref.scene(hs)
        pix, sn = gc.sample_ids(hs.film.contents.full_resolution[0], hs.film.contents.full_resolution[1],
                                hs.params.contents.samples_per_pixel, 3000, 13)
        li, _ = rs.li_samples(pix, sn)
        img, _, st = rs.render(n_threads=0)
        out["lights_" + strategy] = dict(light_distribution=gc.digest(rs.light_distribution(gc.points_for(hs.nodes(), 400, 15))),
                                         li=gc.digest(li), image=gc.digest(img),
                                         rays=[int(st.camera_rays), int(st.regular_rays), int(st.shadow_rays)])
    out["pyramids"] = {case: [[list(lv.shape), gc.digest(lv)] for lv in ref.texture_pyramid(t)] for case, t, _ in gc.pyramid_textures(pb)}
    _, mats = ref.sobol_tables(1)
    out["sobol_matrices32"] = gc.digest(mats)
    out["vdc_sobol"] = {str(m): gc.digest(ref.sobol_tables(m)[0]) for m in range(1, 26)}
    with open(os.path.join(OUT, "reference_digests.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("reference digests:", ", ".join(sorted(out)))


def main():
    ref = pyoracle.reference()
    if ref is None:
        raise SystemExit("oracle/_ref is not built: run `make -C oracle -f Makefile.ref` where /root/reference exists")
    os.makedirs(OUT, exist_ok=True)
    record_scene(ref, gc.soup_scene(pb), "soup")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "killeroo_like.pbrt")), "killeroo_like")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "materials.pbrt")), "materials")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "instances.pbrt")), "instances")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "specular.pbrt")), "specular")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "substrate.pbrt")), "substrate")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "metal.pbrt")), "metal")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "uber.pbrt")), "uber")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "roughglass.pbrt")), "roughglass")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "lights.pbrt")), "lights")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "params.pbrt")), "params")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "envlight.pbrt")), "envlight")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "textured.pbrt")), "textured")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "textured_lens.pbrt")), "textured_lens")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "sobol.pbrt")), "sobol")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "envmap.pbrt")), "envmap")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "bumpmap.pbrt")), "bumpmap")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "texcombine.pbrt")), "texcombine")
    record_scene(ref, pb.HostScene.from_file(os.path.join(ROOT, "tests", "scenes", "checker.pbrt")), "checker")
    record_texture_evaluations(ref)
    record_differentials(ref)
    record_bsdfs(ref)
    record_env_distribution(ref)
    record_textures(ref)
    record_filters(ref)
    record_hlbvh(ref)
    record_reference_digests(ref)
    # the metal material's default eta / k: copper's measured spectra through Spectrum::FromSampled (metal.cpp:121-126)
    eta, k = ref.copper_rgb()
    np.savez_compressed(os.path.join(OUT, "metal_defaults.npz"), eta=eta, k=k)
    # low-discrepancy known answers (src/tests/sampling.cpp:15-74 checks the same functions against naive versions)
    a = np.concatenate([np.arange(0, 64), np.array([1023, 65535, 1234567, 2 ** 31 + 12345, 2 ** 40 + 7, 2 ** 62 + 99])]).astype(np.uint64)
    np.savez_compressed(os.path.join(OUT, "lowdiscrepancy.npz"), a=a,
                        **{"ri_%d" % b: ref.radical_inverse(b, a) for b in (0, 1, 2, 3, 10, 50, 127, 500, 999)},
                        **{"sri_%d" % b: ref.radical_inverse(b, a, scrambled=True) for b in (0, 1, 2, 3, 10, 50, 127, 500, 999)})
    # host math: transforms, camera matrices, loop subdivision
    tr = {}
    for i, (kind, args) in enumerate([(0, [400, 20, 30, 0, 63, -110, 0, 0, 1]), (0, [0, -4.2, .6, 0, 0, 0, 0, 0, 1]), (1, [-5, 0, 0, 1]),
                                      (1, [-60, 0, 0, 1]), (1, [33, .3, -2, .7]), (2, [39, .01, 1000]), (2, [35, .01, 1000]),
                                      (3, [150, 0, 20]), (4, [.5, .5, .5])]):
        m, mi = ref.transform(kind, args)
        tr["kind_%d" % i], tr["args_%d" % i], tr["m_%d" % i], tr["minv_%d" % i] = np.int32(kind), np.array(args, np.float32), m, mi
    np.savez_compressed(os.path.join(OUT, "transforms.npz"), n=np.int32(9), **tr)
    P = np.array([[0, 0, 160], [120, 0, 40], [0, 120, 40], [-120, 0, 40], [0, -120, 40], [0, 0, -80]], np.float32)
    I = np.array([0, 1, 2, 0, 2, 3, 0, 3, 4, 0, 4, 1, 5, 2, 1, 5, 3, 2, 5, 4, 3, 5, 1, 4], np.int32)
    P2 = np.array([[-90, -90, 0], [0, -90, 30], [90, -90, 0], [-90, 0, 40], [0, 0, 110], [90, 0, 40], [-90, 90, 0], [0, 90, 30], [90, 90, 0]], np.float32)
    I2 = np.array([0, 1, 4, 0, 4, 3, 1, 2, 5, 1, 5, 4, 3, 4, 7, 3, 7, 6, 4, 5, 8, 4, 8, 7], np.int32)
    sub = {"closed_P": P, "closed_I": I, "open_P": P2, "open_I": I2}
    for tag, (pp, ii) in (("closed", (P, I)), ("open", (P2, I2))):
        for lv in (1, 2, 3):
            oP, oN, oI = ref.loop_subdivide(lv, ii, pp)
            sub["%s_%d_P" % (tag, lv)], sub["%s_%d_N" % (tag, lv)], sub["%s_%d_I" % (tag, lv)] = oP, oN, oI
    np.savez_compressed(os.path.join(OUT, "loopsubdiv.npz"), **sub)
    hs = gc.soup_scene(pb, xres=1920, yres=1080)
    r2c, dx, dy = ref.camera_derived(hs.camera, hs.film)
    np.savez_compressed(os.path.join(OUT, "camera.npz"), raster_to_camera=r2c, dx=dx, dy=dy)
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
