"""Seeded inputs shared by tests/make_golden.py (which records the reference's outputs for them) and the tests."""
import numpy as np

SOUP = dict(n_tris=2000, seed=77, jitter=0.05, xres=32, yres=18, spp=4, maxdepth=5)


def soup_scene(pb, **over):
    kw = dict(SOUP)
    kw.update(over)
    return pb.HostScene.soup(kw.pop("n_tris"), **kw)


def rays_for(pb, nodes, n, seed, shadow=False):
    rng = np.random.RandomState(seed)
    lo, hi = nodes["bmin"][0], nodes["bmax"][0]
    ext = hi - lo
    rays = np.zeros(n, pb.RAY_DTYPE)
    rays["o"] = rng.uniform(lo - 0.1 * ext, hi + 0.1 * ext, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    # a few axis-parallel directions: zero components make invDir infinite (bvh.cpp:666)
    d[: n // 50, 0] = 0
    d[n // 50: n // 25, 1:] = 0
    if shadow:
        rays["d"] = (d * 0.3 * float(ext.max())).astype(np.float32)
        rays["t_max"] = np.float32(1 - 1e-4)
    else:
        rays["d"] = d
        rays["t_max"] = np.inf
    return rays


def sample_ids(xres, yres, spp, n, seed, max_dim=None):
    rng = np.random.RandomState(seed)
    pix = np.stack([rng.randint(0, xres, n), rng.randint(0, yres, n)], 1).astype(np.int32)
    sn = rng.randint(0, spp, n).astype(np.int64)
    if max_dim is None:
        return pix, sn
    return pix, sn, rng.randint(0, max_dim, n).astype(np.int32)


def points_for(nodes, n, seed):
    rng = np.random.RandomState(seed)
    lo, hi = nodes["bmin"][0], nodes["bmax"][0]
    ext = hi - lo
    return rng.uniform(lo - 0.05 * ext, hi + 0.05 * ext, (n, 3)).astype(np.float32)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# Reconstruction filters (src/filters/): the PixelFilter line and the Film line of each case; geometry, lights and
# materials are tests/scenes/materials.pbrt's.  Wider-than-a-pixel filters make neighbouring tiles overlap in the film,
# so the order in which tiles are merged shows in the last bit: these cases are rendered by ONE thread on the CPU side.
FILTER_CASES = {
    "gaussian": ('PixelFilter "gaussian"', ""),
    "mitchell": ('PixelFilter "mitchell"', ""),
    "sinc": ('PixelFilter "sinc"', ""),
    "triangle": ('PixelFilter "triangle"', ""),
    "gaussian_aniso_crop": ('PixelFilter "gaussian" "float xwidth" [1.25] "float ywidth" [3] "float alpha" [1]',
                            ' "float cropwindow" [.2 .9 .1 .7]'),
    "mitchell_sharp": ('PixelFilter "mitchell" "float B" [0] "float C" [.5] "float xwidth" [2.5] "float ywidth" [1.5]', ""),
    "sinc_narrow": ('PixelFilter "sinc" "float xwidth" [2] "float ywidth" [3] "float tau" [2]', ""),
    "box_wide": ('PixelFilter "box" "float xwidth" [1.5] "float ywidth" [.75]', ""),
}


def filter_scene_text(scene_dir, case):
    import os
    import re
    pixel_filter, film_extra = FILTER_CASES[case]
    text = open(os.path.join(scene_dir, "materials.pbrt")).read()
    text, n = re.subn(r'Film "image"[^\n]*', 'Film "image" "integer xresolution" [40] "integer yresolution" [28]' + film_extra, text)
    assert n == 1
    text, n = re.subn(r'"integer pixelsamples" \[8\]', '"integer pixelsamples" [4]', text)
    assert n == 1
    return text.replace("WorldBegin", pixel_filter + "\nWorldBegin", 1)


def with_accelerator(text, split, maxprims, device_build=False):
    extra = ' "bool devicebuild" "true"' if device_build else ""
    return text.replace("WorldBegin", 'Accelerator "bvh" "string splitmethod" "%s" "integer maxnodeprims" [%d]%s\nWorldBegin' % (split, maxprims, extra), 1)


def random_mesh_scene_text(n_tris, seed):
    """A scene file with one trianglemesh of n_tris small random triangles inside the unit cube (for BVH-build tests)."""
    rng = np.random.RandomState(seed)
    c = rng.rand(n_tris, 1, 3).astype(np.float32)
    P = (c + 0.03 * (rng.rand(n_tris, 3, 3).astype(np.float32) - 0.5)).reshape(-1, 3)
    idx = np.arange(3 * n_tris)
    return ('LookAt .5 -2 .5  .5 .5 .5  0 0 1\nCamera "perspective" "float fov" 40\nSampler "halton" "integer pixelsamples" 1\n'
            'Film "image" "integer xresolution" 16 "integer yresolution" 16\nWorldBegin\n'
            'AttributeBegin\nAreaLightSource "diffuse" "rgb L" [5 5 5]\nShape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 2 1 0 2 0 1 2]\nAttributeEnd\n'
            'Shape "trianglemesh" "integer indices" [%s] "point P" [%s]\nWorldEnd\n'
            % (" ".join(map(str, idx)), " ".join("%.9g" % v for v in P.ravel())))


# The reference's own end-to-end tests of this path (src/tests/analytic_scenes.cpp:68-248, 270-296, 54-66): furnace scenes
# inside a unit sphere seen by a perspective camera at its centre, PathIntegrator depth 8, Halton 256 spp, 10 x 10 film;
# the average pixel value must be 1 within 0.02.
ANALYTIC_SCENES = {
    "one_point_light": 'LightSource "point" "rgb I" [3.14159265358979 3.14159265358979 3.14159265358979]\n'
                       'Material "matte" "rgb Kd" [.5 .5 .5]\n',
    "four_point_lights": 'LightSource "point" "rgb I" [.785398163397448 .785398163397448 .785398163397448]\n' * 4
                         + 'Material "matte" "rgb Kd" [.5 .5 .5]\n',
    "emissive_sphere": 'Material "matte" "rgb Kd" [.5 .5 .5]\nAreaLightSource "diffuse" "rgb L" [.5 .5 .5]\n',
    "uber_kd_kr": 'LightSource "point" "rgb I" [9.42477796076938 9.42477796076938 9.42477796076938]\n'
                  'Material "uber" "rgb Kd" [.25 .25 .25] "rgb Ks" [0 0 0] "rgb Kr" [.5 .5 .5] "rgb Kt" [0 0 0] "float roughness" 0 '
                  '"rgb opacity" [1 1 1] "float index" 1 "bool remaproughness" "false"\n',
}
ANALYTIC_EXPECTED, ANALYTIC_DELTA = 1.0, 0.02


def analytic_scene_text(case):
    return ('Camera "perspective" "float fov" 45 "float screenwindow" [-1 1 -1 1]\n'
            'Film "image" "integer xresolution" 10 "integer yresolution" 10 "float diagonal" 1\n'
            'Sampler "halton" "integer pixelsamples" 256\nIntegrator "path" "integer maxdepth" 8\nWorldBegin\n'
            + ANALYTIC_SCENES[case] + 'ReverseOrientation\nShape "sphere" "float radius" 1\nWorldEnd\n')


def sphere_reintersect_case(pb, i, partial):
    """One case of FullSphere.Reintersect / PartialSphere.Reintersect (src/tests/shapes.cpp:427-497): a sphere whose radius
    spans eight decades, rays from far-away origins (coordinates up to 1e8) into its bounding box.  Returns (scene text, rays)."""
    rng = np.random.RandomState(1000 + i)

    def pexp(e=8):   # shapes.cpp:18-25: +- 10^[-e, e]
        return (1 if rng.rand() < .5 else -1) * 10.0 ** rng.uniform(-e, e)
    radius = abs(pexp(4))
    zmin, zmax, phimax = -radius, radius, 360.0
    if partial:
        if rng.rand() >= .5:
            zmin = rng.uniform(-radius, radius)
        if rng.rand() >= .5:
            zmax = rng.uniform(-radius, radius)
        if rng.rand() >= .5:
            phimax = rng.rand() * 360
    text = ('Camera "perspective"\nFilm "image" "integer xresolution" [4] "integer yresolution" [4]\nWorldBegin\n'
            'Shape "sphere" "float radius" %.9g "float zmin" %.9g "float zmax" %.9g "float phimax" %.9g\nWorldEnd\n' % (radius, zmin, zmax, phimax))
    n = 400
    rays = np.zeros(n, pb.RAY_DTYPE)
    rays["o"] = np.array([[pexp() for _ in range(3)] for _ in range(n)], np.float32)
    lo, hi = np.float32(min(zmin, zmax)), np.float32(max(zmin, zmax))
    box_lo, box_hi = np.array([-radius, -radius, lo], np.float32), np.array([radius, radius, hi], np.float32)
    target = (box_lo + rng.rand(n, 3).astype(np.float32) * (box_hi - box_lo)).astype(np.float32)
    d = target - rays["o"]
    norm = rng.rand(n) < .5
    d[norm] /= np.linalg.norm(d[norm], axis=1, keepdims=True)
    rays["d"] = d
    rays["t_max"] = np.inf
    return text, rays, rng


def spawned_rays(pb, hits, rng):
    """Interaction::SpawnRay (interaction.h:64-67, OffsetRayOrigin geometry.h:1440-1454) in a random direction on the
    normal's side of every hit."""
    n = len(hits)
    w = rng.normal(size=(n, 3)).astype(np.float32)
    w /= np.linalg.norm(w, axis=1, keepdims=True)
    nrm, p, pe = hits["n"], hits["p"], hits["p_error"]
    w[(w * nrm).sum(axis=1) < 0] *= -1                     # Faceforward(w, isect.n)
    d = (np.abs(nrm) * pe).sum(axis=1, keepdims=True)
    off = (d * nrm).astype(np.float32)
    po = (p + off).astype(np.float32)
    up, dn = off > 0, off < 0
    po[up] = np.nextafter(po[up], np.float32(np.inf))
    po[dn] = np.nextafter(po[dn], np.float32(-np.inf))
    rays = np.zeros(n, pb.RAY_DTYPE)
    rays["o"], rays["d"], rays["t_max"] = po, w, np.inf
    return rays


def texture_lookup_inputs(n, seed):
    """(st, dst) batches for MIPMap::Lookup: footprints from none at all to several times the whole image, isotropic
    and up to 60 : 1 anisotropic (beyond every maxanisotropy in use), one derivative zero, st outside [0, 1] for the wrap modes."""
    rs = np.random.RandomState(seed)
    st = rs.uniform(-0.6, 1.6, (n, 2)).astype(np.float32)
    kind = rs.randint(0, 7, n)
    size = np.exp(rs.uniform(np.log(1e-4), np.log(3.0), n))
    ang = rs.uniform(0, 2 * np.pi, n)
    ratio = np.exp(rs.uniform(0, np.log(60.0), n))
    d0 = np.stack([np.cos(ang), np.sin(ang)], 1) * size[:, None]
    ang1 = ang + np.where(kind == 5, rs.uniform(0, np.pi, n), np.pi / 2)   # kind 5: not orthogonal
    d1 = np.stack([np.cos(ang1), np.sin(ang1)], 1) * (size / ratio)[:, None]
    d1[kind == 1] = d0[kind == 1][:, ::-1] * [1, -1]    # isotropic
    d0[kind == 0] = 0                                  # no differentials at all
    d1[kind == 0] = 0
    d1[kind == 2] = 0                                  # one derivative zero
    swap = kind == 3                                   # the second one is the longer
    d0[swap], d1[swap] = d1[swap].copy(), d0[swap].copy()
    exact = kind == 6                                  # footprints of exactly 2^-k texture widths
    d0[exact] = np.stack([2.0 ** -rs.randint(0, 8, exact.sum()), np.zeros(exact.sum())], 1)
    d1[exact] = d0[exact][:, ::-1]
    return st, np.concatenate([d0, d1], 1).astype(np.float32)


TEXTURE_EVAL_SCENES = ("textured", "texcombine", "checker")


def texture_eval_inputs(n, seed):
    """(u, v) in [-1, 3]^2 and (dudx, dvdx, dudy, dvdy) from 1e-4 to 0.7, every fifth point without differentials."""
    rs = np.random.RandomState(seed)
    uv = rs.uniform(-1, 3, (n, 2)).astype(np.float32)
    mag = np.exp(rs.uniform(np.log(1e-4), np.log(.7), (n, 1)))
    duv = (rs.normal(size=(n, 4)) * mag).astype(np.float32)
    duv[::5] = 0
    return uv, duv

DIFFERENTIAL_SCENES = ("textured", "textured_lens", "bumpmap", "instances")


BSDF_SCENES = ("materials", "specular", "substrate", "metal", "uber", "roughglass")


def bsdf_frames(n, seed):
    """Random shading frames for BSDF evaluation: geometric normal, a shading normal near it (a third of them equal), a shading
    dpdu (a quarter of them not perpendicular to ns), wo and wi anywhere on the sphere, a 2D sample."""
    rs = np.random.RandomState(seed)

    def unit(v):
        return v / np.linalg.norm(v, axis=1, keepdims=True)
    nrm = unit(rs.normal(size=(n, 3)))
    ns = unit(nrm + 0.3 * rs.normal(size=(n, 3)))
    ns[::3] = nrm[::3]
    t = rs.normal(size=(n, 3))
    dpdu = (t - ns * (t * ns).sum(1, keepdims=True)) * rs.uniform(.2, 3, (n, 1))
    dpdu[::4] += 0.2 * ns[::4]
    wo, wi = unit(rs.normal(size=(n, 3))), unit(rs.normal(size=(n, 3)))
    return np.ascontiguousarray(np.concatenate([nrm, ns, dpdu, wo, wi, rs.uniform(0, 1, (n, 2))], 1), np.float32)


def digest(a):
    """sha256 of an array's bytes: what tests/golden/reference_digests.json stores where the test asks for every bit."""
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


LIGHT_STRATEGIES = ("spatial", "uniform")


def light_strategy_scene_text(scenes_dir, strategy):
    """tests/scenes/lights.pbrt with another "lightsamplestrategy" than its "power"."""
    import os
    text = open(os.path.join(scenes_dir, "lights.pbrt")).read()
    return text.replace('"string lightsamplestrategy" "power"', '"string lightsamplestrategy" "%s"' % strategy)


PYRAMID_CASES = [(1, 1, 1, 0), (1, 7, 3, 0), (5, 1, 1, 2), (13, 31, 3, 1), (16, 4, 1, 0), (33, 64, 3, 2), (100, 3, 1, 1)]   # w, h, channels, wrap


def pyramid_textures(pb):
    """Random images of awkward sizes (1 x N, N x 1, primes, already a power of two) as pb2_textures: (case, texture, texels);
    the texels array must outlive the texture."""
    import ctypes as C
    rs = np.random.RandomState(9)
    for (w, h, ch, wrap) in PYRAMID_CASES:
        texels = rs.uniform(0, 2, (h, w, ch)).astype(np.float32)
        t = pb.Texture(channels=ch, width=w, height=h, wrap=wrap, do_trilinear=0, max_anisotropy=8.0, su=1, sv=1, du=0, dv=0,
                       texels=texels.ctypes.data_as(C.POINTER(C.c_float)))
        yield "%dx%dx%d_wrap%d" % (w, h, ch, wrap), t, texels
