"""Mutated fixture scenes for the GPU-vs-oracle fuzz (tests/test_gpu_parity.py, tools/gpu_fuzz.py): stored fixture
scenes with random motion flags, BRDF models, roughness, reflective materials, glossy flags and settings, and random scenes
no builder of the reference ever produced.  The CPU twin (tests/test_oracle_fuzz.py) pins the oracle on the compiled
reference for the same mutations and the same random scenes."""
import numpy as np

from conftest import GOLDEN_CASES, load_case


def mutated_case(seed):
    """-> (fixture name, Scene, settings); deterministic in `seed`."""
    from distraytracer_b200 import abi
    from distraytracer_b200.scene import Scene
    rng = np.random.default_rng(9000 + seed)
    case = GOLDEN_CASES[int(rng.integers(len(GOLDEN_CASES)))]
    scene, settings, _ = load_case(case)
    s = abi.copy_struct(settings)
    s.xRes, s.yRes = int(rng.integers(24, 65)), int(rng.integers(18, 49))
    s.antialias_samples = int(rng.choice([1, 4, 9]))
    s.aperture = float(rng.choice([0.0, 0.2]))
    s.brdf_samples = int(rng.integers(1, 4))
    s.max_depth = int(rng.integers(1, 7))
    s.blur_samples = int(rng.integers(0, 4))
    s.frame_range = int(rng.integers(1, 9))
    if rng.random() < 0.4:
        s.frame_prism, s.frame_blur = 0, int(rng.choice([0, 100000]))
    s.seed = int(rng.integers(1, 1 << 30))
    prims = [abi.copy_struct(p) for p in scene.prims]
    for p in prims:
        if p.flags & abi.FLAG_LIGHT:
            continue
        if rng.random() < 0.3:
            p.flags ^= abi.FLAG_MOTION
        if rng.random() < 0.5:
            p.model = int(rng.choice([abi.MODEL_LAMBERT, abi.MODEL_OREN_NAYAR, abi.MODEL_COOK_TORRANCE]))
            p.roughness = float(np.float32(rng.uniform(0.1, 0.9)))
            p.refr[0], p.refr[1] = 0.958, 6.69
        if rng.random() < 0.3:
            p.material = int(rng.choice([abi.MAT_NONE, abi.MAT_STEEL, abi.MAT_ALUMINUM, abi.MAT_LINOLEUM]))
            if rng.random() < 0.5:
                p.flags ^= abi.FLAG_GLOSSY
    return case, Scene(prims, scene.lights, scene.textures), s


def random_scene(seed):
    """A scene the reference never built: random spheres, cylinders, triangles, rectangles (corners in any order, so some
    are the diagonal kind) and checkerboards around the origin, random materials / models, one to three lights."""
    import numpy as np
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    rng = np.random.default_rng(55000 + seed)
    base, settings, _ = load_case("checkertexture")
    P = lambda s=3.0: rng.uniform(-s, s, 3)
    col = lambda: tuple(rng.uniform(0.2, 1.0, 3))
    mat = lambda: int(rng.choice([abi.MAT_NONE, abi.MAT_NONE, abi.MAT_STEEL, abi.MAT_ALUMINUM]))
    mod = lambda: int(rng.choice([abi.MODEL_LAMBERT, abi.MODEL_OREN_NAYAR, abi.MODEL_COOK_TORRANCE]))
    prims = []
    for _ in range(int(rng.integers(3, 14))):
        kind = int(rng.integers(5))
        if kind == 0:
            p = scenes.sphere(P(), float(rng.uniform(0.2, 1.2)), col(), material=mat(), model=mod())
        elif kind == 1:
            a = P(); p = scenes.cylinder(a, a + rng.normal(0, 1.0, 3), float(rng.uniform(0.1, 0.5)), col(), material=mat(), model=mod())
        elif kind == 2:
            a = P(); p = scenes.triangle(a, a + rng.normal(0, 1.5, 3), a + rng.normal(0, 1.5, 3), col(), material=mat(), model=mod())
        else:
            a = P(4.0); u = rng.normal(0, 2.0, 3); v = np.cross(u, rng.normal(0, 1, 3)); v *= float(rng.uniform(0.5, 3.0)) / max(np.linalg.norm(v), 1e-9)
            corners = [a, a + u, a + u + v, a + v]
            if rng.random() < 0.35:
                corners = [corners[i] for i in rng.permutation(4)]       # any corner order: the reference takes what it is given
            if kind == 3:
                p = scenes.rectangle(*corners, col(), material=mat(), model=mod(), name=int(rng.choice([abi.NAME_RECTANGLE, abi.NAME_OTHER])))
            else:
                p = scenes.checkerboard(*corners, col(), col(), float(rng.uniform(0.2, 1.0)), material=mat(), model=mod())
        p.roughness = float(np.float32(rng.uniform(0.1, 0.9))); p.refr[0], p.refr[1] = 0.958, 6.69
        if rng.random() < 0.3: p.flags |= abi.FLAG_GLOSSY
        prims.append(p)
    lights = []
    for _ in range(int(rng.integers(1, 4))):
        kind = int(rng.integers(3))
        if kind == 0:
            lights.append(scenes.point_light(P(6.0) + np.array([0, 4, 0]), col()))
        elif kind == 1:
            a = P(3.0) + np.array([0, 5, 0]); u = np.array([float(rng.uniform(0.5, 2)), 0, 0]); v = np.array([0, 0, float(rng.uniform(0.5, 2))])
            lp, ll = scenes.rectangle_light(a, a + u, a + u + v, a + v, col(), len(prims)); prims.append(lp); lights.append(ll)
        else:
            lp, ll = scenes.sphere_light(P(4.0) + np.array([0, 5, 0]), float(rng.uniform(0.2, 0.8)), col(), len(prims)); prims.append(lp); lights.append(ll)
    s = abi.copy_struct(settings)
    s.xRes, s.yRes = int(rng.integers(24, 65)), int(rng.integers(18, 49))
    s.antialias_samples = int(rng.choice([1, 4, 9])); s.aperture = float(rng.choice([0.0, 0.2]))
    s.brdf_samples = int(rng.integers(1, 4)); s.max_depth = int(rng.integers(1, 6)); s.blur_samples = 0
    s.seed = int(rng.integers(1, 1 << 30))
    v = rng.normal(0, 1, 3); v /= np.linalg.norm(v)
    eye = v * float(rng.uniform(5, 9)); eye[1] = abs(eye[1]) * 0.6
    s.eye[:] = [float(x) for x in eye]; s.lookingAt[:] = [float(x) for x in rng.uniform(-0.5, 0.5, 3)]; s.up[:] = [0, 1, 0]
    s.focal_length = float(np.linalg.norm(eye))
    return "random_scene", Scene(prims, lights, base.textures), s


def random_mesh_scene(seed):
    """A random triangle mesh (a bumpy grid with random holes, or a soup of random triangles; 40 to ~2000 triangles, with
    texcoords and, half of the time, a per-triangle material table) plus a sphere or two, one or two lights, depth of
    field.  -> (name, Scene with the mesh -- what the CUDA path takes, through its device-built 4-wide LBVH --, the same
    scene with the triangles as Triangle primitives -- what the oracle's reference-order walk takes --, settings)."""
    import numpy as np
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    rng = np.random.default_rng(66000 + seed)
    base, settings, _ = load_case("checkertexture")
    if rng.random() < 0.6:
        n = int(rng.integers(6, 33))
        mesh = scenes.terrain_mesh(n, size=float(rng.uniform(3, 10)), height=float(rng.uniform(0.2, 2.0)))
        keep = rng.random(len(mesh["indices"])) > float(rng.uniform(0.0, 0.3))
        mesh["indices"] = np.ascontiguousarray(mesh["indices"][keep])
    else:
        nt = int(rng.integers(40, 400))
        a = rng.uniform(-4, 4, (nt, 1, 3)); a[:, :, 1] *= 0.3
        verts = (a + rng.normal(0, float(rng.uniform(0.2, 1.0)), (nt, 3, 3))).reshape(-1, 3).astype(np.float32)
        mesh = {"vertices": verts, "indices": np.arange(3 * nt, dtype=np.int32).reshape(nt, 3),
                "texcoords": rng.uniform(0, 1, (3 * nt, 2)).astype(np.float32)}
    textured = rng.random() < 0.5
    mesh["material"] = scenes.mesh_material(tex_frame=2 if textured else -1,
                                            model=int(rng.choice([abi.MODEL_LAMBERT, abi.MODEL_OREN_NAYAR, abi.MODEL_COOK_TORRANCE])),
                                            roughness=float(rng.uniform(0.2, 0.8)))
    mesh["material"].refr[0], mesh["material"].refr[1] = 0.958, 6.69
    if rng.random() < 0.5:
        mats = []
        for v in rng.uniform(0.1, 0.9, 5):
            m = abi.copy_struct(mesh["material"]); m.roughness = float(np.float32(v)); m.color[0] = float(v); mats.append(m)
        mesh["materials"] = mats
        mesh["material_ids"] = rng.integers(0, 5, len(mesh["indices"])).astype(np.int32)
    prims = [scenes.sphere(rng.uniform(-2, 2, 3) + np.array([0, 1.5, 0]), float(rng.uniform(0.3, 0.9)), tuple(rng.uniform(0.2, 1, 3)),
                           material=int(rng.choice([abi.MAT_NONE, abi.MAT_STEEL])))]
    if rng.random() < 0.5:
        prims.append(scenes.rectangle((-6, -1.5, 6), (6, -1.5, 6), (6, -1.5, -6), (-6, -1.5, -6), (0.6, 0.6, 0.6), name=abi.NAME_OTHER))
    lights = [scenes.point_light(rng.uniform(-5, 5, 3) + np.array([0, 7, 0]), (1.0, 1.0, 1.0))]
    if rng.random() < 0.5:
        lp, ll = scenes.sphere_light(rng.uniform(-3, 3, 3) + np.array([0, 6, 0]), 0.5, (0.8, 0.8, 1.0), len(prims))
        prims.append(lp); lights.append(ll)
    s = abi.copy_struct(settings)
    s.xRes, s.yRes = int(rng.integers(24, 65)), int(rng.integers(18, 49))
    s.antialias_samples = int(rng.choice([1, 4])); s.aperture = float(rng.choice([0.0, 0.2]))
    s.brdf_samples = int(rng.integers(1, 3)); s.max_depth = int(rng.integers(1, 5)); s.blur_samples = 0
    s.seed = int(rng.integers(1, 1 << 30))
    v = rng.normal(0, 1, 3); v /= np.linalg.norm(v)
    eye = v * float(rng.uniform(6, 11)); eye[1] = abs(eye[1]) * 0.7 + 1.0
    s.eye[:] = [float(x) for x in eye]; s.lookingAt[:] = [0.0, 0.0, 0.0]; s.up[:] = [0, 1, 0]
    s.focal_length = float(np.linalg.norm(eye))
    with_mesh = Scene(prims, lights, base.textures, mesh=mesh)
    flat = Scene(list(prims) + scenes.mesh_to_prims(mesh), lights, base.textures)
    return "random_mesh", with_mesh, flat, s


def random_motion_scene(seed):
    """random_scene with the library's own blur mode (DRT_BLUR_VELOCITY, SURVEY 8(f)1: the reference has no counterpart, the
    oracle twin is the checker): random velocities on flagged primitives, cylinders partly with two-pose end points."""
    import numpy as np
    from distraytracer_b200 import abi
    from distraytracer_b200.scene import Scene
    case, scene, s = random_scene(seed)
    rng = np.random.default_rng(88000 + seed)
    prims = [abi.copy_struct(p) for p in scene.prims]
    for p in prims:
        if (p.flags & abi.FLAG_LIGHT) or rng.random() < 0.5:
            continue
        p.flags |= abi.FLAG_MOTION
        v = rng.normal(0, 0.6, 3)
        p.velocity[0], p.velocity[1], p.velocity[2] = (float(x) for x in v)
        if p.type == abi.PRIM_CYLINDER and rng.random() < 0.6:
            p.flags |= abi.FLAG_VERTEX_MOTION
            w = rng.normal(0, 0.6, 3)
            p.velocity2[0], p.velocity2[1], p.velocity2[2] = (float(x) for x in w)
    s.blur_mode, s.blur_samples, s.frame_range = abi.BLUR_VELOCITY, int(rng.integers(1, 4)), 1
    return "random_motion", Scene(prims, scene.lights, scene.textures), s


def random_big_scene(seed):
    """More analytic shapes than the CUDA path's shared-memory filter table holds (257 .. 700): small spheres, cylinders and
    rectangles scattered over a floor -- the CUDA path gathers through its 4-wide tree over the geoms."""
    import numpy as np
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    rng = np.random.default_rng(99000 + seed)
    base, settings, _ = load_case("checkertexture")
    prims = [scenes.rectangle((-9, 0, 9), (9, 0, 9), (9, 0, -9), (-9, 0, -9), (0.7, 0.7, 0.7),
                              material=int(rng.choice([abi.MAT_NONE, abi.MAT_STEEL])), name=abi.NAME_OTHER)]
    for _ in range(int(rng.integers(257, 700))):
        c = rng.uniform(-8, 8, 3); c[1] = float(rng.uniform(0.1, 2.5))
        col = tuple(rng.uniform(0.2, 1.0, 3))
        kind = int(rng.integers(3))
        if kind == 0:
            prims.append(scenes.sphere(c, float(rng.uniform(0.08, 0.35)), col, material=int(rng.choice([abi.MAT_NONE, abi.MAT_NONE, abi.MAT_STEEL]))))
        elif kind == 1:
            prims.append(scenes.cylinder(c, c + rng.normal(0, 0.4, 3), float(rng.uniform(0.05, 0.15)), col))
        else:
            u = rng.normal(0, 0.4, 3); v = np.cross(u, rng.normal(0, 1, 3)); v *= 0.4 / max(np.linalg.norm(v), 1e-9)
            prims.append(scenes.rectangle(c, c + u, c + u + v, c + v, col, name=abi.NAME_OTHER))
    lp, ll = scenes.rectangle_light((-1, 6, -1), (1, 6, -1), (1, 6, 1), (-1, 6, 1), (1.0, 1.0, 0.9), len(prims))
    prims.append(lp)
    lights = [ll, scenes.point_light(rng.uniform(-6, 6, 3) + np.array([0, 8, 0]), (0.7, 0.7, 0.7))]
    s = abi.copy_struct(settings)
    s.xRes, s.yRes = int(rng.integers(24, 65)), int(rng.integers(18, 49))
    s.antialias_samples = int(rng.choice([1, 4])); s.aperture = float(rng.choice([0.0, 0.2]))
    s.brdf_samples = int(rng.integers(1, 3)); s.max_depth = int(rng.integers(1, 5)); s.blur_samples = 0
    s.seed = int(rng.integers(1, 1 << 30))
    v = rng.normal(0, 1, 3); v /= np.linalg.norm(v)
    eye = v * float(rng.uniform(7, 14)); eye[1] = abs(eye[1]) * 0.6 + 1.5
    s.eye[:] = [float(x) for x in eye]; s.lookingAt[:] = [0.0, 0.5, 0.0]; s.up[:] = [0, 1, 0]
    s.focal_length = float(np.linalg.norm(eye))
    return "random_big", Scene(prims, lights, base.textures), s


def sky_case(seed):
    """mutated_case with the value-noise cloud background switched on (perlin_cloud: cloud_corners + the per-sample corner
    offsets) at a small size -- the oracle marches 200 noise steps per pixel corner."""
    case, scene, s = mutated_case(seed)
    s.perlin_cloud = 1
    s.xRes, s.yRes = min(s.xRes, 40), min(s.yRes, 28)
    return case + "+sky", scene, s


def random_moving_mesh_scene(seed):
    """random_mesh_scene in velocity-blur mode with the MESH in motion (DRT_BLUR_VELOCITY moves a mesh as a whole by its
    materials' common velocity) and, half of the time, the sphere too."""
    import numpy as np
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    case, with_mesh, flat, s = random_mesh_scene(seed)
    rng = np.random.default_rng(44000 + seed)
    vel = rng.normal(0, 0.5, 3)
    mesh = dict(with_mesh.mesh)
    def move(m):
        m = abi.copy_struct(m); m.flags |= abi.FLAG_MOTION
        m.velocity[0], m.velocity[1], m.velocity[2] = (float(x) for x in vel)
        return m
    mesh["material"] = move(mesh["material"])
    if mesh.get("materials"):
        mesh["materials"] = [move(m) for m in mesh["materials"]]
    prims = [abi.copy_struct(p) for p in with_mesh.prims]
    if rng.random() < 0.5:
        prims[0].flags |= abi.FLAG_MOTION
        w = rng.normal(0, 0.5, 3); prims[0].velocity[0], prims[0].velocity[1], prims[0].velocity[2] = (float(x) for x in w)
    s.blur_mode, s.blur_samples, s.frame_range = abi.BLUR_VELOCITY, int(rng.integers(1, 4)), 1
    return ("random_moving_mesh", Scene(prims, with_mesh.lights, with_mesh.textures, mesh=mesh),
            Scene(list(prims) + scenes.mesh_to_prims(mesh), with_mesh.lights, with_mesh.textures), s)


def random_prism_scene(seed):
    """The slab-box prism classes (RectPrism / RectPrismWithCylinder / RectPrismWithHoles, SURVEY 8a a14) with random
    extents and random holes (spheres and cylinders, inside, across and outside the box), over a floor, next to a sphere,
    under random lights, seen from anywhere -- including from inside the prism."""
    import numpy as np
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    rng = np.random.default_rng(33000 + seed)
    base, settings, _ = load_case("checkertexture")
    prims = [scenes.rectangle((-6, -2.2, -6), (8, -2.2, -6), (8, -2.2, 6), (-6, -2.2, 6), (0.7, 0.7, 0.7), name=abi.NAME_OTHER),
             scenes.sphere((3.0, 0.0, 2.6), 0.8, (0.2, 0.9, 0.3), material=int(rng.choice([abi.MAT_NONE, abi.MAT_STEEL])))]
    for _ in range(int(rng.integers(1, 3))):
        kind = int(rng.choice([abi.PRIM_RECTPRISM, abi.PRIM_RECTPRISM_CYL, abi.PRIM_RECTPRISM_HOLES]))
        lo = rng.uniform(-3, 1, 3); hi = lo + rng.uniform(0.6, 3.5, 3)
        p = scenes.new_prim(); p.type = kind
        A = np.array([lo[0], lo[1], lo[2]]); B = np.array([lo[0], lo[1], hi[2]]); C = np.array([lo[0], hi[1], hi[2]]); D = np.array([lo[0], hi[1], lo[2]])
        back = np.array([hi[0] - lo[0], 0, 0])
        for dst, v in zip((p.A, p.B, p.C, p.D, p.E, p.F, p.G, p.H), (A, B, C, D, A + back, B + back, C + back, D + back)):
            dst[:] = list(v)
        p.color[:] = list(rng.uniform(0.2, 1.0, 3)); p.center[:] = list((lo + hi) / 2)
        p.material = int(rng.choice([abi.MAT_NONE, abi.MAT_NONE, abi.MAT_STEEL]))
        p.model = int(rng.choice([abi.MODEL_LAMBERT, abi.MODEL_OREN_NAYAR])); p.roughness = float(np.float32(rng.uniform(0.2, 0.8)))
        if kind != abi.PRIM_RECTPRISM:
            p.n_holes = int(rng.integers(1, 4))
            for k in range(p.n_holes):
                sph = kind == abi.PRIM_RECTPRISM_HOLES and rng.random() < 0.5
                c1 = rng.uniform(lo - 0.5, hi + 0.5)
                p.holes[k].type = abi.PRIM_SPHERE if sph else abi.PRIM_CYLINDER
                p.holes[k].c1[:] = list(c1); p.holes[k].c2[:] = list(c1 + rng.normal(0, 1.2, 3))
                p.holes[k].radius = float(np.float32(rng.uniform(0.2, 1.0))); p.holes[k].color[:] = list(rng.uniform(0, 1, 3))
        prims.append(p)
    lights = [scenes.point_light(rng.uniform(-6, 6, 3) + np.array([0, 5, 0]), (1, 1, 1))]
    if rng.random() < 0.5:
        lights.append(scenes.point_light(rng.uniform(-6, 6, 3) + np.array([0, 4, 0]), (0.6, 0.6, 0.9)))
    s = abi.copy_struct(settings)
    s.xRes, s.yRes = int(rng.integers(24, 65)), int(rng.integers(18, 49))
    s.antialias_samples = int(rng.choice([1, 4])); s.aperture = float(rng.choice([0.0, 0.2]))
    s.brdf_samples = int(rng.integers(1, 3)); s.max_depth = int(rng.integers(1, 5)); s.blur_samples = 0
    s.seed = int(rng.integers(1, 1 << 30))
    v = rng.normal(0, 1, 3); v /= np.linalg.norm(v)
    eye = v * float(rng.uniform(0.5, 9)); eye[1] = abs(eye[1]) * 0.7
    s.eye[:] = [float(x) for x in eye]; s.lookingAt[:] = [float(x) for x in rng.uniform(-1, 1, 3)]; s.up[:] = [0, 1, 0]
    s.focal_length = float(max(np.linalg.norm(eye), 1.0))
    return "random_prism", Scene(prims, lights, base.textures), s


def random_glass_scene(seed):
    """random_scene plus one or two closed blocks of glass triangles (the reference's refraction path is only reachable on
    `mesh` triangles): Fresnel split, total internal reflection, rays starting inside the glass."""
    import numpy as np
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    case, scene, s = random_scene(seed)
    rng = np.random.default_rng(22000 + seed)
    prims = [abi.copy_struct(p) for p in scene.prims]
    lights = [abi.copy_struct(l) for l in scene.lights]
    extra = []
    for _ in range(int(rng.integers(1, 3))):
        lo = rng.uniform(-2.5, 1.5, 3); hi = lo + rng.uniform(0.5, 2.0, 3)
        extra.extend(scenes.glass_block(lo, hi))
    # area lights point at their shapes by index: the blocks go in front, the indices move up
    for l in lights:
        if l.prim_index >= 0: l.prim_index += len(extra)
    s.max_depth = int(rng.integers(2, 8))
    return "random_glass", Scene(extra + prims, lights, scene.textures), s


# ---- sized scenes: the same picture with more or fewer scene records -------------------------------------------------
# render_wave's launcher picks its instantiation by scene size (csrc/drt_launch.h): more than SMEM_GEOMS geoms sets FT_BIG
# (the geom tree, or the global slab table when a slab-box prism is present), and records of more than SMEM_RECS bytes are
# read from global memory instead of the CTA's shared copy (no FT_RECS).  Bytes of one Geom<R>, PrimD<R>, LightD<R> record
# per precision (drt_settings.precision: 0 double, 1 float); a mesh's material table adds one PrimD per entry.
SMEM_GEOMS, SMEM_RECS = 256, 32 * 1024
RECORD_BYTES = {0: (224, 1280, 160), 1: (160, 784, 96)}
SIZED_KINDS = ("scene", "textured", "motion", "glass", "refblur", "prism", "mesh", "moving_mesh")
ENCLOSURE_CENTER, ENCLOSURE_RADIUS = (24.0, 1.0, 0.0), 3.0


def geom_count(prims):
    """Geoms flatten (csrc/drt_api.cu) makes of `prims`: one per primitive, two for a checkerboard with a hole (board and
    hole), six for a RectPrismV2 (its faces)."""
    from distraytracer_b200 import abi
    return sum(2 if p.type == abi.PRIM_CHECKERBOARD_HOLE else 6 if p.type == abi.PRIM_RECTPRISMV2 else 1 for p in prims)


def mesh_materials(scene):
    """Entries of the mesh's material table (0 without a mesh; 1 when every triangle takes drt_mesh.material)."""
    if scene.mesh is None:
        return 0
    return len(scene.mesh.get("materials") or []) or 1


def record_bytes(scene, precision):
    """Bytes of the geom, primitive and light records render_wave stages in shared memory when they fit."""
    g, p, l = RECORD_BYTES[precision]
    return g * geom_count(scene.prims) + p * (len(scene.prims) + mesh_materials(scene)) + l * len(scene.lights)


def _filler(rng, geoms):
    """One small opaque shape of `geoms` geoms (1: sphere, cylinder, rectangle or triangle; 2: checkerboard with a hole;
    6: RectPrismV2) somewhere inside the enclosing sphere."""
    from distraytracer_b200 import abi, scenes
    c = np.asarray(ENCLOSURE_CENTER) + rng.uniform(-0.35, 0.35, 3) * ENCLOSURE_RADIUS
    col = tuple(rng.uniform(0.2, 1.0, 3))
    s = float(rng.uniform(0.05, 0.2))
    if geoms == 1:
        kind = int(rng.integers(4))
        if kind == 0:
            return scenes.sphere(c, s, col)
        if kind == 1:
            return scenes.cylinder(c, c + rng.normal(0, s, 3), 0.3 * s, col)
        if kind == 2:
            return scenes.triangle(c, c + rng.normal(0, s, 3), c + rng.normal(0, s, 3), col)
        return scenes.rectangle(c, c + (s, 0, 0), c + (s, s, 0), c + (0, s, 0), col, name=abi.NAME_OTHER)
    if geoms == 2:
        p = scenes.checkerboard(c, c + (0, 0, s), c + (s, 0, s), c + (s, 0, 0), col, (0.1, 0.1, 0.1), 0.05)
        p.type = abi.PRIM_CHECKERBOARD_HOLE
        q = 0.25 * s
        for dst, v in zip(p.hole, (c + (q, 0, q), c + (q, 0, 3 * q), c + (3 * q, 0, 3 * q), c + (3 * q, 0, q))):
            dst[:] = list(v)
        return p
    assert geoms == 6
    p = scenes.new_prim(); p.type = abi.PRIM_RECTPRISMV2
    A, B, C, D = c, c + (0, 0, s), c + (0, s, s), c + (0, s, 0)
    for dst, v in zip((p.A, p.B, p.C, p.D, p.E, p.F, p.G, p.H), (A, B, C, D, A + (s, 0, 0), B + (s, 0, 0), C + (s, 0, 0), D + (s, 0, 0))):
        dst[:] = list(v)
    p.color[:] = list(col); p.center[:] = list(c + 0.5 * s)
    return p


def _base(kind, seed):
    """-> (name, scene for the CUDA path, the same with the mesh as Triangle primitives or None, settings)."""
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    flat = None
    if kind in ("scene", "textured"):
        name, scene, s = random_scene(seed)
        if kind == "textured":              # a textured floor under the shapes (FT_TEX)
            floor = scenes.rectangle((-8, -3.5, 8), (8, -3.5, 8), (8, -3.5, -8), (-8, -3.5, -8), (0.7, 0.7, 0.7),
                                     tex_frame=0, name=abi.NAME_OTHER)
            floor.flags |= abi.FLAG_TEXTURE
            scene = Scene(scene.prims + [floor], scene.lights, scene.textures)
    elif kind == "motion":
        name, scene, s = random_motion_scene(seed)
    elif kind == "glass":
        name, scene, s = random_glass_scene(seed)
    elif kind == "refblur":
        name, scene, s = random_refblur_scene(seed)
    elif kind == "prism":
        name, scene, s = random_prism_scene(seed)
    elif kind == "mesh":
        name, scene, flat, s = random_mesh_scene(seed)
    else:
        assert kind == "moving_mesh", kind
        name, scene, flat, s = random_moving_mesh_scene(seed)
    return name, scene, flat, s


def sized_scene(kind, seed, precision=0, geoms=None, recs=None, recs_at_most=False, extra_materials=0, frame_range=None,
                twins=False):
    """A base scene drawn like random_scene / random_mesh_scene / ... (`kind`, one of SIZED_KINDS) plus an opaque enclosing
    sphere on the +x side, far from the camera and the shapes, and "filler": small shapes inside that sphere.  No camera,
    reflection, refraction or shadow ray reaches the filler (each one crosses the sphere first), so the filler changes the
    scene's tables but not its picture.  The filler goes after every other primitive (area lights keep their prim_index);
    in the reference's candidate order it comes first, so the base scene's geoms keep the end of the slab table.

    geoms: add 1-geom filler up to that many geoms in all.  recs: add filler (spheres, checkerboards with a hole, RectPrismV2)
    up to exactly that many record bytes in `precision` (recs_at_most: the most the filler can make without exceeding
    `recs`; the byte counts it can add are combinations of three record sizes).  extra_materials: entries appended to the
    mesh's material table, which no triangle uses.  frame_range: override (velocity blur: 1 keeps the swept boxes, more re-traces unfiltered).
    twins: every rectangle and triangle of the base gets a coplanar copy of another colour, appended (exact ties of t: the
    first in the reference's candidate order must win).
    -> (name, scene, flat, settings); `flat` is the scene the oracle takes (mesh triangles as Triangle primitives)."""
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    name, scene, flat, s = _base(kind, seed)
    rng = np.random.default_rng(123000 + seed)
    s.xRes, s.yRes = min(s.xRes, 64), min(s.yRes, 48)
    s.antialias_samples = min(s.antialias_samples, 4)
    if frame_range is not None:
        s.frame_range = frame_range
    prims = [abi.copy_struct(p) for p in scene.prims]
    if twins:
        for p in scene.prims:
            if p.type in (abi.PRIM_RECTANGLE, abi.PRIM_TRIANGLE) and not (p.flags & abi.FLAG_LIGHT):
                q = abi.copy_struct(p); q.color[:] = [1.0 - x for x in p.color]; prims.append(q)
    prims.append(scenes.sphere(ENCLOSURE_CENTER, ENCLOSURE_RADIUS, (0.55, 0.5, 0.45)))
    mesh = dict(scene.mesh) if scene.mesh is not None else None
    if extra_materials:
        assert mesh is not None, "extra_materials needs a mesh"
        mats = list(mesh.get("materials") or [mesh["material"]])
        if not mesh.get("materials"):
            mesh["material_ids"] = np.zeros(len(mesh["indices"]), dtype=np.int32)
        mesh["materials"] = mats + [abi.copy_struct(mats[0]) for _ in range(extra_materials)]
    def sized(extra):
        return Scene(prims + extra, scene.lights, scene.textures, mesh=mesh)
    extra = []
    if geoms is not None:
        n = geoms - geom_count(prims)
        assert n >= 0, (kind, seed, "base scene has more geoms than", geoms)
        extra = [_filler(rng, 1) for _ in range(n)]
    if recs is not None:
        G, P, _ = RECORD_BYTES[precision]
        base = record_bytes(sized([]), precision)
        plan = None
        for target in range(recs, base - 1, -16) if recs_at_most else (recs,):
            need = target - base
            plan = next(((n1, n2, n6) for n6 in range(12) for n2 in range(5)
                         for n1 in [(need - n6 * (6 * G + P) - n2 * (2 * G + P)) // (G + P)]
                         if n1 >= 0 and n1 * (G + P) + n2 * (2 * G + P) + n6 * (6 * G + P) == need), None)
            if plan is not None:
                break
        assert plan is not None, (kind, seed, "no filler makes", recs, "record bytes from", base)
        extra += [_filler(rng, g) for g, k in zip((1, 2, 6), plan) for _ in range(k)]
    out = sized(extra)
    if recs is not None:
        assert record_bytes(out, precision) == target
    if flat is not None:
        flat = Scene(prims + extra + scenes.mesh_to_prims(mesh), scene.lights, scene.textures)
    return f"{name}+{kind}", out, flat if flat is not None else out, s


def one_more_record(scene, seed=0):
    """The scene of sized_scene with one more record and the same picture: one more unused entry in the mesh's material
    table, or, without a mesh, one more 1-geom filler shape.  -> (scene, flat)."""
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    if scene.mesh is not None:
        mesh = dict(scene.mesh)
        mesh["materials"] = list(mesh["materials"]) + [abi.copy_struct(mesh["materials"][0])]
        more = Scene(scene.prims, scene.lights, scene.textures, mesh=mesh)
        return more, Scene(scene.prims + scenes.mesh_to_prims(mesh), scene.lights, scene.textures)
    more = Scene(scene.prims + [_filler(np.random.default_rng(124000 + seed), 1)], scene.lights, scene.textures)
    return more, more


def random_refblur_scene(seed):
    """random_scene in the REFERENCE's blur mode after frame_prism: shapes named "rectangle" move in y during the blur
    re-traces of samples that hit a primitive flagged `motion` (render_final_project.cpp:1095-1210), leaf boxes are widened
    but interior ones are not (bumpBVH, Q14) -- on random geometry, rectangles of the diagonal kind included."""
    import numpy as np
    from distraytracer_b200 import abi
    from distraytracer_b200.scene import Scene
    case, scene, s = random_scene(seed)
    rng = np.random.default_rng(11000 + seed)
    prims = [abi.copy_struct(p) for p in scene.prims]
    for p in prims:
        if not (p.flags & abi.FLAG_LIGHT) and rng.random() < 0.5:
            p.flags |= abi.FLAG_MOTION
        # the reference's Rectangle constructor names every rectangle and checkerboard "rectangle" (geometry.cpp:618,636):
        # those are the shapes its blur moves.  The library takes the name as data; the reference cannot build the others.
        if p.type in (abi.PRIM_RECTANGLE, abi.PRIM_CHECKERBOARD, abi.PRIM_CHECKERBOARD_HOLE) and p.name == abi.NAME_OTHER:
            p.name = abi.NAME_RECTANGLE
    s.blur_mode = abi.BLUR_REFERENCE
    s.blur_samples, s.frame_range = int(rng.integers(1, 4)), int(rng.integers(1, 9))
    s.frame = int(rng.integers(0, 2000)); s.frame_prism = 0; s.frame_blur = int(rng.choice([0, 100000]))
    return "random_refblur", Scene(prims, scene.lights, scene.textures), s
