"""Randomised pin of the CPU restatement on the compiled reference.  Beyond the 15 stored fixtures: reference scene builders
at random frames with random settings (resolution, spp, aperture, lobes, depth, switches, seed), and generated scenes
loaded into the reference, rendered by the UNMODIFIED reference rayColor and by oracle/drt_oracle.cpp under the same
sequential sample stream -- floats and abort masks must agree to the bit.  The comparisons against the live reference
need oracle/_ref and the reference's tree; for the generated scenes the reference's images are also stored, as digests
(tests/golden/reference_pins.json), so those cases are checked without the reference too."""
import os

import numpy as np
import pytest

from conftest import assert_pinned

BUILDERS = ["hw4", "reflectance", "dof", "spherelight", "spheres", "checkertexture", "texture", "textureog", "window",
            "staircase", "rectprism", "checkercylinder", "chkpt2", "boundary"]


def _have_reference():
    from oracle.harness import ref_available, REFERENCE_ROOT
    return ref_available() and os.path.isdir(os.path.join(REFERENCE_ROOT, "textures"))


def _reference_render(scene, s, mocap):
    from oracle.harness import Ref
    r = Ref(mocap=mocap)
    r.reset()
    r.load(scene)
    r.set_settings(s)
    r.rng(1, s.seed, 0)
    ref_img, ref_ab, _ = r.render_loop(int(s.frame), reset_policy=1, seed=s.seed)
    return ref_img, ref_ab


def _pinned_render(key, scene, s, mocap=False):
    """The restatement's image of `scene` is the reference's: compared with the compiled reference where it is built,
    and with the stored pin everywhere."""
    from oracle.harness import Oracle, ORACLE_STREAM
    img, ab, cnt, _ = Oracle(scene).render(s, mode=ORACLE_STREAM)
    live = _have_reference()
    if live:
        ref_img, ref_ab = _reference_render(scene, s, mocap)
        assert (ab == ref_ab).all(), (key, "abort masks differ")
        assert np.array_equal(ref_img, img, equal_nan=True), (key, float(np.nanmax(np.abs(ref_img - img))))
    assert_pinned(key, img, ab, matched_reference=live)
    return img, ab, cnt


@pytest.mark.parametrize("seed", range(28))
def test_restatement_matches_reference_on_random_settings(oracle_lib, seed):
    if not _have_reference():
        pytest.skip("reference tree not present (GPU box): pinned by the stored fixtures instead")
    from oracle.harness import Ref, Oracle, ORACLE_STREAM
    rng = np.random.default_rng(1000 + seed)
    builder = BUILDERS[seed % len(BUILDERS)] if seed < len(BUILDERS) else BUILDERS[int(rng.integers(len(BUILDERS)))]
    frame = int(rng.integers(0, 120))
    if builder == "boundary":                       # buildSceneBoundary only knows its stages -1, 0, 1, 2 (scene.h:2273-2613)
        frame = int(rng.integers(0, 3))
    r = Ref(mocap=True)
    r.reset()
    r.build(builder, frame)
    s = r.settings()
    s.xRes, s.yRes = int(rng.integers(24, 57)), int(rng.integers(18, 41))
    s.antialias_samples = int(rng.choice([1, 2, 4, 9]))
    s.aperture = float(rng.choice([0.0, 0.2, 0.5]))
    s.brdf_samples = int(rng.integers(1, 4))
    s.max_depth = int(rng.integers(1, 7))
    s.nogloss = int(rng.random() < 0.25)
    s.reflect = int(rng.random() < 0.85)
    s.frame, s.seed = frame, int(rng.integers(1, 1 << 30))
    r.set_settings(s)
    scene = r.export()
    r.rng(1, s.seed, 0)
    ref_img, ref_ab, _ = r.render_loop(frame, reset_policy=1, seed=s.seed)
    img, ab, _, _ = Oracle(scene).render(s, mode=ORACLE_STREAM)
    assert (ab == ref_ab).all(), (builder, frame, "abort masks differ")
    assert np.array_equal(ref_img, img, equal_nan=True), (builder, frame, float(np.nanmax(np.abs(ref_img - img))))


@pytest.mark.parametrize("seed", range(40))
def test_restatement_matches_reference_on_mutated_scenes(oracle_lib, seed):
    """Same pin, wider domain: the exported scene is mutated (motion flags, BRDF model, roughness, reflective material,
    glossy flag; motion-blur settings incl. the reference's own "rectangle" translation after frame_prism) and loaded
    back INTO the reference, so material x shape x blur combinations no stock builder produces are compared too."""
    if not _have_reference():
        pytest.skip("reference tree not present (GPU box): pinned by the stored fixtures instead")
    from distraytracer_b200 import abi
    from distraytracer_b200.scene import Scene
    from oracle.harness import Ref, Oracle, ORACLE_STREAM
    rng = np.random.default_rng(5000 + seed)
    builder = BUILDERS[int(rng.integers(len(BUILDERS)))]
    frame = int(rng.integers(0, 3)) if builder == "boundary" else int(rng.integers(0, 120))
    r = Ref(mocap=True)
    r.reset()
    r.build(builder, frame)
    s = r.settings()
    s.xRes, s.yRes = int(rng.integers(24, 49)), int(rng.integers(18, 37))
    s.antialias_samples = int(rng.choice([1, 4]))
    s.aperture = float(rng.choice([0.0, 0.2]))
    s.brdf_samples = int(rng.integers(1, 4))
    s.max_depth = int(rng.integers(1, 6))
    s.blur_samples = int(rng.integers(0, 4))
    s.frame_range = int(rng.integers(1, 9))
    if rng.random() < 0.4:                           # frame >= frame_prism: shapes named "rectangle" move during blur re-traces
        s.frame_prism, s.frame_blur = 0, int(rng.choice([0, 100000]))
    s.frame, s.seed = frame, int(rng.integers(1, 1 << 30))
    scene = r.export()
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
    scene = Scene(prims, scene.lights, scene.textures)
    r.load(scene)
    r.set_settings(s)
    r.rng(1, s.seed, 0)
    ref_img, ref_ab, _ = r.render_loop(frame, reset_policy=1, seed=s.seed)
    img, ab, _, _ = Oracle(scene).render(s, mode=ORACLE_STREAM)
    assert (ab == ref_ab).all(), (builder, frame, "abort masks differ")
    assert np.array_equal(ref_img, img, equal_nan=True), (builder, frame, float(np.nanmax(np.abs(ref_img - img))))


@pytest.mark.parametrize("seed", range(30))
def test_restatement_matches_reference_on_random_scenes(oracle_lib, seed):
    """Scenes no builder of the reference produces (fuzz_cases.random_scene: random spheres, cylinders, triangles,
    rectangles with their corners in ANY order -- a third of them therefore with D - A a diagonal, Q20 -- checkerboards,
    all three light kinds) loaded INTO the compiled reference: the restatement reproduces them to the bit."""
    from fuzz_cases import random_scene
    _, scene, s = random_scene(seed)
    _pinned_render(f"random_scenes/{seed}", scene, s)


@pytest.mark.parametrize("seed", range(30))
def test_restatement_matches_reference_on_random_scenes_with_its_own_blur(oracle_lib, seed):
    """fuzz_cases.random_refblur_scene: the random scenes in the REFERENCE's blur mode after frame_prism -- every rectangle
    and checkerboard moves in y during the blur re-traces (the reference names them all "rectangle"), leaf boxes are bumped,
    interior ones are not -- loaded into the compiled reference: reproduced to the bit."""
    from fuzz_cases import random_refblur_scene
    _, scene, s = random_refblur_scene(seed)
    _pinned_render(f"random_refblur_scenes/{seed}", scene, s)


@pytest.mark.parametrize("seed", range(8))
def test_restatement_matches_reference_on_big_random_scenes(oracle_lib, seed):
    """fuzz_cases.random_big_scene: 257 .. 700 small shapes over a floor (the scenes on which the CUDA path gathers through
    its tree over the geoms) loaded INTO the compiled reference: reproduced to the bit."""
    from fuzz_cases import random_big_scene
    _, scene, s = random_big_scene(seed)
    _pinned_render(f"big_random_scenes/{seed}", scene, s)


@pytest.mark.parametrize("seed", range(4))
def test_restatement_matches_reference_with_the_cloud_background(oracle_lib, seed):
    """fuzz_cases.sky_case: mutated fixture scenes in front of the value-noise clouds (perlin_cloud: cloudColor per missed
    sample, noise.h) loaded INTO the compiled reference: reproduced to the bit."""
    from fuzz_cases import sky_case
    _, scene, s = sky_case(seed)
    _pinned_render(f"cloud_background/{seed}", scene, s)


@pytest.mark.parametrize("cfg", ["config1", "config2", "config3"])
def test_restatement_matches_reference_on_the_bench_workloads(oracle_lib, cfg):
    """The BASELINE configurations themselves (distraytracer_b200.scenes: config 2 is what bench.py times -- glass
    triangles, rectangle light, glossy floor, DOF) loaded INTO the compiled reference at reduced size: the restatement
    reproduces the reference's image to the bit -- except where the reference's own result is undefined (glass, Q3).  (Configs 4 and 5 use per-primitive velocities / a mesh type, which the
    reference does not have; their oracle paths are the same code driven by other inputs.)"""
    from distraytracer_b200 import scenes
    from oracle.harness import Oracle, ORACLE_STREAM
    scene, s = {"config1": scenes.config1, "config2": lambda: scenes.config2(64, 36, 4),
                "config3": lambda: scenes.config3(64, 36, 4)}[cfg]()
    if cfg == "config1":
        s.xRes, s.yRes = 64, 48
    s.seed = 4242
    if cfg != "config2":
        img, _, cnt = _pinned_render(f"bench_workloads/{cfg}", scene, s, mocap=True)
        assert np.nanstd(img) > 5 and cnt.rays > s.xRes * s.yRes
        return
    img, ab, cnt, _ = Oracle(scene).render(s, mode=ORACLE_STREAM)
    assert np.nanstd(img) > 5 and cnt.rays > s.xRes * s.yRes
    # config 2 holds glass.  Where a ray tree reaches a glass surface the reference reads an UNINITIALISED variable
    # (`inside = inside_tmp`, render_final_project.cpp:524,534 -- quirk Q3): what it renders there depends on the compiler, and
    # the restatement implements the evident intent (the inside flag of the closest hit).  Everywhere else: to the bit.
    from distraytracer_b200 import abi
    from distraytracer_b200.scene import Scene
    def recoloured(rgb):                             # the glass triangles as plain "raw"-shaded surfaces of one colour
        out = [abi.copy_struct(p) for p in scene.prims]
        for p in out:
            if p.material == abi.MAT_GLASS:
                p.material, p.model = abi.MAT_NONE, abi.MODEL_RAW
                p.color[:] = rgb
        return out
    plain = recoloured((1.0, 0.0, 1.0))
    no_glass, nab, _, _ = Oracle(Scene(plain, scene.lights, scene.textures)).render(s, mode=ORACLE_STREAM)
    other, oab, _, _ = Oracle(Scene(recoloured((0.0, 1.0, 0.0)), scene.lights, scene.textures)).render(s, mode=ORACLE_STREAM)
    # a pixel whose ray trees reach those triangles (directly or by reflection) changes with their colour
    touches_glass = (nab != oab) | (np.nan_to_num(no_glass, nan=-1.0) != np.nan_to_num(other, nan=-1.0)).any(axis=-1)
    # (+ their 8 neighbours: on the block's silhouette both colourings saturate to white under the light panel)
    grown = touches_glass.copy()
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            grown |= np.roll(np.roll(touches_glass, dy, axis=0), dx, axis=1)
    assert 0 < grown.mean() < 0.25
    live = _have_reference()
    if live:
        ref_img, ref_ab = _reference_render(scene, s, mocap=True)
        same = (ab == ref_ab) & (np.nan_to_num(ref_img, nan=-1.0) == np.nan_to_num(img, nan=-1.0)).all(axis=-1)
        assert same[~grown].all()
        assert 0 < (~same).sum() <= grown.sum()
        # and with the glass taken out of the material the whole frame is bit-identical again
        ref2, ref2_ab = _reference_render(Scene(plain, scene.lights, scene.textures), s, mocap=True)
        assert (ref2_ab == nab).all() and np.array_equal(ref2, no_glass, equal_nan=True)
    assert_pinned("bench_workloads/config2/outside_glass", np.where(grown[..., None], np.float32(0), img), ab & ~grown,
                  matched_reference=live)
    assert_pinned("bench_workloads/config2/glass_as_plain_surfaces", no_glass, nab, matched_reference=live)


def test_restatement_matches_reference_on_a_textured_triangle_terrain(oracle_lib):
    """BASELINE config 5 at reduced size (2 x 11^2 = 242 textured Oren-Nayar triangles with per-vertex UVs + a sphere,
    DOF), its mesh handed to the reference as individual Triangle primitives (what its loadObj path produces) and run
    through the reference's own SAH BVH: the restatement reproduces it to the bit.  The velocity blur of config 5 is
    switched off -- the reference has no per-primitive velocities."""
    from distraytracer_b200 import scenes, abi
    from distraytracer_b200.scene import Scene
    scene, s = scenes.config5(n=12, xres=64, yres=36, spp=4)
    s.blur_samples, s.blur_mode, s.seed = 0, abi.BLUR_REFERENCE, 777
    prims = [abi.copy_struct(p) for p in scene.prims]
    for p in prims:
        p.flags &= ~abi.FLAG_MOTION
        p.velocity[:] = [0.0, 0.0, 0.0]
    flat = Scene(prims + scenes.mesh_to_prims(scene.mesh), scene.lights, scene.textures)
    img, _, cnt = _pinned_render("textured_triangle_terrain", flat, s, mocap=True)
    assert np.nanstd(img) > 5 and cnt.prim_tests[abi.PRIM_TRIANGLE] > 0


def test_glass_divergence_is_the_uninitialised_inside_flag(oracle_lib, tmp_path):
    """Evidence for the Q3 waiver: switching the restatement to what gcc 13 -O3 happens to make of `inside = inside_tmp`
    (the assignment is dropped, so `inside` is the flag of the LAST candidate tested; DRT_ORACLE_Q3=last_tested, a
    diagnostic that exists only for this test) removes most of the glass pixels on which the compiled reference and the
    restatement differ; what remains are NaN-versus-abort swaps on the block's silhouette, i.e. two spellings of garbage."""
    if not _have_reference():
        pytest.skip("reference tree not present (GPU box)")
    import subprocess
    import sys
    from conftest import ROOT
    code = (
        "import sys, numpy as np; sys.path.insert(0, %r)\n"
        "from distraytracer_b200 import scenes\n"
        "from oracle.harness import Ref, Oracle, ORACLE_STREAM\n"
        "scene, s = scenes.config2(64, 36, 4); s.seed = 4242\n"
        "r = Ref(mocap=True); r.reset(); r.load(scene); r.set_settings(s); r.rng(1, s.seed, 0)\n"
        "ref, rab, _ = r.render_loop(s.frame, reset_policy=1, seed=s.seed)\n"
        "img, ab, _, _ = Oracle(scene).render(s, mode=ORACLE_STREAM)\n"
        "same = (ab == rab) & (np.nan_to_num(ref, nan=-1.0) == np.nan_to_num(img, nan=-1.0)).all(axis=-1)\n"
        "print('DIFF', int((~same).sum()))\n" % ROOT)

    def differing(env_value):
        env = dict(os.environ)
        env.pop("DRT_ORACLE_Q3", None)
        if env_value:
            env["DRT_ORACLE_Q3"] = env_value
        out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, check=True).stdout
        return int([ln for ln in out.splitlines() if ln.startswith("DIFF")][-1].split()[1])

    pinned, emulated = differing(None), differing("last_tested")
    assert 20 <= pinned <= 120 and emulated <= pinned // 4, (pinned, emulated)


def test_restatement_equals_the_reference_with_the_inside_flag_fixed(oracle_lib, tmp_path):
    """The other half of the Q3 evidence: compile the reference once more with the one-word fix
    `shape->intersect(ray, eye, t_dist, inside_tmp)` (render_final_project.cpp:526) applied to a temporary copy outside the
    repository, and the restatement reproduces BASELINE config 2 -- the bench workload, glass included -- to the bit,
    abort masks included.  (~40 s: one more build of the reference.)"""
    if not _have_reference():
        pytest.skip("reference tree not present (GPU box)")
    import subprocess
    import sys
    from conftest import ROOT
    from oracle.harness import REFERENCE_ROOT
    src = open(os.path.join(REFERENCE_ROOT, "render_final_project.cpp")).read()
    broken = "bool intersect = shape->intersect(ray, eye, t_dist, inside);"
    assert src.count(broken) == 1
    (tmp_path / "render_final_project.cpp").write_text(src.replace(broken, "bool intersect = shape->intersect(ray, eye, t_dist, inside_tmp);"))
    so = str(tmp_path / "libdrt_ref_fixed.so")
    orc = os.path.join(ROOT, "oracle")
    subprocess.check_call(["/usr/bin/g++", "-O3", "-std=c++17", "-fPIC", "-w", "-shared", "-I" + os.path.join(orc, "ref_shim"),
                           "-I" + os.path.join(orc, "eigen_shim"), "-I" + str(tmp_path), "-I" + REFERENCE_ROOT,
                           os.path.join(orc, "ref_driver.cpp")] +
                          [os.path.join(REFERENCE_ROOT, f) for f in ("geometry.cpp", "skeleton.cpp", "motion.cpp", "displaySkeleton.cpp")] +
                          ["-o", so])
    code = (
        "import sys, numpy as np; sys.path.insert(0, %r)\n"
        "from distraytracer_b200 import scenes\n"
        "from oracle.harness import Ref, Oracle, ORACLE_STREAM\n"
        "for res in ((64, 36, 4), (120, 68, 9)):\n"
        "    scene, s = scenes.config2(*res); s.seed = 4242\n"
        "    r = Ref(mocap=True); r.reset(); r.load(scene); r.set_settings(s); r.rng(1, s.seed, 0)\n"
        "    ref, rab, _ = r.render_loop(s.frame, reset_policy=1, seed=s.seed)\n"
        "    img, ab, _, _ = Oracle(scene).render(s, mode=ORACLE_STREAM)\n"
        "    same = (ab == rab) & (np.nan_to_num(ref, nan=-1.0) == np.nan_to_num(img, nan=-1.0)).all(axis=-1)\n"
        "    print('DIFF', int((~same).sum()), int(np.isnan(img).any(-1).sum()))\n" % ROOT)
    env = dict(os.environ, DRT_REF_SO=so)
    env.pop("DRT_ORACLE_Q3", None)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, check=True).stdout
    rows = [ln.split() for ln in out.splitlines() if ln.startswith("DIFF")]
    assert len(rows) == 2 and all(int(r[1]) == 0 for r in rows), rows
    assert all(int(r[2]) > 0 for r in rows)            # the glass block is in the picture (its NaN Fresnel terms are)
