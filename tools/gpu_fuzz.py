"""GPU vs oracle on mutated fixture scenes, any number of seeds (tests/test_gpu_parity.py runs the first 14).
  python tools/gpu_fuzz.py [n_cases] [cam]
`scenes`: random scenes instead of mutated fixtures (random_scene); `meshes`: random triangle meshes (random_mesh_scene); `motion`: random scenes in velocity-blur mode (random_motion_scene); `big`: more than 256 shapes (random_big_scene);
`sky`: mutated fixtures in front of the value-noise clouds (sky_case); `meshmotion`: a moving mesh in velocity-blur mode; `prisms`: random slab-box prisms with holes (random_prism_scene); `glass`: random scenes with glass blocks; `refblur`: random scenes in the reference's own blur mode; `sizes`: fuzz_cases.sized_scene -- a random kind pushed to 255 / 256 / 257 geoms, 257..400 geoms or records just under the shared-memory bound.  `cam`: the camera is moved as well (eye / lookingAt jittered, focal length and aperture redrawn), so rays reach the scenes
from directions the reference's builders never look from -- grazing walls, looking along an axis, from inside a prism.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from fuzz_cases import mutated_case, random_scene, random_mesh_scene, random_motion_scene, random_big_scene, sky_case, random_moving_mesh_scene, random_prism_scene, random_glass_scene, random_refblur_scene, sized_scene, SIZED_KINDS, SMEM_RECS  # noqa: E402
from distraytracer_b200 import runtime  # noqa: E402
from oracle.harness import Oracle, ORACLE_KEYED, compare  # noqa: E402

n_cases = int(sys.argv[1]) if len(sys.argv) > 1 else 40
move_camera = len(sys.argv) > 2 and sys.argv[2] == "cam"
random_scenes = len(sys.argv) > 2 and sys.argv[2] == "scenes"
random_meshes = len(sys.argv) > 2 and sys.argv[2] == "meshes"
bad = 0
for seed in range(n_cases):
    flat = None
    if random_meshes: case, sc, flat, s = random_mesh_scene(seed)
    elif len(sys.argv) > 2 and sys.argv[2] == "meshmotion": case, sc, flat, s = random_moving_mesh_scene(seed)
    elif len(sys.argv) > 2 and sys.argv[2] == "motion": case, sc, s = random_motion_scene(seed)
    elif len(sys.argv) > 2 and sys.argv[2] == "big": case, sc, s = random_big_scene(seed)
    elif len(sys.argv) > 2 and sys.argv[2] == "sky": case, sc, s = sky_case(seed)
    elif len(sys.argv) > 2 and sys.argv[2] == "prisms": case, sc, s = random_prism_scene(seed)
    elif len(sys.argv) > 2 and sys.argv[2] == "glass": case, sc, s = random_glass_scene(seed)
    elif len(sys.argv) > 2 and sys.argv[2] == "refblur": case, sc, s = random_refblur_scene(seed)
    elif len(sys.argv) > 2 and sys.argv[2] == "sizes":
        import numpy as np
        rng = np.random.default_rng(78000 + seed)
        kind = SIZED_KINDS[int(rng.integers(len(SIZED_KINDS)))]
        size = int(rng.integers(4))
        kw = dict(geoms=int(rng.choice([255, 256, 257]))) if size == 0 else dict(geoms=int(rng.integers(257, 401))) if size == 1 else \
            dict(recs=SMEM_RECS, recs_at_most=True, precision=int(os.environ.get("DRT_FUZZ_PRECISION", "0"))) if size == 2 else {}
        try:
            case, sc, flat, s = sized_scene(kind, seed, **kw)
        except AssertionError:                          # base already past the requested size
            case, sc, flat, s = sized_scene(kind, seed)
    else: case, sc, s = random_scene(seed) if random_scenes else mutated_case(seed)
    if move_camera:
        import numpy as np
        rng = np.random.default_rng(77000 + seed)
        eye, look = np.array(s.eye[:]), np.array(s.lookingAt[:])
        d = np.linalg.norm(look - eye)
        kind = int(rng.integers(4))
        if kind == 0:                                   # jitter
            eye = eye + rng.normal(0, 0.25 * d, 3); look = look + rng.normal(0, 0.15 * d, 3)
        elif kind == 1:                                 # look along a coordinate axis from the old eye
            ax = np.zeros(3); ax[int(rng.integers(3))] = float(rng.choice([-1, 1])); look = eye + ax * d
            if abs(ax[1]) == 1: s.up[:] = [0, 0, 1]
        elif kind == 2:                                 # orbit the old target
            v = rng.normal(0, 1, 3); v /= np.linalg.norm(v); eye = look + v * d * float(rng.uniform(0.3, 1.5))
        else:                                           # stand close to the target
            eye = look + (eye - look) * float(rng.uniform(0.02, 0.3))
        s.eye[:] = [float(x) for x in eye]; s.lookingAt[:] = [float(x) for x in look]
        s.aperture = float(rng.choice([0.0, 0.05, 0.4])); s.focal_length = float(rng.uniform(0.5, 2.0) * d)
    s.precision = int(os.environ.get("DRT_FUZZ_PRECISION", "0"))     # 1: the single-precision build (same bar; rounding-fragile scenes may miss it)
    want, _, _, _ = Oracle(flat if flat is not None else sc).render(s, mode=ORACLE_KEYED)   # meshes: the oracle takes Triangle primitives
    got, _ = runtime.DeviceScene(sc, 0).render_float(s)
    st = compare(want, got)
    ok = st["frac_within_1"] >= 0.999
    bad += not ok
    print(f"seed {seed:3d} {case:24s} {s.xRes}x{s.yRes} aa={s.antialias_samples} depth={s.max_depth} lobes={s.brdf_samples} "
          f"blur={s.blur_samples} within1={st['frac_within_1']:.5f} max={st['max']} {'ok' if ok else 'MISMATCH'}", flush=True)
print("mismatching cases:", bad)
sys.exit(1 if bad else 0)
