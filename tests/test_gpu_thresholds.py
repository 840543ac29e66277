"""render_wave on both sides of its scene-size thresholds, in both precisions.

The launcher picks one render_wave instantiation per render call (csrc/drt_launch.h, DRT_WAVE_FEATS): the smallest
specialised feature mask that covers the scene and settings, with FT_RECS when the geom, primitive and light records fit
DRT_SMEM_RECS bytes (read from the CTA's shared copy), or FT_ALL.  Inside the kernel a ray takes its candidates from the
slab table in shared memory (up to DRT_SMEM_GEOMS geoms), from the same table in global memory (more geoms and a slab-box
prism), or from the 4-wide tree over the geoms (more geoms otherwise).  The scenes here come from
fuzz_cases.sized_scene: a random base scene plus hidden filler that moves it across one of those bounds without changing
its picture.  Every render asserts the instantiation it ran (Counters.kernel_variant) and that the counting build
(Counters.collect) draws the same picture, so a case's name is the path it checks.

  * test_same_picture_across_the_records_bound / _the_geoms_bound: the picture on both sides of a bound, to the bit.
  * test_oracle_parity_at_the_thresholds: the CPU oracle at the edges (255 / 256 / 257 geoms, odd counts, partial 32-geom
    words) and on the big-scene combinations: prisms, velocity blur, reference blur, diagonal-corner rectangles, coplanar
    twins, meshes, glass, unstaged meshes and reference blur.
  * test_every_instantiation_has_a_case: each (precision, mask, staged or not) the launcher can pick has a case here.
"""
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from fuzz_cases import SMEM_RECS, geom_count, one_more_record, record_bytes, sized_scene

TOL_FRAC = 0.999   # the north-star bar: fraction of pixels within 1/255 of the oracle
PRECISIONS = pytest.mark.parametrize("precision", [0, 1], ids=["reference", "fp32"])


def _wave_feats():
    """(WaveFeat name -> value, the masks of DRT_WAVE_FEATS) parsed from csrc/drt_launch.h."""
    text = open(os.path.join(ROOT, "distraytracer_b200", "csrc", "drt_launch.h")).read()
    ft = {k: int(v) for k, v in re.findall(r"\b(FT_[A-Z]+)\s*=\s*(\d+)", text)}
    body = re.search(r"#define\s+DRT_WAVE_FEATS\s*\{([^}]*)\}", text).group(1)
    masks = []
    for term in body.split(","):
        m = 0
        for tok in term.split("|"):
            tok = tok.strip()
            m |= ft[tok] if tok.startswith("FT_") else int(tok)
        masks.append(m)
    return ft, masks


FT, WAVE_FEATS = _wave_feats()
ALL, RECS = FT["FT_ALL"], FT["FT_RECS"]
TEX, GLASS, VEL, MESH, REFBLUR = FT["FT_TEX"], FT["FT_GLASS"], FT["FT_VEL"], FT["FT_MESH"], FT["FT_REFBLUR"]

# (kind, seed, mask) -- records of exactly DRT_SMEM_RECS bytes (mask | FT_RECS) against one record more (mask).  The
# mesh kinds cross the bound through their material table.  A glass scene is near the bound before any filler, and no
# filler adds exactly the bytes it lacks: there the staged side is the nearest byte count below the bound.
RECORD_PAIRS = [("scene", 11, 0), ("textured", 14, TEX), ("glass", 42, GLASS | TEX), ("motion", 15, VEL),
                ("mesh", 0, MESH | TEX), ("moving_mesh", 3, MESH | VEL | TEX)]
# (kind, seed, mask) rendered at 255, 256 and 257 geoms: mask (records far over the bound), then FT_ALL and the geom tree
GEOM_EDGES = [("scene", 15, 0), ("motion", 19, VEL)]
# (id, kind, seed, sized_scene arguments, variant) against the oracle
ORACLE_CASES = [
    ("geoms255", "scene", 14, dict(geoms=255), 0),                       # odd count, partial group of 8 and 32-geom word
    ("geoms256", "scene", 14, dict(geoms=256), 0),                       # the shared-memory slab table exactly full
    ("geoms257_tree", "scene", 14, dict(geoms=257), ALL),
    ("geoms258_tree_twins", "scene", 4, dict(geoms=258, twins=True), ALL),   # coplanar twins: ties of t in the geom tree
    ("geoms288_tree_twins", "scene", 7, dict(geoms=288, twins=True), ALL),
    ("big_prism257_global_table", "prism", 0, dict(geoms=257), ALL),     # a prism: no geom tree, the global slab table
    ("big_prism264_global_table", "prism", 3, dict(geoms=264), ALL),     # partial 32-geom word, whole groups of 8
    ("big_prism288_global_table", "prism", 1, dict(geoms=288), ALL),     # whole 32-geom words
    ("big_velocity_swept_tree", "motion", 2, dict(geoms=300, frame_range=1), ALL),
    ("big_velocity_unfiltered", "motion", 9, dict(geoms=300, frame_range=3), ALL),
    ("big_refblur_reference_tree", "refblur", 11, dict(geoms=300), ALL),
    ("spill_small", "scene", 0, dict(), ALL),                            # diagonal-corner rectangles alone pick FT_ALL
    ("big_spill_tree", "scene", 0, dict(geoms=300), ALL),
    ("big_spill_tree_twins", "scene", 6, dict(geoms=300, twins=True), ALL),
    ("big_mesh", "mesh", 0, dict(geoms=300), ALL),
    ("big_glass", "glass", 12, dict(geoms=300), ALL),
    ("unstaged_mesh", "mesh", 3, dict(extra_materials=45), MESH | TEX),
    ("unstaged_moving_mesh", "moving_mesh", 0, dict(extra_materials=45), MESH | VEL | TEX),
    ("staged_refblur", "refblur", 4, dict(), REFBLUR | GLASS | TEX | RECS),
    ("unstaged_refblur", "refblur", 5, dict(geoms=60), REFBLUR | GLASS | TEX),
]


def _reached():
    """Every instantiation some case here asserts, for each precision (all cases run in both)."""
    v = set()
    for _, _, m in RECORD_PAIRS:
        v |= {m | RECS, m}
    for _, _, m in GEOM_EDGES:
        v |= {m, ALL}
    v |= {c[-1] for c in ORACLE_CASES}
    return {(p, x) for p in (0, 1) for x in v}


def _pickable():
    """What launchRenderSamples can launch: every mask of DRT_WAVE_FEATS but FT_ALL with and without FT_RECS, FT_ALL."""
    assert WAVE_FEATS[-1] == ALL
    return {(p, x) for p in (0, 1) for m in WAVE_FEATS for x in ((m, m | RECS) if m != ALL else (ALL,))}


# collection fails when an instantiation is added without a case for it
assert _pickable() <= _reached(), f"render_wave instantiations without a case here: {sorted(_pickable() - _reached())}"


def test_every_instantiation_has_a_case():
    assert len(WAVE_FEATS) == 8 and len(_pickable()) == 2 * 15
    assert _pickable() <= _reached(), sorted(_pickable() - _reached())


@pytest.mark.parametrize("kind,seed", [(k, s) for k, s, _ in RECORD_PAIRS + GEOM_EDGES],
                         ids=[k for k, _, _ in RECORD_PAIRS + GEOM_EDGES])
def test_filler_leaves_the_oracle_picture_alone(oracle_lib, kind, seed):
    """What the pictures of the GPU pairs below rest on: the filler inside the enclosing sphere changes no pixel of the
    oracle's picture, from the smallest scene to 257 geoms and across the records bound."""
    from oracle.harness import Oracle, ORACLE_KEYED
    mesh = kind in ("mesh", "moving_mesh")
    _, base, base_flat, s = sized_scene(kind, seed, extra_materials=1 if mesh else 0)
    _, under, under_flat, _ = sized_scene(kind, seed, recs=SMEM_RECS, recs_at_most=True, extra_materials=1 if mesh else 0)
    _, over_flat = one_more_record(under, seed)
    _, _, big_flat, _ = sized_scene(kind, seed, geoms=257, extra_materials=1 if mesh else 0)
    want = Oracle(base_flat).render(s, mode=ORACLE_KEYED)[0]
    assert want.std() > 5
    for flat in (under_flat, over_flat, big_flat):
        assert np.array_equal(want, Oracle(flat).render(s, mode=ORACLE_KEYED)[0], equal_nan=True)


def _render(scene, s, precision, variant):
    """The production build's float and u8 images; asserts the instantiation launched, and that the counting build
    (render_wave<R, FT_ALL, true>) draws the same picture."""
    from distraytracer_b200 import abi, runtime
    assert runtime.device_count() >= 1, "no CUDA device: the product path has no CPU fallback"
    s.precision = precision
    dev = runtime.DeviceScene(scene, 0)
    c = abi.Counters()
    got, got_u8 = dev.render_float(s, counters=c)
    assert c.kernel_variant == variant, ("kernel_variant", c.kernel_variant, "expected", variant)
    k = abi.Counters(); k.collect = 1
    cnt, cnt_u8 = dev.render_float(s, counters=k)
    assert k.kernel_variant == ALL and k.rays > 0
    _same((got, got_u8), (cnt, cnt_u8), "counting build", exact=precision == 0 or variant == ALL)
    dev.close()
    return got, got_u8


def _same(a, b, what, exact=True):
    """Same float and u8 images, to the bit.  exact=False: the single-precision build across two feature masks.  Those
    kernels are compiled with FMA contraction (csrc/drt_launch.h), and an instantiation with more features can fuse a
    multiply-add that another rounds twice (shiftPoint's `p + vel * time`, for one), so the two pictures may differ in the
    last bits of a few pixels; there the bar is the oracle's."""
    from oracle.harness import compare
    if not exact:
        st = compare(a[0], b[0])
        assert st["frac_within_1"] >= TOL_FRAC, (what, st)
        return
    assert np.array_equal(a[0], b[0], equal_nan=True), (what, "float images differ", float(np.nanmax(np.abs(a[0] - b[0]))))
    assert np.array_equal(a[1], b[1]), (what, "u8 images differ")


@pytest.mark.gpu
@PRECISIONS
@pytest.mark.parametrize("kind,seed,mask", RECORD_PAIRS, ids=[k for k, _, _ in RECORD_PAIRS])
def test_same_picture_across_the_records_bound(kind, seed, mask, precision):
    """Records of exactly DRT_SMEM_RECS bytes are staged in shared memory; one record more and they are read from global
    memory.  Same picture, to the bit."""
    mesh = kind in ("mesh", "moving_mesh")
    _, under, _, s = sized_scene(kind, seed, precision, recs=SMEM_RECS, recs_at_most=True, extra_materials=1 if mesh else 0)
    over, _ = one_more_record(under, seed)
    assert record_bytes(under, precision) == SMEM_RECS or kind == "glass"
    assert record_bytes(under, precision) <= SMEM_RECS < record_bytes(over, precision)
    a = _render(under, s, precision, mask | RECS)
    b = _render(over, s, precision, mask)
    _same(a, b, (kind, seed))
    assert a[1].std() > 5, "nothing in view"


@pytest.mark.gpu
@PRECISIONS
@pytest.mark.parametrize("kind,seed,mask", GEOM_EDGES, ids=[k for k, _, _ in GEOM_EDGES])
def test_same_picture_across_the_geoms_bound(kind, seed, mask, precision):
    """255 geoms (odd: the padding pair entry; partial group of 8 and 32-geom word), 256 (the shared-memory slab table
    exactly full) and 257 (FT_BIG: FT_ALL and the tree over the geoms).  Same picture, to the bit (see _same for the
    single-precision build across feature masks)."""
    pics = []
    for n, variant in ((255, mask), (256, mask), (257, ALL)):
        _, scene, _, s = sized_scene(kind, seed, precision, geoms=n)
        assert geom_count(scene.prims) == n
        pics.append(_render(scene, s, precision, variant))
    _same(pics[0], pics[1], (kind, seed, "255 / 256 geoms"))
    _same(pics[1], pics[2], (kind, seed, "256 / 257 geoms"), exact=precision == 0 or mask == ALL)


@pytest.mark.gpu
@PRECISIONS
@pytest.mark.parametrize("case,kind,seed,kwargs,variant", ORACLE_CASES, ids=[c[0] for c in ORACLE_CASES])
def test_oracle_parity_at_the_thresholds(oracle_lib, case, kind, seed, kwargs, variant, precision):
    """The CUDA path against the CPU oracle on identical sample positions (the tests/test_gpu_parity.py bar)."""
    from oracle.harness import Oracle, ORACLE_KEYED, compare
    _, scene, flat, s = sized_scene(kind, seed, precision, **kwargs)
    want, _, _, _ = Oracle(flat).render(s, mode=ORACLE_KEYED)
    got, _ = _render(scene, s, precision, variant)
    st = compare(want, got)
    print(f"threshold-oracle {case} precision={precision} variant={variant} geoms={geom_count(scene.prims)} "
          f"recs={record_bytes(scene, precision)} frac_within_1={st['frac_within_1']:.5f} max={st['max']}")
    assert st["frac_within_1"] >= TOL_FRAC, (case, precision, st)
    assert float(np.nanmax(np.abs(want))) > 0.2               # not a black frame
