"""Rays that leave a planar surface do not exact-test that surface again.

Shadow rays and glass / mirror children start 1e-3 along a unit direction from the surface they leave.  The slab-filter
boxes of rectangles and triangles are padded by their rounding error only (padBounds in csrc/drt_box.cuh), far less than
that offset, so the filter drops the plane behind such a ray before its exact test.  These tests count the exact tests
of one instrumented frame (Counters.collect)."""
import pytest

pytestmark = pytest.mark.gpu


def _counted(scene, s):
    from distraytracer_b200 import abi, runtime
    assert runtime.device_count() >= 1, "no CUDA device: the product path has no CPU fallback"
    c = abi.Counters()
    c.collect = 1
    runtime.DeviceScene(scene, 0).render(s, counters=c)
    return c


def _looking_down(eye, xres, yres):
    from distraytracer_b200 import runtime
    s = runtime.default_settings()
    s.xRes, s.yRes, s.aspect = xres, yres, xres / yres
    s.eye[:] = list(eye); s.lookingAt[:] = [0.0, 0.0, 0.0]; s.up[:] = [0.0, 0.0, -1.0]
    s.antialias_samples, s.aperture, s.blur_samples, s.reflect = 1, 0.0, 0, 0
    return s


@pytest.mark.parametrize("precision", [0, 1], ids=["reference", "fp32"])
def test_shadow_rays_leaving_the_floor_add_no_rectangle_tests(precision):
    """One rectangle floor under a point light, seen from above: every camera ray hits the floor and casts one shadow
    ray, which leaves the floor upwards and must not exact-test it.  With the old 1e-3 pad each shadow ray did."""
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    floor = scenes.rectangle((-10, 0, 10), (10, 0, 10), (10, 0, -10), (-10, 0, -10), (0.8, 0.8, 0.8), name=abi.NAME_OTHER)
    s = _looking_down((0.0, 4.0, 0.0), 64, 48)
    s.precision = precision
    c = _counted(Scene([floor], [scenes.point_light((0.5, 5.0, -0.5), (1.0, 1.0, 1.0))]), s)
    assert c.rays == 64 * 48
    assert c.shadow_rays >= 0.99 * c.rays                 # the floor fills the view: nearly every camera ray hits it
    assert c.prim_tests[abi.PRIM_RECTANGLE] <= c.rays


@pytest.mark.parametrize("precision", [0, 1], ids=["reference", "fp32"])
def test_rays_leaving_a_glass_face_skip_its_two_triangles(precision):
    """A glass block (12 triangles) under a point light: refraction and mirror children and shadow rays leave a face of
    the block, which is two triangles with one box.  Only the faces ahead of a ray are to be tested."""
    from distraytracer_b200 import abi, scenes
    from distraytracer_b200.scene import Scene
    prims = scenes.glass_block((-1.0, -0.5, -0.8), (1.0, 0.5, 0.8))
    s = _looking_down((1.5, 4.0, 2.5), 64, 48)
    s.up[:] = [0.0, 1.0, 0.0]
    s.reflect = 1                                           # refraction and mirror children
    s.precision = precision
    c = _counted(Scene(prims, [scenes.point_light((2.0, 6.0, 1.0), (1.0, 1.0, 1.0))]), s)
    traced = c.rays + c.shadow_rays
    assert c.rays > 64 * 48 and c.shadow_rays > 0          # the block is in view and spawns children
    # 2.27 triangle tests per traced ray with the old pad; 0.91 (reference) and 0.98 (fp32) with the planar pad
    assert c.prim_tests[abi.PRIM_TRIANGLE] <= 1.5 * traced
