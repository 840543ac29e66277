"""ASF/AMC mocap ingest + forward kinematics (BASELINE config 4).

CPU: the oracle's restatement (oracle/drt_skeleton_oracle.cpp) is pinned bit-for-bit on the bone end points
the compiled reference produced (tests/golden/mocap_bones_880_999.npy, written by make_golden.py through
drtref_mocap_bones) and, where the reference tree is present, on frames over the whole clip.
GPU: the device table of drt_skeleton_create (kernel skeleton_fk) is bit-identical to the oracle, and a scene
re-posed from it renders the same image as one given the reference's bones."""
import os

import numpy as np
import pytest

from conftest import GOLDEN

ASF = os.path.join(GOLDEN, "mocap_90.asf")
AMC = os.path.join(GOLDEN, "mocap_90_16_frames880_1000.amc")


def _clip():
    with open(ASF, "rb") as f:
        asf = f.read()
    with open(AMC, "rb") as f:
        amc = f.read()
    return asf, amc


def test_oracle_fk_is_pinned_on_the_reference_bones(oracle_lib):
    from oracle.harness import SkeletonOracle
    sk = SkeletonOracle(*_clip())
    assert (sk.n_cylinders, sk.n_frames) == (30, 121)
    gold = np.load(os.path.join(GOLDEN, "mocap_bones_880_999.npy"))
    got = np.stack([sk.bones(f) for f in range(120)])
    assert np.array_equal(got, gold)                      # bit-exact, all 120 x 30 x 6 doubles
    # past the clip the reference clamps to the last frame (scene.h:117-121); negative frames are fatal (:111-115)
    assert np.array_equal(sk.bones(5000), sk.bones(120))
    with pytest.raises(RuntimeError):
        sk.bones(-1)


def test_oracle_fk_matches_compiled_reference_over_the_whole_clip(oracle_lib):
    from oracle.harness import SkeletonOracle, Ref, ref_available, REFERENCE_ROOT
    if not (ref_available() and os.path.exists(os.path.join(REFERENCE_ROOT, "90_16_v3.amc"))):
        pytest.skip("reference tree not present (GPU box): pinned by the golden bones instead")
    with open(os.path.join(REFERENCE_ROOT, "90.asf"), "rb") as f:
        asf = f.read()
    with open(os.path.join(REFERENCE_ROOT, "90_16_v3.amc"), "rb") as f:
        amc = f.read()
    sk = SkeletonOracle(asf, amc)
    assert sk.n_frames == 2964
    ref = Ref(mocap=True)
    for frame in list(range(0, 2964, 97)) + [2963, 4000]:
        assert np.array_equal(sk.bones(frame), ref.mocap_bones(frame)), frame


def test_skeleton_needs_a_device():
    """No CPU fallback: without a GPU the ingest fails with DRT_ERR_NO_DEVICE."""
    from distraytracer_b200 import runtime, abi
    if runtime.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(runtime.DrtError) as e:
        runtime.DeviceSkeleton(*_clip())
    assert e.value.code == abi.ERR_NO_DEVICE


@pytest.mark.gpu
def test_cuda_fk_table_is_bit_identical_to_the_oracle(oracle_lib):
    from distraytracer_b200 import runtime
    from oracle.harness import SkeletonOracle
    asf, amc = _clip()
    dev = runtime.DeviceSkeleton(asf, amc)
    orc = SkeletonOracle(asf, amc)
    assert (dev.n_cylinders, dev.n_frames) == (orc.n_cylinders, orc.n_frames) == (30, 121)
    got = dev.bones()
    want = np.stack([orc.bones(f) for f in range(orc.n_frames)])
    assert np.array_equal(got, want)
    assert np.array_equal(got[:120], np.load(os.path.join(GOLDEN, "mocap_bones_880_999.npy")))
    # file-path entry point, and a sub-range read
    dev2 = runtime.DeviceSkeleton(ASF, AMC)
    assert np.array_equal(dev2.bones(7, 3), want[7:10])
    assert dev.fk_ms > 0
    # a long clip (the 121 frames repeated to ~3000, renumbered): every frame block equals the first
    lines = amc.split(b"\n")
    head, body = lines[:3], lines[3:3 + 121 * 30]
    long_amc = b"\n".join(head + body * 25) + b"\n"
    big = runtime.DeviceSkeleton(asf, long_amc)
    assert big.n_frames == 121 * 25
    tab = big.bones()
    assert np.array_equal(tab.reshape(25, 121, 30, 2, 3), np.broadcast_to(want, (25,) + want.shape))


@pytest.mark.gpu
def test_cuda_posed_scene_renders_like_the_reference_bones(oracle_lib):
    from distraytracer_b200 import runtime, scenes, abi
    asf, amc = _clip()
    skel = runtime.DeviceSkeleton(asf, amc)
    for frame in (0, 57, 118):      # the golden table ends at 119, whose velocity needs frame 120
        scene, st = scenes.config4_frame(frame, 160, 90, 4)       # bones from the reference's golden table
        first = next(i for i, p in enumerate(scene.prims) if p.type == abi.PRIM_CYLINDER)
        want, _ = runtime.DeviceScene(scene, 0).render_float(st)
        base, _ = scenes.config4_frame(0, 160, 90, 4)
        dev = runtime.DeviceScene(base, 0)
        dev.pose_skeleton(skel, frame, first, 0.0, True)
        got, _ = dev.render_float(st)
        assert np.array_equal(np.nan_to_num(got), np.nan_to_num(want)), frame
    # two poses (set_velocity 2): each end point heads for its own position at frame + 1
    two, st2 = scenes.config4_frame(57, 160, 90, 4, two_pose=True)
    want2, _ = runtime.DeviceScene(two, 0).render_float(st2)
    dev.pose_skeleton(skel, 57, first, 0.0, 2)
    got2, _ = dev.render_float(st2)
    assert np.array_equal(np.nan_to_num(got2), np.nan_to_num(want2))
    dev.pose_skeleton(skel, 57, first, 0.0, True)
    one2, _ = dev.render_float(st2)
    assert not np.array_equal(np.nan_to_num(one2), np.nan_to_num(got2))    # rotating bones sweep differently than translated ones
    # clamped past the clip, rejected below it and when the target primitives are not cylinders
    dev.pose_skeleton(skel, 10_000, first)
    a, _ = dev.render_float(st)
    dev.pose_skeleton(skel, 120, first)
    b, _ = dev.render_float(st)
    assert np.array_equal(np.nan_to_num(a), np.nan_to_num(b))
    with pytest.raises(runtime.DrtError):
        dev.pose_skeleton(skel, -1, first)
    with pytest.raises(runtime.DrtError):
        dev.pose_skeleton(skel, 0, 0 if first != 0 else len(scene.prims) - 1)
    # drop_y lowers the figure (scene.h:646-650): same as posing, then translating the bones
    dev.pose_skeleton(skel, 3, first, 0.5, False)
    lowered, _ = dev.render_float(st)
    ref_scene, _ = scenes.config4_frame(3, 160, 90, 4)
    for p in ref_scene.prims:
        if p.type == abi.PRIM_CYLINDER:
            p.c1[1] -= 0.5; p.c2[1] -= 0.5; p.center[1] = (p.c1[1] + p.c2[1]) / 2
            p.velocity[:] = [0.0, 0.0, 0.0]
    want, _ = runtime.DeviceScene(ref_scene, 0).render_float(st)
    assert np.array_equal(np.nan_to_num(lowered), np.nan_to_num(want))


@pytest.mark.gpu
def test_cuda_skeleton_rejects_malformed_clips():
    from distraytracer_b200 import runtime, abi
    asf, amc = _clip()
    with pytest.raises(runtime.DrtError) as e:
        runtime.DeviceSkeleton(b"no bone data here\n", amc)
    assert e.value.code == abi.ERR_INVALID
    with pytest.raises(runtime.DrtError):
        runtime.DeviceSkeleton(asf.replace(b"lfemur ltibia", b"lfemur nosuchbone"), amc)
    with pytest.raises(runtime.DrtError):
        runtime.DeviceSkeleton(asf, amc.replace(b"lowerback", b"lowerbach", 1))
    with pytest.raises(runtime.DrtError):
        runtime.DeviceSkeleton(asf, b":FULLY-SPECIFIED\n:DEGREES\n")
    with pytest.raises(runtime.DrtError):
        runtime.DeviceSkeleton("/nonexistent.asf", "/nonexistent.amc")


def _force_3dof(lines):
    """The clip re-written as a :FORCE-ALL-JOINTS-BE-3DOF file: every moving joint carries three rotations, the ones
    the skeleton does not declare appended as zeros (the order enableAllRotationalDOFs gives them)."""
    out = [lines[0], lines[1], b":FORCE-ALL-JOINTS-BE-3DOF", lines[2]]
    for ln in lines[3:3 + 121 * 30]:
        w = ln.split()
        if len(w) > 1 and w[0] != b"root":
            w += [b"0"] * (3 - (len(w) - 1))
        out.append(b" ".join(w))
    return b"\n".join(out) + b"\n"


SYNTH_ASF = b"""# hand-written skeleton: translational and mixed degrees of freedom on inner bones (90.asf has them on the root only),
# a bone without a length line (the reference carries the previous bone's length over), a branching hierarchy
:version 1.10
:name synth
:units
  mass 1.0
  length 0.45
  angle deg
:root
   order TX TY TZ RX RY RZ
   axis XYZ
   position 0 0 0
   orientation 0 0 0
:bonedata
  begin
     id 1
     name hip
     direction 0.6 -0.7 0.387298
     length 2.5
     axis 10 -20 30  XYZ
    dof rx ry rz
  end
  begin
     id 2
     name slider
     direction 0 -1 0
     length 4.25
     axis 0 45 -15  XYZ
    dof tx ty tz rx
  end
  begin
     id 3
     name tip
     direction 0.267261 0.534522 0.801784
     axis -90 5 20  XYZ
  end
  begin
     id 4
     name arm
     direction -1 0 0
     length 3
     axis 0 0 90  XYZ
    dof rz ty
  end
:hierarchy
  begin
    root hip arm
    hip slider
    slider tip
  end
"""


def _synth_amc(n_frames=40):
    rng = np.random.default_rng(7)
    out = [b"# synthetic motion", b":FULLY-SPECIFIED", b":DEGREES"]
    for f in range(n_frames):
        v = rng.uniform(-1, 1, 16)
        out.append(b"%d" % (f + 1))
        out.append(b"root %.6g %.6g %.6g %.6g %.6g %.6g" % (tuple(v[:3] * 20) + tuple(v[3:6] * 180)))
        out.append(b"hip %.6g %.6g %.6g" % tuple(v[6:9] * 120))
        out.append(b"slider %.6g %.6g %.6g %.6g" % (v[9] * 3, v[10] * 3, v[11] * 3, v[12] * 90))
        out.append(b"arm %.6g %.6g" % (v[13] * 170, v[14] * 2))
    return b"\n".join(out) + b"\n"


def _variants():
    asf, amc = _clip()                      # 90.asf has CRLF line ends, the .amc LF
    lines = amc.split(b"\n")
    asf_lf = asf.replace(b"\r\n", b"\n")
    assert asf_lf != asf
    return {
        "fixture": (asf, amc),
        "lf": (asf_lf, amc),
        "crlf": (asf, amc.replace(b"\n", b"\r\n")),                                            # both written on Windows (removeCR)
        "force3dof": (asf, _force_3dof(lines)),                                                  # skeleton.cpp:467-499
        "truncated": (asf, b"\n".join(lines[:3 + 100 * 30 + 7]) + b"\n"),                         # 100 whole frames + 7 stray lines
        # a blank line re-runs the previous keyword on an empty string (sscanf leaves `keyword` alone): harmless after "begin"
        # (after "end" the reference would start a phantom bone and index out of bounds; the library rejects that)
        "blank_lines": (asf_lf.replace(b"  begin\n", b"  begin\n\n"), amc),
        "synthetic": (SYNTH_ASF, _synth_amc()),
    }


@pytest.mark.parametrize("name", ["fixture", "lf", "crlf", "force3dof", "truncated", "blank_lines"])
def test_host_parser_agrees_with_the_oracle_on_structure(oracle_lib, name):
    """The library's host-side ASF/AMC parser (no GPU needed) and the oracle's agree on bones, hierarchy, degrees of
    freedom and the reference's frame-count formula, for the fixture clip and for awkward spellings of it."""
    from distraytracer_b200 import runtime
    from oracle.harness import SkeletonOracle
    asf, amc = _variants()[name]
    nb, nf, parents, dofs = runtime.parse_skeleton(asf, amc)
    orc = SkeletonOracle(asf, amc)
    op, od = orc.structure()
    assert (nb, nf) == (orc.n_cylinders + 1, orc.n_frames)
    assert np.array_equal(parents, op) and np.array_equal(dofs, od)
    assert nb == 31 and parents[0] == -1 and (parents[1:] >= 0).all()
    assert nf == {"truncated": 100}.get(name, 121)         # force3dof: (4 + 121*30 - 3) // 30 is still 121
    if name == "force3dof":
        assert all((d & 7) == 7 for d in dofs if d)        # every moving bone has all three rotations
    else:
        assert dofs[0] == 63 and dofs[3] == 1               # root: 6 DOF; ltibia: rx only


def test_host_parser_rejects_malformed_clips():
    from distraytracer_b200 import runtime, abi
    asf, amc = _clip()
    for bad_asf, bad_amc in [(b"no bone data here\n", amc), (asf.replace(b"lfemur ltibia", b"lfemur nosuchbone"), amc),
                             (asf, amc.replace(b"lowerback", b"lowerbach", 1)), (asf, b":FULLY-SPECIFIED\n:DEGREES\n"),
                             (asf.replace(b"    lfemur ltibia\r\n", b""), amc),
                             (asf.replace(b"  end\r\n", b"  end\r\n\r\n", 1), amc)]:          # phantom bone after a blank line          # ltibia (and its subtree) detached from the root
        with pytest.raises(runtime.DrtError) as e:
            runtime.parse_skeleton(bad_asf, bad_amc)
        assert e.value.code == abi.ERR_INVALID


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lf", "crlf", "force3dof", "truncated", "blank_lines", "synthetic"])
def test_cuda_fk_matches_oracle_on_awkward_clips(oracle_lib, name):
    from distraytracer_b200 import runtime
    from oracle.harness import SkeletonOracle
    asf, amc = _variants()[name]
    dev = runtime.DeviceSkeleton(asf, amc)
    orc = SkeletonOracle(asf, amc)
    assert dev.n_frames == orc.n_frames
    assert np.array_equal(dev.bones(), np.stack([orc.bones(f) for f in range(orc.n_frames)]))


@pytest.mark.parametrize("name", ["lf", "crlf", "force3dof", "truncated", "blank_lines", "synthetic"])
def test_oracle_matches_compiled_reference_on_awkward_clips(oracle_lib, tmp_path, name):
    """Pins the restatement's handling of line ends, :FORCE-ALL-JOINTS-BE-3DOF (enableAllRotationalDOFs), the
    frame-count formula and blank lines on the compiled reference itself: the variant is written out as 90.asf /
    90_16_v3.amc, the reference loads it the way its main() does (fresh process: its mocap state is global).  Without
    oracle/_ref the bones are compared with the reference's, stored as digests."""
    import subprocess
    import sys
    from conftest import ROOT
    from oracle.harness import SkeletonOracle, ref_available
    from conftest import assert_pinned
    asf, amc = _variants()[name]
    orc = SkeletonOracle(asf, amc)
    frames = [0, 1, orc.n_frames // 2, orc.n_frames - 1, orc.n_frames + 5]
    got = np.stack([orc.bones(f) for f in frames])
    live = ref_available()
    if live:
        (tmp_path / "90.asf").write_bytes(asf)
        (tmp_path / "90_16_v3.amc").write_bytes(amc)
        out = tmp_path / "bones.npy"
        code = ("import sys, numpy as np; sys.path.insert(0, %r); from oracle.harness import Ref; "
                "r = Ref(asset_root=%r, mocap=True); np.save(%r, np.stack([r.mocap_bones(f) for f in %r]))"
                % (ROOT, str(tmp_path), str(out), frames))
        subprocess.check_call([sys.executable, "-c", code], stdout=subprocess.DEVNULL)
        assert np.array_equal(got, np.load(out))
    assert_pinned(f"awkward_clips/{name}", got, matched_reference=live)
