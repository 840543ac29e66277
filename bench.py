#!/usr/bin/env python
"""bench.py -- throughput of the distributed ray-tracing hot path.

Workload (BASELINE.json configs[1]): the reference's checkertexture scene at 1920x1080,
64 spp, with depth of field, glossy reflection, rectangle-light soft shadows and glass
refraction (distraytracer_b200.scenes.config2).  One "step" = one full frame
(132.7 M camera samples).  With N GPUs every rank renders its own frames (frames sharded
across ranks, no data-path collective): weak scaling.

  value : whole-job Msamples/s with the scene already resident in HBM, device-timed
          (CUDA events on the launching stream inside libdrt.so, max over ranks).
  e2e   : the same metric through drt_render() with HOST buffers: per step the scene
          primitives are re-uploaded (drt_scene_update_prims, H2D) and the finished
          u8 frame is copied back (D2H), host wall clock around the calls.
  roofline : the FP pipe (what bounds the path, SURVEY.md 8d): algorithmic ops from the kernel's own
          event counters x the 8(d) cost table / live step time, against SMs x 64 DFMA x 2 x observed clock.
          `traffic` and the instruction count of roofline_issue come from the committed ncu launch list of this
          same command (profiles/current_launch_metrics.json, written by tools/launch_metrics.py with a hash of the
          kernel sources); they are marked "stale" when the sources have changed since.
  configs : after the timed region, the other BASELINE configurations on one GPU (C1, C3, C5 device-timed,
          C4 as a 120-frame video through the mocap skeleton path, wall clock).
  tiles : (N > 1) ONE frame of C2 / C3 / C5 cut across the N GPUs of the box (strong scaling of the
          single-frame path), driven by rank 0 after the frame-sharded legs.
  --dump-outputs DIR : DIR/frame_r<rank>.npy, the frame each rank's e2e leg received in its last timed step (float32
          copy of the u8 frame; a fixed seeded pixel sample where N full frames would pass 64 MB).  Frames and seeds depend
          only on --gpus / --warmup / --steps, so two builds run with the same arguments can be compared pixel for pixel.
  --impl reference : the reference's own CPU renderer (oracle/_ref, the unmodified
          reference sources compiled here) on all host cores, one process per core on
          a fixed stratified sample of the same frame.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

XRES, YRES, SPP = 1920, 1080, 64
METRIC = "samples_per_s_1080p_64spp"
UNIT = "Msamples/s"

# algorithmic cost table, SURVEY.md 8(d): FP32-equivalent ops per event
COST = {"node": 20, "sphere": 32, "triangle": 52, "rectangle": 36, "cylinder": 70, "shade": 110, "ray": 60}

# the fixed stratified CPU sample both CPU legs time (cpu_baseline and --impl reference): rows x segments x pixels
CPU_ROWS, CPU_SEGS, CPU_SEG_PX = 32, 8, 30


def workload():
    from distraytracer_b200 import scenes
    scene, settings = scenes.config2(XRES, YRES, SPP)
    return scene, settings


def config_dict(n_gpus):
    return {
        "workload": "configs[1]: checkertexture scene 1920x1080 64spp, DOF aperture 0.2 / focal 10, glossy floor+doors, "
                    "rectangle-light soft shadows, glass block (Fresnel refraction), max_depth 10, brdf_samples 2",
        "samples_per_step": XRES * YRES * SPP,
        "partition": f"frames round-robin over {n_gpus} rank(s), no collective; scene replicated",
        "precision": "reference: f64 vectors, f32 scalar temporaries where the reference narrows, no FMA contraction",
        "l2": "working set is the 2.1 GB per-frame sample buffer (> 126 MB L2); no explicit flush",
    }


def source_hash():
    """Hash of everything that decides the kernels' machine code: profiles/current_launch_metrics.json carries the hash
    of the build it was captured from."""
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "distraytracer_b200", "csrc")
    for f in sorted(os.listdir(csrc)):
        h.update(f.encode()); h.update(open(os.path.join(csrc, f), "rb").read())
    h.update(open(os.path.join(ROOT, "include", "drt.h"), "rb").read())
    return h.hexdigest()[:16]


def launch_metrics():
    """ncu counters of the render_wave launch of one bench step, from the committed launch list."""
    try:
        m = json.load(open(os.path.join(ROOT, "profiles", "current_launch_metrics.json")))
    except Exception:
        return None
    m["stale"] = m.get("source_hash") != source_hash()
    return m


# ---------------------------------------------------------------------------
# clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.dev = device_index

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if p[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(mx))
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


# ---------------------------------------------------------------------------
# CPU reference leg
_WORKER = {}


def _ref_worker(args):
    """One task = one segment of one row of the frame on one reference renderer instance (the reference is not
    thread-safe: one process per core, state cached per process)."""
    scene_npz, settings_bytes, y0, x0, x1, use_ref = args
    y1 = y0 + 1
    if "st" not in _WORKER:
        sys.path.insert(0, ROOT)
        from distraytracer_b200.scene import Scene, settings_from_bytes
        import numpy as _np
        scene = Scene.from_npz_dict(_np.load(scene_npz))
        st = settings_from_bytes(settings_bytes)
        _WORKER["st"] = st
        if use_ref:
            from oracle.harness import Ref
            r = Ref()
            r.load(scene)
            r.set_settings(st)
            r.rng(0)                  # the reference's own mt19937 / random_device draws
            _WORKER["ref"] = r
        else:
            from oracle.harness import Oracle
            _WORKER["oracle"] = Oracle(scene)
    st = _WORKER["st"]
    if use_ref:
        _, _, sec = _WORKER["ref"].render_loop(st.frame, y0, y1, reset_policy=0, seed=0, x0=x0, x1=x1)
    else:
        from oracle.harness import ORACLE_KEYED
        from distraytracer_b200 import abi
        _, _, _, sec = _WORKER["oracle"].render(st, abi.Tile(x0, y0, x1 - x0, y1 - y0, 0), mode=ORACLE_KEYED)
    return sec


class CpuReference:
    """Times the reference's CPU implementation on a bounded, FIXED sample of the frame -- CPU_ROWS rows evenly spaced
    over the height and in each row CPU_SEGS segments of CPU_SEG_PX pixels evenly spaced over the width, so that sky,
    floor, doors and glass are all sampled -- the same sample whatever the core count and whichever leg
    (cpu_baseline or --impl reference) runs it."""

    def __init__(self, scene, settings):
        import multiprocessing as mp
        from oracle.harness import ref_available
        from distraytracer_b200.scene import settings_to_bytes
        self.cores = os.cpu_count() or 1
        self.kind = "reference" if ref_available() else "port"
        self.tmp = tempfile.mktemp(suffix=".npz")
        np.savez(self.tmp, **scene.to_npz_dict())
        self.settings = settings
        self.sbytes = settings_to_bytes(settings)
        self.pool = mp.get_context("spawn").Pool(self.cores)
        ys = np.linspace(0, settings.yRes - 1, CPU_ROWS).astype(int)
        xs = np.linspace(0, settings.xRes - CPU_SEG_PX, CPU_SEGS).astype(int)
        # (row, segment) tasks are handed out dynamically (some pixels cost 1000x others: glass + glossy ray trees)
        self.bands = [(int(y), int(x), int(x) + CPU_SEG_PX) for y in ys for x in xs]
        self.samples = len(self.bands) * CPU_SEG_PX * (int(np.sqrt(settings.antialias_samples)) ** 2)

    def _run(self, bands):
        t0 = time.perf_counter()
        list(self.pool.imap_unordered(_ref_worker, [(self.tmp, self.sbytes, y, a, b, self.kind == "reference")
                                                    for y, a, b in bands], chunksize=1))
        return time.perf_counter() - t0

    def warm(self):
        """Untimed: every worker process loads the scene and renders a few pixels."""
        self._run([(0, x, x + 2) for x in range(0, 4 * self.cores, 2)])

    def step(self):
        return self._run(self.bands)

    def close(self):
        self.pool.close(); self.pool.join()
        try:
            os.unlink(self.tmp)
        except OSError:
            pass

    def describe(self):
        return (f"stratified sample of the {self.settings.xRes}x{self.settings.yRes} {SPP}spp frame: {CPU_ROWS} rows x {CPU_SEGS} segments "
                f"of {CPU_SEG_PX} px = {self.samples} samples per step, {len(self.bands)} tasks over {self.cores} processes "
                f"(one per core); "
                + ("oracle/_ref (unmodified reference sources, its own RNG)" if self.kind == "reference"
                   else "oracle/ C++ restatement (reference tree not built)"))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    scene, settings = workload()
    ref = CpuReference(scene, settings)
    ref.warm()
    for _ in range(args.warmup):
        ref.step()
    t = 0.0
    for _ in range(args.steps):
        t += ref.step()
    ref.close()
    value = ref.samples * args.steps / t / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args.gpus),
        "frames_per_s": value * 1e6 / (XRES * YRES * SPP),
        "ms_per_frame_extrapolated": 1e3 * (XRES * YRES * SPP) / (value * 1e6),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores, "kind": ref.kind, "sample": ref.describe()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------
# the other BASELINE configurations (after the timed region)
def _device_timed(dev, st, reps=2):
    from distraytracer_b200 import abi
    cnt = abi.Counters()
    ms = []
    for _ in range(reps + 1):
        dev.render_device(st, None, cnt)
        ms.append(cnt.kernel_ms)
    spp = int(np.sqrt(st.antialias_samples)) ** 2
    n = st.xRes * st.yRes * spp
    best = min(ms[1:])
    return {"res": [st.xRes, st.yRes], "spp": spp, "samples": n, "ms": best, "Msamples_per_s": n / best / 1e3,
            "frames_per_s": 1e3 / best, "launches": cnt.kernel_launches, "kernel_variant": cnt.kernel_variant, "timing": "device (CUDA events), best of 2 after 1 warm-up"}


def run_configs(local):
    """C1, C3, C5 device-timed on one GPU; C4 = the 120-frame mocap video end to end (skeleton path)."""
    from distraytracer_b200 import runtime, abi, scenes
    out = {}

    def guarded(tag, fn):
        t0 = time.perf_counter()
        try:
            out[tag] = fn()
        except Exception as e:      # noqa: BLE001 -- the headline numbers above stand on their own
            out[tag] = {"error": f"{type(e).__name__}: {e}"}
        out[tag]["wall_s"] = round(time.perf_counter() - t0, 2)

    def static(builder, what):
        def f():
            scene, st = builder()
            dev = runtime.DeviceScene(scene, local)
            r = _device_timed(dev, st)
            dev.close()
            r["workload"] = what
            return r
        return f

    guarded("C1", static(scenes.config1, "configs[0]: checkertexture 640x480 1 spp, aperture 0"))
    guarded("C3", static(scenes.config3, "configs[2]: Oren-Nayar spheres + value-noise cloud background, 1080p 256 spp, one GPU"))
    guarded("C5", static(scenes.config5, "configs[4]: 999 698-triangle textured terrain (device-built LBVH), DOF + motion blur, 3840x2160 64 spp, one GPU"))

    def c4():
        n_frames, xres, yres, spp = 120, 1920, 1080, 16
        t0 = time.perf_counter()
        skel = runtime.DeviceSkeleton(scenes.data_path("mocap_90.asf"), scenes.data_path("mocap_90_16_frames880_1000.amc"), device=local)
        t_load = time.perf_counter() - t0
        scene, st = scenes.config4_frame(0, xres, yres, spp)
        first = next(i for i, p in enumerate(scene.prims) if p.type == abi.PRIM_CYLINDER)
        dev = runtime.DeviceScene(scene, local)
        import torch
        frame = torch.empty((yres, xres, 3), dtype=torch.uint8).pin_memory().numpy()
        cnt = abi.Counters()
        kernel_ms = 0.0

        def one(f):
            st.frame = f; st.seed = 1000 + f
            dev.pose_skeleton(skel, f, first)
            dev.render(st, out=frame, counters=cnt)
            return cnt.kernel_ms

        for f in range(3):
            one(f)
        t0 = time.perf_counter()
        for f in range(n_frames):
            kernel_ms += one(f)
        dt = time.perf_counter() - t0
        dev.close(); skel.close()
        n = xres * yres * spp
        return {"workload": f"configs[3]: ASF/AMC mocap clip, {n_frames}-frame motion-blurred video {xres}x{yres} {spp} spp, velocity blur, "
                            "per frame drt_scene_pose_skeleton + drt_render into a pinned host frame, one GPU",
                "frames": n_frames, "frames_per_s": n_frames / dt, "ms_per_frame": 1e3 * dt / n_frames, "kernel_ms_per_frame": kernel_ms / n_frames,
                "Msamples_per_s": n * n_frames / dt / 1e6, "skeleton_load_s": t_load, "fk_kernel_ms": skel.fk_ms,
                "kernel_variant": cnt.kernel_variant, "timing": "host wall clock around the 120 frames (H2D pose + kernels + D2H frame)"}

    guarded("C4", c4)
    return out


def run_tiles(n_gpus):
    """ONE frame cut across the GPUs of the box, rank 0 driving all of them (the other ranks are idle by now):
    wall ms per frame at 1 GPU and at N, speed-up, image identity."""
    from distraytracer_b200 import runtime, scenes, shard
    import torch
    out = {}
    for tag, builder in (("C2", lambda: workload()), ("C3", scenes.config3), ("C5", scenes.config5)):
        t_all = time.perf_counter()
        try:
            scene, st = builder()
            frame = torch.empty((st.yRes, st.xRes, 3), dtype=torch.uint8).pin_memory().numpy()
            spp = int(np.sqrt(st.antialias_samples)) ** 2
            samples = st.xRes * st.yRes * spp
            group = shard.FrameGroup(scene, list(range(n_gpus)))
            try:
                group.render(st, frame, gpus=n_gpus)
            except runtime.DrtError as e:
                if e.code != -2:                                        # DRT_ERR_UNSUPPORTED: no peer access on this box
                    raise
                group.close()
                group = shard.FrameGroup(scene, list(range(n_gpus)), method="blocks")
            res = {"res": [st.xRes, st.yRes], "spp": spp, "method": group.method}
            ref = None
            for use in (1, n_gpus):
                group.render(st, frame, gpus=use)                        # warm-up: scratch allocation, clocks
                dt = min(group.render(st, frame, gpus=use) for _ in range(2))
                if use == 1:
                    ref, t1 = frame.copy(), dt
                    res["ms_1gpu"] = 1e3 * dt
                else:
                    res.update({"gpus": use, "ms": 1e3 * dt, "frames_per_s": 1 / dt, "Msamples_per_s": samples / dt / 1e6,
                                "speedup_vs_1gpu": t1 / dt, "efficiency": t1 / dt / use,
                                "same_image_as_1gpu": bool(np.array_equal(ref, frame))})
            group.close()
            out[tag] = res
        except Exception as e:      # noqa: BLE001
            out[tag] = {"error": f"{type(e).__name__}: {e}"}
        out[tag]["wall_s"] = round(time.perf_counter() - t_all, 2)
    out["timing"] = "host wall clock around one whole frame (launch on every GPU -> gathered u8 frame in pinned host memory), best of 2 after 1 warm-up"
    return out


# ---------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from distraytracer_b200 import runtime, abi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or runtime.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: distraytracer_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    host_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
        # host-side rendezvous for the end of the run: an NCCL barrier would leave a spinning kernel on the GPUs rank 0
        # is about to use for the single-frame (tiles) leg
        host_group = dist.new_group(backend="gloo")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    scene, settings = workload()
    dev = runtime.DeviceScene(scene, local)
    tile = abi.Tile(0, 0, settings.xRes, settings.yRes, local)
    samples_per_step = XRES * YRES * SPP
    frame_bytes = XRES * YRES * 3
    host_frame = torch.empty((YRES, XRES, 3), dtype=torch.uint8).pin_memory().numpy()
    prims = list(scene.prims)

    from distraytracer_b200 import shard
    my_frames = shard.frames_for_rank(rank, world, (args.warmup + args.steps) * world)

    def set_frame(step):
        # frames are sharded round-robin (SURVEY.md 8e): rank r renders frames r, r+world, ...
        settings.frame = my_frames[step]
        settings.seed = 1000 + settings.frame

    # ---- device-resident leg (value) ------------------------------------------------
    cnt = abi.Counters()
    for w in range(args.warmup):
        set_frame(w)
        dev.render_device(settings, tile, cnt)
    clocks = ClockSampler(local) if rank == 0 else None
    barrier()
    if clocks:
        clocks.start()
    t_wall0 = time.perf_counter()
    dev_ms, launches = 0.0, 0
    for k in range(args.steps):
        set_frame(args.warmup + k)
        dev.render_device(settings, tile, cnt)          # synchronises its stream; kernel_ms from CUDA events
        dev_ms += cnt.kernel_ms
        launches += cnt.kernel_launches
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t_wall0)
    clock_info = clocks.stop() if clocks else None
    variant = cnt.kernel_variant

    # ---- end-to-end leg (e2e): host buffers in, host frame out ----------------------
    for w in range(min(args.warmup, 2)):
        dev.update_prims(prims); dev.render(settings, tile, out=host_frame)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        set_frame(args.warmup + k)
        dev.update_prims(prims)                          # H2D: the frame's primitives
        dev.render(settings, tile, out=host_frame)       # kernels + D2H of the u8 frame
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    if args.dump_outputs:
        # the device-resident leg's last step rendered the same frame and seed into device memory only
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, f"frame_r{rank}.npy"), dump_sample(host_frame, world))

    def maxr(x):
        return shard.max_over_ranks(x, dist if world > 1 else None, device="cuda")

    dev_ms, wall_ms, e2e_ms = maxr(dev_ms), maxr(wall_ms), maxr(e2e_ms)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=host_group)                   # every rank's GPU is idle from here on

    if rank == 0:
        total = samples_per_step * args.steps * world
        value = total / (dev_ms * 1e-3) / 1e6
        e2e_value = total / (e2e_ms * 1e-3) / 1e6
        step_s = dev_ms * 1e-3 / args.steps
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_dict(world),
            "frames_per_s": value * 1e6 / samples_per_step,
            "wall_ms_per_step": wall_ms / args.steps,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_scene_bytes(dev, scene)),
                    "d2h_bytes_per_step": frame_bytes, "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": launches,
            "kernel_variant": variant,
            "clocks": clock_info,
        }
        if not args.no_extras:
            line.update(roofline_blocks(dev, settings, tile, step_s, clock_info, local, launches, args.steps))
            # informational: the same frame through the single-precision build of the kernels (settings.precision = FP32;
            # passes the <= 1/255 on >= 99.9 % of pixels bar on every fixture except the degenerate boundary scene)
            try:
                s32 = abi.copy_struct(settings); s32.precision = abi.PRECISION_FP32
                c32 = abi.Counters()
                dev.render_device(s32, tile, c32); dev.render_device(s32, tile, c32)
                line["fp32_variant"] = {"value": samples_per_step / (c32.kernel_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": c32.kernel_ms,
                                        "note": "one GPU, device-timed, not the headline: the headline runs in the reference's precision"}
            except Exception as e:      # noqa: BLE001
                line["fp32_variant"] = {"error": str(e)}
        dev.close()
        if not args.no_extras:
            line["configs"] = run_configs(local)
            if world > 1:
                line["tiles"] = run_tiles(world)
        if world == 1 and not args.no_cpu_baseline:
            ref = CpuReference(scene, settings)
            ref.warm()
            sec = ref.step()
            ref.close()
            line["cpu_baseline"] = {"value": ref.samples / sec / 1e6, "unit": UNIT, "cores": ref.cores, "kind": ref.kind,
                                    "sample": ref.describe(), "seconds": sec}
        print(json.dumps(line))
    if world > 1:
        dist.barrier(group=host_group)
        dist.destroy_process_group()
    return 0


def roofline_blocks(dev, settings, tile, step_s, clock_info, local, launches, steps):
    """roofline (FP pipe, live), roofline_hbm and roofline_issue (live time over counters of the committed ncu launch list)."""
    import torch
    from distraytracer_b200 import abi
    samples_per_step = XRES * YRES * SPP
    frame_bytes = XRES * YRES * 3
    # one untimed instrumented frame for the roofline accounting
    c2 = abi.Counters(); c2.collect = 1
    events_note = None
    try:
        dev.render_device(settings, tile, c2)
    except Exception as e:      # noqa: BLE001 -- the timed numbers stand on their own; report the accounting as missing
        c2 = abi.Counters(); events_note = f"instrumented frame failed: {e}"
    pt = list(c2.prim_tests)
    ops = (c2.node_tests * COST["node"] + pt[abi.PRIM_SPHERE] * COST["sphere"] + pt[abi.PRIM_TRIANGLE] * COST["triangle"]
           + pt[abi.PRIM_RECTANGLE] * COST["rectangle"] + pt[abi.PRIM_CYLINDER] * COST["cylinder"]
           + c2.shade_evals * COST["shade"] + (c2.rays + c2.shadow_rays) * COST["ray"])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    sm_mhz = (clock_info or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
    props = torch.cuda.get_device_properties(local)
    sms = props.multi_processor_count
    fp64_peak = sms * 64 * 2 * sm_mhz * 1e6 / 1e12      # TFLOP/s at the observed clock
    fp32_peak = sms * 128 * 2 * sm_mhz * 1e6 / 1e12
    # algorithmic bytes per frame: 16 B sample record written by render_wave and read once by resolve, plus the
    # 3 B/pixel frame (SURVEY.md 8d: the scene itself lives in L1/shared memory)
    alg_bytes = samples_per_step * 32 + frame_bytes
    wave_launches_per_step = max(1, launches // max(1, steps) // 2)      # render_wave + resolve per row chunk
    lm = launch_metrics()
    usable = bool(lm) and wave_launches_per_step == int(lm.get("wave_launches_per_step", 1))
    traffic = int(lm["dram_bytes_read"] + lm["dram_bytes_write"]) if usable else None
    prof = None
    if lm:
        prof = {k: lm.get(k) for k in ("source", "source_hash", "commit", "kernel", "stale")}
        if not usable:
            prof["unusable"] = "this run cuts a step into a different number of render_wave launches than the profiled one"
    achieved = ops / step_s / 1e12
    out = {
        "roofline": {"bound": "fp_pipe", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
                     "traffic": traffic, "traffic_from_profile": prof,
                     "frac_of_fp32_peak": achieved / fp32_peak, "fp32_peak": fp32_peak,
                     "note": events_note or "kernel render_wave<double>: the path is issue/latency bound in the FP64 + ALU pipes, not HBM bound "
                             "(SURVEY.md 8d). achieved = algorithmic ops of the launch (the kernel's own event counters x the 8(d) cost "
                             "table, counted on an extra untimed frame) / its device time (CUDA events on the library's stream); "
                             "peak = SMs x 64 DFMA x 2 x observed SM clock (the reference precision computes in f64); traffic = DRAM "
                             "bytes of the launch from the committed ncu launch list",
                     "events": {"samples": c2.samples, "rays": c2.rays, "shadow_rays": c2.shadow_rays, "node_tests": c2.node_tests,
                                "rect_tests": pt[abi.PRIM_RECTANGLE], "sphere_tests": pt[abi.PRIM_SPHERE],
                                "tri_tests": pt[abi.PRIM_TRIANGLE], "cyl_tests": pt[abi.PRIM_CYLINDER], "shade_evals": c2.shade_evals}},
        "roofline_hbm": {"bound": "hbm", "achieved": alg_bytes / step_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": alg_bytes / step_s / 1e9 / hbm_peak, "traffic": traffic,
                         "traffic_gbs": (traffic / step_s / 1e9) if traffic else None,
                         "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                         "note": "secondary: algorithmic bytes (16 B sample record written + read, 3 B/pixel frame) over the live step time; "
                                 "the measured DRAM traffic above them is the CTA ray pools and hit buffers streaming through L2/HBM"},
    }
    if usable and lm.get("inst_executed"):
        inst = float(lm["inst_executed"])
        out["roofline_issue"] = {"bound": "warp_issue", "achieved": inst / step_s / 1e9, "peak": sms * 4 * sm_mhz * 1e6 / 1e9,
                                 "unit": "Gwarp-inst/s", "frac": inst / step_s / (sms * 4 * sm_mhz * 1e6),
                                 "inst_executed": inst, "from_profile": prof,
                                 "note": "warp instructions of the launch (ncu smsp__inst_executed.sum, committed launch list) over the live step "
                                         "time; peak = SMs x 4 schedulers x observed SM clock"}
    return out


DUMP_BYTES = 64 << 20


def dump_sample(frame, world):
    """The frame as float32 (h, w, 3); when the frames of all ranks would exceed DUMP_BYTES, the same seeded sample of
    pixels on every rank instead, as float32 (n, 3) in ascending row-major pixel order."""
    f = frame.astype(np.float32)
    budget = (DUMP_BYTES - 4096 * world) // world
    if f.nbytes <= budget:
        return f
    keep = np.sort(np.random.default_rng(0).choice(f.shape[0] * f.shape[1], budget // (3 * 4), replace=False))
    return f.reshape(-1, 3)[keep]


def h2d_scene_bytes(dev, scene):
    """Bytes drt_scene_update_prims uploads per call (both precisions' geom/prim/node/light tables
    are small; counted from the POD input the host hands over)."""
    import ctypes as C
    from distraytracer_b200 import abi
    return len(scene.prims) * C.sizeof(abi.Prim)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="only the timed legs (A/B runs, ncu launch lists)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write each rank's frame of the last timed step as DIR/frame_r<rank>.npy (float32, PPM row order)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference leg times a sample of the frame and keeps no image")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
