"""render_wave's pass statistics on the bench frame.  Needs a library built with -DDRT_PASS_STATS (each CTA prints one
PASS_STATS line at exit); renders frame 0 of bench.py's workload once and sums the lines.
usage: DRT_LIB=variants/libdrt_x.so python tools/pass_stats.py"""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

if len(sys.argv) > 1 and sys.argv[1] == "worker":
    import bench
    from distraytracer_b200 import runtime
    scene, settings = bench.workload()
    settings.frame, settings.seed = 0, 1000
    runtime.DeviceScene(scene, 0).render_float(settings)
    sys.exit(0)

out = subprocess.run([sys.executable, __file__, "worker"], check=True, capture_output=True, text=True).stdout
rows = [list(map(int, l.split()[2:])) for l in out.splitlines() if l.startswith("PASS_STATS ")]
if not rows:
    raise SystemExit("no PASS_STATS lines: is DRT_LIB a -DDRT_PASS_STATS build?")
tot = [sum(c) for c in zip(*rows)]
batches, passes, slots, empty, bites, partial = tot[:6]
hist = tot[6:]
print(f"CTAs {len(rows)}  batches {batches}  passes {passes}  passes per batch {passes / batches:.2f}")
print(f"slots traced {slots}  empty {empty} ({100 * empty / slots:.2f} %)  rays traced {slots - empty}  "
      f"rays per pass {(slots - empty) / passes:.0f}")
print(f"SHADE bites {bites}  per pass {bites / passes:.1f}  partly filled chunks pushed {partial}  per pass {partial / passes:.2f}")
print("rays traced in a TRACE pass | passes | share of passes | share of rays (at the bucket's midpoint)")
mid = [0] + [1.5 * 2 ** (b - 1) for b in range(1, 16)]
w = sum(h * m for h, m in zip(hist, mid))
for b, h in enumerate(hist):
    if h:
        lo, hi = (0, 0) if b == 0 else (2 ** (b - 1), 2 ** b - 1)
        rng = "0" if b == 0 else (f">= {lo}" if b == 15 else f"{lo}-{hi}")
        print(f"  {rng:>12} | {h:8d} | {100 * h / passes:5.1f} % | {100 * h * mid[b] / w:5.1f} %")
