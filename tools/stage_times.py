"""Per-stage device times of C2 passes (CUDA events around every launch; RTX_OPT_STAGE_TIMING).
usage: [RTX_B200_LIB=build/variants/X.so] python tools/stage_times.py [--passes N] [--scene mesh|inst] [--tag T]"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rtdx  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--scene", default="mesh")
ap.add_argument("--side", type=int, default=296)
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--bounces", type=int, default=6)
ap.add_argument("--passes", type=int, default=8)
ap.add_argument("--flags", type=int, default=0)
ap.add_argument("--tag", default="")
ap.add_argument("--opt", action="append", default=[], help="engine option NAME=VALUE (rtdx.OPT_<NAME>), e.g. PASS_PARTS=1 PASS_GRAPH=0")
a = ap.parse_args()
sc = rtdx.scenes.mesh_room(n=a.side) if a.scene == "mesh" else (rtdx.scenes.instanced_blobs() if a.scene == "inst" else rtdx.scenes.cornell())
ctx = rtdx.Context(a.width, a.height, bounces=a.bounces, flags=a.flags)
ctx.upload_scene(sc)
for o in a.opt:
    k, v = o.split("=")
    ctx.set_option(getattr(rtdx, "OPT_" + k), int(v, 0))
for p in range(3):
    ctx.render_pass(p, 1)
ctx.synchronize()
ctx.reset_counters(); ctx.set_option(rtdx.OPT_TRACE_STATS, 1)
ctx.render_pass(0, 1); ctx.synchronize()
s0 = ctx.counters(); ctx.set_option(rtdx.OPT_TRACE_STATS, 0)
nc = max(s0["closest_rays"], 1)
stats = "N/ray node %.2f tri %.2f inst %.2f" % (s0["nodes_visited"] / nc, s0["tris_tested"] / nc, s0["instances_entered"] / nc)
ctx.set_option(rtdx.OPT_STAGE_TIMING, 1)
ctx.reset_counters()
acc, tot = {}, 0.0
for p in range(a.passes):
    ctx.render_pass(3 + p, 1)
    k, t = ctx.last_pass_stage_ms()
    tot += t
    for n, v in k.items():
        acc[n] = acc.get(n, 0.0) + v
c = ctx.counters()
rays = c["closest_rays"] + c["shadow_rays"]
tag = a.tag or os.environ.get("RTX_B200_LIB", "default")
print("%-28s pass %.3f ms  %.0f Mrays/s | " % (tag, tot / a.passes, rays / tot / 1e3) +
      "  ".join("%s %.3f" % (n, v / a.passes) for n, v in acc.items() if v > 0) + " | " + stats, flush=True)
