"""Per-warp timeline of the traversal launches of one C2 pass (build with -DRTX_TRACE_TIMELINE: python tools/build_variant.py timeline
-DRTX_TRACE_TIMELINE; RTX_B200_LIB=build/variants/timeline.so python tools/pass_timeline.py > out.txt; --analyse out.txt for percentiles)."""
import re
import sys
if len(sys.argv) > 2 and sys.argv[1] == "--analyse":
    import numpy as np
    launches = []
    for l in open(sys.argv[2]):
        if l.startswith("=== pass"):
            launches = []
        m = re.match(r"TL (\d+) n (\d+) start (\d+) exhausted_at (\d+) end (\d+) steps (\d+) drain_steps (\d+)", l)
        if m:
            r = tuple(int(x) for x in m.groups())
            if not launches or launches[-1][0][1] != r[1]:
                launches.append([])
            launches[-1].append(r)
    for k, rows in enumerate(launches):
        b = np.array(rows)
        ex = b[:, 3] / 1e3; en = b[:, 4] / 1e3
        print("launch %d: n = %d rays, %d warps sampled" % (k, b[0, 1], len(b)))
        for nm, v in (("queue found drained at [us]", ex), ("warp finished at [us]", en), ("drain = finished - drained [us]", en - ex), ("steps", b[:, 5]),
                      ("steps after the queue drained", b[:, 6]), ("us per step while draining", (en - ex) / np.maximum(b[:, 6], 1))):
            print("  %-34s min %7.1f  p10 %7.1f  p50 %7.1f  p90 %7.1f  max %7.1f" % (nm, v.min(), np.percentile(v, 10), np.percentile(v, 50), np.percentile(v, 90), v.max()))
    sys.exit(0)
import os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rtdx  # noqa: E402
sc = rtdx.scenes.mesh_room(n=296)
ctx = rtdx.Context(1920, 1080, bounces=6)
ctx.upload_scene(sc)
ctx.set_option(rtdx.OPT_PASS_PARTS, 1)
ctx.render_pass(0, 1); ctx.synchronize()
print("=== pass", flush=True)
ctx.render_pass(1, 1); ctx.synchronize()
