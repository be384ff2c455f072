"""Deforming meshes on BASELINE config C2 (1,051,392-triangle mesh, 1920x1080, depth 8 = bounces 6): what rtx_update_model_device costs
with RTX_UPDATE_REFIT and with RTX_UPDATE_REBUILD, what refitting costs in tree quality (closest-hit traversal time of the same camera and
bounce rays on a tree refitted k times against a tree rebuilt at the same deformation), and the per-frame time of the deforming frame
loop (update_model_device -> set_instances -> set_camera -> render_pass -> read_output_async) against the same loop without the update.
The card's name, power limit and maximum SM clock are read in the same run.
usage: python tools/deform_time.py [--side 296] [--reps 15] [--frames 30] [--out FILE]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import rtdx  # noqa: E402
from util import bounce_rays  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--side", type=int, default=296)
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--bounces", type=int, default=6)
ap.add_argument("--amplitude", type=float, default=0.3)
ap.add_argument("--reps", type=int, default=15)
ap.add_argument("--frames", type=int, default=30)
ap.add_argument("--out", default="")
a = ap.parse_args()
lines = []


def emit(s):
    print(s, flush=True)
    lines.append(s)


q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip()
emit("device: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(0), q))
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream)
sc = rtdx.scenes.mesh_room(n=a.side)
base = sc.models[0]["vertices"]
nv = base.size
emit("scene: %s, model 0: %d vertices, %d triangles; %dx%d, bounces %d" % (sc.name, nv, sc.models[0]["indices"].size // 3, a.width,
                                                                        a.height, a.bounces))


def dev(v):
    return torch.from_numpy(np.ascontiguousarray(v).view(np.uint8)).to("cuda")


def med(x):
    return float(np.median(x))


# ---- 1. the call: REFIT (device events around the call on the context stream) and REBUILD (host clock, it synchronises), alternating
ctx = rtdx.Context(a.width, a.height, bounces=a.bounces, stream=stream.cuda_stream)
up = ctx.upload_scene(sc)
states = [dev(rtdx.scenes.deform(base, 0.1 * k, a.amplitude, seed=1)) for k in range(4)]
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
refit_ms, rebuild_ms, rebuild_dev_ms = [], [], []
for r in range(a.reps + 3):
    s = states[r % 4]
    e0.record(stream); ctx.update_model_device(0, s, nv, rtdx.UPDATE_REFIT); e1.record(stream)
    e1.synchronize()
    if r >= 3:
        refit_ms.append(e0.elapsed_time(e1))
    ctx.synchronize()
    t0 = time.perf_counter()
    e0.record(stream); ctx.update_model_device(0, states[(r + 1) % 4], nv, rtdx.UPDATE_REBUILD); e1.record(stream)
    e1.synchronize()
    if r >= 3:
        rebuild_ms.append((time.perf_counter() - t0) * 1e3); rebuild_dev_ms.append(e0.elapsed_time(e1))
emit("update_model_device REFIT   : median %.3f ms (device events, whole call: vertex copy, attribute records, BLAS refit, instance "
     "boxes, TLAS), min %.3f, max %.3f, %d runs" % (med(refit_ms), min(refit_ms), max(refit_ms), len(refit_ms)))
emit("update_model_device REBUILD : median %.3f ms host wall clock (device events %.3f ms), min %.3f, max %.3f, %d runs"
     % (med(rebuild_ms), med(rebuild_dev_ms), min(rebuild_ms), max(rebuild_ms), len(rebuild_ms)))
emit("REBUILD / REFIT: %.1fx" % (med(rebuild_ms) / med(refit_ms)))
ctx.close()

# ---- 2. tree quality: the same final deformation reached by k refits from the build of the undeformed mesh, against a rebuild there
final = rtdx.scenes.deform(base, 0.5, a.amplitude, seed=2)
cam = up["camera"]
rays = rtdx.scenes.camera_rays(cam, a.width, a.height)
probe = rtdx.Context(64, 64); probe.upload_scene(sc); probe.update_model(0, final, rtdx.UPDATE_REBUILD)
hits = probe.trace(rays)
rays2 = bounce_rays(rtdx, rays, hits, np.random.RandomState(5))
probe.close()
sets = {"camera": rays, "bounce": rays2}
d_rays = {k: torch.from_numpy(np.ascontiguousarray(v).view(np.uint8)).to("cuda") for k, v in sets.items()}
d_hits = {k: torch.empty(v.size * 20, dtype=torch.uint8, device="cuda") for k, v in sets.items()}
torch.cuda.synchronize()


def trace_ms(c):
    out = {}
    for k, v in sets.items():
        for _ in range(2):
            c.trace_device(d_rays[k].data_ptr(), v.size, d_hits[k].data_ptr())
        ts = []
        for _ in range(5):
            e0.record(stream); c.trace_device(d_rays[k].data_ptr(), v.size, d_hits[k].data_ptr()); e1.record(stream)
            e1.synchronize(); ts.append(e0.elapsed_time(e1))
        out[k] = ts
    return out


ctxs = {}
for k in (1, 4, 16):
    c = rtdx.Context(64, 64, stream=stream.cuda_stream); c.upload_scene(sc)
    for j in range(1, k + 1):
        c.update_model(0, rtdx.scenes.deform(base, 0.5 * j / k, a.amplitude * j / k, seed=2), rtdx.UPDATE_REFIT)
    ctxs["refit x%d" % k] = c
c = rtdx.Context(64, 64, stream=stream.cuda_stream); c.upload_scene(sc); c.update_model(0, final, rtdx.UPDATE_REBUILD)
ctxs["rebuild"] = c
res = {name: {"camera": [], "bounce": []} for name in ctxs}
for rnd in range(3):                                    # alternating rounds over the trees
    for name, c in ctxs.items():
        for k, ts in trace_ms(c).items():
            res[name][k] += ts
emit("closest-hit traversal of the final deformation (rtx_trace_device, %d camera rays, %d bounce rays; median of 15 in 3 alternating "
     "rounds):" % (rays.size, rays2.size))
for name in ctxs:
    emit("  %-11s camera %.3f ms (%.2fx rebuild)   bounce %.3f ms (%.2fx rebuild)" % (
        name, med(res[name]["camera"]), med(res[name]["camera"]) / med(res["rebuild"]["camera"]),
        med(res[name]["bounce"]), med(res[name]["bounce"]) / med(res["rebuild"]["bounce"])))
for c in ctxs.values():
    c.close()

# ---- 3. the deforming frame loop against the same loop without the update (host clock per frame, one frame in flight), alternating
ctx = rtdx.Context(a.width, a.height, bounces=a.bounces, stream=stream.cuda_stream)
up = ctx.upload_scene(sc)
pinned = [torch.empty((a.height, a.width, 4), dtype=torch.uint8).pin_memory().numpy() for _ in range(2)]
frame_states = [dev(rtdx.scenes.deform(base, 0.05 * k, a.amplitude, seed=3)) for k in range(8)]
torch.cuda.synchronize()


def loop(n, first, deform):
    for f in range(n):
        if deform:
            ctx.update_model_device(0, frame_states[f % 8], nv)
        ctx.set_instances(up["descs"], up["props"])
        ctx.set_camera(up["camera"])
        ctx.render_pass(first + f, 1)
        if f > 0:
            ctx.wait_output()
        ctx.read_output_async(pinned[f & 1])
    ctx.wait_output()


per = {True: [], False: []}
loop(6, 0, True); loop(6, 0, False)
for rnd in range(3):
    for deform in (True, False):
        ctx.synchronize()
        t0 = time.perf_counter()
        loop(a.frames, 0, deform)
        ctx.synchronize()
        per[deform].append((time.perf_counter() - t0) * 1e3 / a.frames)
emit("frame loop, %d frames per run, 3 alternating runs each (ms per frame): deforming %s (median %.3f), static %s (median %.3f), "
     "difference %.3f ms" % (a.frames, " ".join("%.3f" % x for x in per[True]), med(per[True]), " ".join("%.3f" % x for x in per[False]),
                            med(per[False]), med(per[True]) - med(per[False])))
ctx.close()
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
