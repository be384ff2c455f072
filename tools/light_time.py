"""The emissive-triangle list built on the device (rtx_collect_emissive_triangles) against the host path (read the deformed vertices
back, rtdx.collect_emissive_triangles, rtx_set_emissive_triangles), on Cornell, the garage + monke fixture, one 10k-triangle emissive
blob, BASELINE config C3 (504,600 records) and C2's mesh with emissive materials:
  - the steady-state call (after an update_model_device refit of the emissive model): device events around the call;
  - the count-changing call (the first one after rtx_set_materials, which rebuilds the emissive index and synchronises): host clock;
  - the host path, each step on the host clock;
and the per-frame loop update_model_device -> collect -> set_instances -> set_camera -> render_pass -> read_output_async on C3 at
1920x1080 against the same loop with the host path.  The card's name, power limit and maximum SM clock are read in the same run.
usage: python tools/light_time.py [--reps 15] [--frames 20] [--out FILE]"""
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
from deform_util import with_vertices  # noqa: E402
from util import load_scene_npz  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=15)
ap.add_argument("--frames", type=int, default=20)
ap.add_argument("--width", type=int, default=1920)
ap.add_argument("--height", type=int, default=1080)
ap.add_argument("--out", default="")
a = ap.parse_args()
lines = []


def emit(s):
    print(s, flush=True)
    lines.append(s)


def med(x):
    return float(np.median(x))


q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip()
emit("device: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(0), q))
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream)


def emissive_model(sc):
    """the model of the most emissive records (the one a deforming emitter would be)"""
    lights = rtdx.collect_emissive_triangles(sc)
    inst = np.bincount(lights["instanceID"], minlength=len(sc.instances))
    per_model = np.zeros(len(sc.models))
    for i, (m, _) in enumerate(sc.instances):
        per_model[m] += inst[i]
    return int(np.argmax(per_model))


def c2_emissive():
    sc = rtdx.scenes.mesh_room()
    mats = sc.materials.copy()
    mats["Ke"][1:9] = (2.0, 2.0, 2.0)           # the eight PBR materials of the mesh
    sc.materials = mats
    return sc


SCENES = [("cornell", rtdx.scenes.cornell),
          ("garage+monke", lambda: load_scene_npz(rtdx, os.path.join(ROOT, "tests", "golden", "reference_scene.npz"))),
          ("emissive blob 10k", lambda: rtdx.scenes.instanced_blobs(n_models=1, lattice=1, emissive_fraction=1.0)),
          ("C3 defaults", rtdx.scenes.instanced_blobs),
          ("C2 mesh emissive", c2_emissive)]

e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
emit("per scene: median over %d runs (ms)" % a.reps)
for name, make in SCENES:
    sc = make()
    m = emissive_model(sc)
    base = sc.models[m]["vertices"]
    states = [rtdx.scenes.deform(base, 0.1 * k, 0.02, seed=1) for k in range(4)]
    dev = [torch.from_numpy(np.ascontiguousarray(v).view(np.uint8).copy()).cuda() for v in states]
    ctx = rtdx.Context(64, 64, stream=stream.cuda_stream)
    ctx.upload_scene(sc)
    n = ctx.collect_emissive_triangles()
    torch.cuda.synchronize()
    steady, changing, readback, host_collect, host_set = [], [], [], [], []
    for r in range(a.reps + 2):
        ctx.update_model_device(m, dev[r % 4], base.size)
        e0.record(stream); ctx.collect_emissive_triangles(); e1.record(stream)
        e1.synchronize()
        ctx.set_materials(sc.materials)
        ctx.synchronize()
        t0 = time.perf_counter(); ctx.collect_emissive_triangles(); ctx.synchronize(); t1 = time.perf_counter()
        # the host path for the same deformed state
        t2 = time.perf_counter()
        v = dev[r % 4].cpu().numpy().view(rtdx.vertex_dt)
        t3 = time.perf_counter()
        lights = rtdx.collect_emissive_triangles(with_vertices(sc, m, v))
        t4 = time.perf_counter()
        ctx.set_emissive_triangles(lights)
        t5 = time.perf_counter()
        if r >= 2:
            steady.append(e0.elapsed_time(e1)); changing.append((t1 - t0) * 1e3)
            readback.append((t3 - t2) * 1e3); host_collect.append((t4 - t3) * 1e3); host_set.append((t5 - t4) * 1e3)
    host = med(readback) + med(host_collect) + med(host_set)
    emit("  %-18s %8d records: device steady %.3f (min %.3f, max %.3f) | count-changing (index rebuild) %.3f | host path %.3f = "
         "vertex read-back %.3f + collect %.3f + set %.3f | host / device steady %.1fx"
         % (name, n, med(steady), min(steady), max(steady), med(changing), host, med(readback), med(host_collect), med(host_set),
            host / med(steady)))
    ctx.close()

# ---- the per-frame loop of a deforming emitter on C3, device list against host list (host clock per frame, one frame in flight)
sc = rtdx.scenes.instanced_blobs()
m = emissive_model(sc)
base = sc.models[m]["vertices"]
ctx = rtdx.Context(a.width, a.height, stream=stream.cuda_stream)
up = ctx.upload_scene(sc)
pinned = [torch.empty((a.height, a.width, 4), dtype=torch.uint8).pin_memory().numpy() for _ in range(2)]
frame_states = [torch.from_numpy(rtdx.scenes.deform(base, 0.05 * k, 0.02, seed=3).view(np.uint8).copy()).cuda() for k in range(8)]
torch.cuda.synchronize()


def loop(n, device):
    for f in range(n):
        ctx.update_model_device(m, frame_states[f % 8], base.size)
        if device:
            ctx.collect_emissive_triangles()
        else:
            v = frame_states[f % 8].cpu().numpy().view(rtdx.vertex_dt)
            ctx.set_emissive_triangles(rtdx.collect_emissive_triangles(with_vertices(sc, m, v)))
        ctx.set_instances(up["descs"], up["props"])
        ctx.set_camera(up["camera"])
        ctx.render_pass(f, 1)
        if f > 0:
            ctx.wait_output()
        ctx.read_output_async(pinned[f & 1])
    ctx.wait_output()


per = {True: [], False: []}
loop(4, True); loop(4, False)
for rnd in range(3):
    for device in (True, False):
        ctx.synchronize()
        t0 = time.perf_counter()
        loop(a.frames, device)
        ctx.synchronize()
        per[device].append((time.perf_counter() - t0) * 1e3 / a.frames)
emit("C3 frame loop %dx%d, bounces 3, %d frames per run, 3 alternating runs (ms per frame): device list %s (median %.3f), host list %s "
     "(median %.3f)" % (a.width, a.height, a.frames, " ".join("%.3f" % x for x in per[True]), med(per[True]),
                        " ".join("%.3f" % x for x in per[False]), med(per[False])))
ctx.close()
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
