"""Whole-pass device time of a bench scene (CUDA events around N passes on the engine's stream; no per-launch events, so the pass runs with
its concurrent parts).  usage: python tools/pass_time.py [--opt PASS_PARTS=k] [--scene mesh|inst] [--passes N] [--tag T]"""
import argparse
import os
import sys

import torch

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
ap.add_argument("--spp", type=int, default=1, help="samples per pass (paths in flight = W*H*spp)")
ap.add_argument("--refit", type=int, default=0, help="call rtx_set_instances this many times after the upload (TLAS refit)")
ap.add_argument("--tag", default="")
ap.add_argument("--opt", action="append", default=[], help="engine option NAME=VALUE (rtdx.OPT_<NAME>), e.g. PASS_PARTS=1 PASS_GRAPH=0")
a = ap.parse_args()
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream)
sc = rtdx.scenes.mesh_room(n=a.side) if a.scene == "mesh" else rtdx.scenes.instanced_blobs()
ctx = rtdx.Context(a.width, a.height, bounces=a.bounces, flags=a.flags, samples_per_pass=a.spp, stream=stream.cuda_stream)
up = ctx.upload_scene(sc)
for o in a.opt:
    k, v = o.split("=")
    ctx.set_option(getattr(rtdx, "OPT_" + k), int(v, 0))
for _ in range(a.refit):
    ctx.set_instances(up["descs"], up["props"])
for p in range(3):
    ctx.render_pass(p * a.spp, a.spp)
ctx.synchronize(); ctx.reset_counters()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for p in range(a.passes):
    ctx.render_pass((3 + p) * a.spp, a.spp)
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / a.passes
c = ctx.counters()
rays = (c["closest_rays"] + c["shadow_rays"]) / a.passes
print("%-16s pass %.3f ms  %.0f Mrays/s  (%d rays/pass)" % (a.tag, ms, rays / ms / 1e3, rays), flush=True)
